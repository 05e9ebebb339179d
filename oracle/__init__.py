"""CPU oracle for the nvdiffrecmc hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Thin numpy/ctypes wrapper around ``oracle/mcoracle.c`` (see that file's header for what it
restates and how it is pinned).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this package; ``nvdiffrecmc_b200`` never
does.

``build_ref()`` / ``Reference`` compile and drive the reference's OWN raygen source on the CPU (oracle/ref_shim -> oracle/_ref, only
where /root/reference exists; the built library is git-ignored and travels to the GPU box) -- the check of this restatement
against the reference itself, and the `--impl reference` arm of bench.py.

Two builds of the same source exist: fp32 (the oracle proper, ``Oracle()``) and fp64
(``Oracle(f64=True)``), the latter used only to validate the hand-derived adjoints by finite
differences.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")
_SRC = [os.path.join(_HERE, "mcoracle.c"), os.path.join(_HERE, "detmath.h")]


def _lib_path(f64):
    return os.path.join(_BUILD, "libmcoracle_f64.so" if f64 else "libmcoracle_f32.so")


def _cpu_has_fma():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return " fma " in (line + " ")
    except OSError:
        pass
    return False


def build(force=False):
    """Compile the C restatement with gcc (fp32 + fp64 variants). -ffp-contract=off is mandatory.  In a read-only tree (a
    benchmark run from an installed checkout) a library that has to be (re)built goes to a fresh temporary directory instead."""
    global _BUILD
    fresh = lambda p: os.path.exists(p) and all(os.path.getmtime(p) >= os.path.getmtime(s) for s in _SRC)
    todo = [f64 for f64 in (False, True) if force or not fresh(_lib_path(f64))]
    if todo and not os.access(_BUILD if os.path.isdir(_BUILD) else _HERE, os.W_OK):
        _BUILD, todo = tempfile.mkdtemp(prefix="mcoracle-"), [False, True]
        atexit.register(shutil.rmtree, _BUILD, True)        # a loaded library stays mapped after its file is removed
    os.makedirs(_BUILD, exist_ok=True)
    for f64 in todo:
        out = _lib_path(f64)
        cmd = ["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-o", out, _SRC[0], "-lm"]
        if _cpu_has_fma():
            cmd.insert(2, "-mfma")       # only the explicit fmaf()/fma() calls of mt_eval use it (contraction stays off)
        if f64:
            cmd.insert(1, "-DORACLE_F64")
        subprocess.run(cmd, check=True)


# ------------------------------------------------------------------------------------------------
# oracle/_ref: the UNMODIFIED reference raygen program compiled for the host (oracle/ref_shim/), only where /root/reference exists
# ------------------------------------------------------------------------------------------------
REF_KERNEL = "/root/reference/render/optixutils/c_src/envsampling/kernel.cu"
REF_DENOISE = "/root/reference/render/optixutils/c_src/denoising.cu"
REF_RU_BSDF = "/root/reference/render/renderutils/c_src/bsdf.cu"
REF_RU_NORMAL = "/root/reference/render/renderutils/c_src/normal.cu"
REF_RU_LOSS = "/root/reference/render/renderutils/c_src/loss.cu"
REF_RU_MESH = "/root/reference/render/renderutils/c_src/mesh.cu"
_REF_DIR = os.path.join(_HERE, "_ref")
_REF_LIB = os.path.join(_REF_DIR, "libref_envshade.so")
_REF_LIB_DN = os.path.join(_REF_DIR, "libref_denoise.so")
_REF_LIB_RU = os.path.join(_REF_DIR, "libref_renderutils.so")
_SHIM = os.path.join(_HERE, "ref_shim")


def build_ref(force=False):
    """g++ on the reference's own kernel.cu / denoising.cu (and the headers they include) where they lie, through the host shims.  Returns
    the env_shade library path, or None when the reference tree is not present (GPU box) and no prebuilt library travelled with the snapshot."""
    if not os.path.exists(REF_KERNEL):
        return _REF_LIB if all(os.path.exists(l) for l in (_REF_LIB, _REF_LIB_DN, _REF_LIB_RU)) else None
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    jobs = [(_REF_LIB, "ref_env_shade.cpp", {"REF_KERNEL": REF_KERNEL}), (_REF_LIB_DN, "ref_denoise.cpp", {"REF_DENOISE": REF_DENOISE}),
            (_REF_LIB_RU, "ref_renderutils.cpp", {"REF_RU_BSDF": REF_RU_BSDF, "REF_RU_NORMAL": REF_RU_NORMAL, "REF_RU_LOSS": REF_RU_LOSS, "REF_RU_MESH": REF_RU_MESH})]
    for out, shim, macros in jobs:
        srcs = [os.path.join(_SHIM, shim), os.path.join(_SHIM, "optix.h")] + list(macros.values())
        if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
            continue
        os.makedirs(_REF_DIR, exist_ok=True)
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-w", "-I" + cuda_inc, "-I" + _SHIM]
        cmd += ["-I" + d for d in sorted({os.path.dirname(v) for v in macros.values()})] + ['-D%s="%s"' % kv for kv in macros.items()]
        subprocess.run(cmd + [srcs[0], "-o", out], check=True)
    return _REF_LIB


class Reference:
    """The reference's own __raygen__rg / process_sample (kernel.cu:403-542) running on the CPU.  Visibility comes from `scene`
    (an fp32 oracle Scene): OptiX itself is closed source.  Raises RuntimeError when oracle/_ref cannot be built or found."""

    def __init__(self, orc):
        path = build_ref()
        if path is None:
            raise RuntimeError("oracle/_ref unavailable: /root/reference is not present and no prebuilt libref_envshade.so was found")
        assert not orc.f64, "the reference kernel is fp32"
        self.orc = orc
        self.lib = C.CDLL(path)
        self.lib.ref_set_visibility.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        self.lib.ref_env_shade.argtypes = [C.c_int] * 7 + [C.c_uint, C.c_uint, C.c_float, C.c_int] + [C.c_void_p] * 21
        self.lib.ref_set_ray_log.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        self.dn = C.CDLL(_REF_LIB_DN)
        self.dn.ref_bilateral_fwd.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float] + [C.c_void_p] * 4
        self.dn.ref_bilateral_bwd.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float] + [C.c_void_p] * 5

        self.ru = C.CDLL(_REF_LIB_RU)

        class _Desc(C.Structure):
            _fields_ = [("val", C.c_void_p), ("d_val", C.c_void_p), ("dims", C.c_int * 4)]
        self._Desc = _Desc
        self.ru.ref_ru_run.argtypes = [C.c_char_p, C.c_int, C.POINTER(_Desc), C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int]

    def image_loss(self, img, target, loss="l1", tonemapper="none", dout=None):
        """imgLossFwdKernel / imgLossBwdKernel (loss.cu:105-227).  Forward -> the mean of the per-pixel loss, as renderutils/ops.py:494 returns
        it; with dout (upstream gradient of that mean) -> (img_grad, target_grad)."""
        li = {"l1": 0, "mse": 1, "relmse": 2, "smape": 3, "n2n": 4}[loss]
        ti = 1 if tonemapper == "log_srgb" else 0
        img = np.ascontiguousarray(img, np.float32); target = np.ascontiguousarray(target, np.float32)
        n = img.shape[0] * img.shape[1] * img.shape[2]
        if dout is None:
            return float(self.renderutils("loss_fwd", [img, target], 1, i0=ti, i1=li).astype(np.float64).sum() / n)
        g = np.full(img.shape[:3] + (1,), np.float32(dout) / np.float32(n), np.float32)
        return self.renderutils("loss_bwd", [img, target], dout=g, i0=ti, i1=li)

    def xfm(self, points, matrix, is_points=True, dout=None):
        """xfmPointsFwdKernel / xfmPointsBwdKernel (mesh.cu:19-90).  points [B|1,V,3], matrix [B,4,4] -> [B,V,4|3]; with dout -> points gradient
        on the full batch [B,V,3] (the Python side sums it for a broadcast input)."""
        pts = np.ascontiguousarray(points, np.float32); mtx = np.ascontiguousarray(matrix, np.float32)
        B, V = mtx.shape[0], pts.shape[1]
        D = self._Desc
        descs = (D * 3)()
        out = np.zeros((B, V, 4 if is_points else 3), np.float32) if dout is None else np.ascontiguousarray(dout, np.float32)
        grad = np.zeros((B, V, 3), np.float32)
        for i, a in enumerate((pts, mtx, out)):
            descs[i].val = a.ctypes.data
            for k, v in enumerate(a.shape + (1,)):
                descs[i].dims[k] = v
        if dout is not None:
            descs[0].d_val = grad.ctypes.data
        rc = self.ru.ref_ru_run(b"xfm_bwd" if dout is not None else b"xfm_fwd", 3, descs, V, 1, B, 0.0, 1 if is_points else 0, 0)
        assert rc == 0
        return grad if dout is not None else out

    def renderutils(self, kernel, ins, out_channels=None, dout=None, f0=0.0, i0=0, i1=0):
        """Run one per-pixel kernel of render/renderutils/c_src/{bsdf,normal}.cu.  `kernel`: lambert|frostbite|fresnel|ndf|lambda|masking|
        specular|bsdf|psn + _fwd / _bwd.  ins: [N|1, H|1, W|1, C] arrays in the order of the kernel's parameter struct.  Forward returns
        out [N,H,W,out_channels]; backward (dout = upstream gradient) returns one full-grid gradient per input, as the plugin does
        before the Python side sums broadcast dimensions (renderutils/ops.py)."""
        ins = [np.ascontiguousarray(a, np.float32) for a in ins]
        grid = np.broadcast_shapes(*[a.shape[:3] for a in ins])
        N, H, W = grid
        bwd = dout is not None
        keep, descs = [], (self._Desc * (len(ins) + 1))()
        grads = []
        for i, a in enumerate(ins):
            descs[i].val = a.ctypes.data
            if bwd:
                g = np.zeros((N, H, W, a.shape[3]), np.float32); grads.append(g); descs[i].d_val = g.ctypes.data
            for k in range(4):
                descs[i].dims[k] = a.shape[k]
        out = np.ascontiguousarray(dout, np.float32) if bwd else np.zeros((N, H, W, out_channels), np.float32)
        descs[len(ins)].val = out.ctypes.data
        for k, v in enumerate(out.shape):
            descs[len(ins)].dims[k] = v
        rc = self.ru.ref_ru_run(kernel.encode(), len(ins) + 1, descs, W, H, N, float(f0), int(i0), int(i1))
        if rc != 0:
            raise ValueError("ref_ru_run(%s): %s" % (kernel, {1: "unknown kernel", 2: "wrong tensor count"}.get(rc, rc)))
        return grads if bwd else out

    def bilateral_fwd(self, col, nrm, zdz, sigma):
        """bilateral_denoiser_fwd_kernel (denoising.cu:14-72): -> [B,H,W,4] (rgb weighted sum, weight)."""
        f = lambda a: np.ascontiguousarray(a, np.float32)
        col, nrm, zdz = f(col), f(nrm), f(zdz)
        B, H, W = col.shape[:3]
        out = np.zeros((B, H, W, 4), np.float32)
        self.dn.ref_bilateral_fwd(B, H, W, float(sigma), col.ctypes.data, nrm.ctypes.data, zdz.ctypes.data, out.ctypes.data)
        return out

    def bilateral_bwd(self, nrm, zdz, sigma, out_grad, col=None):
        """bilateral_denoiser_bwd_kernel (denoising.cu:74-130): out_grad [B,H,W,4] -> col_grad [B,H,W,3]."""
        f = lambda a: np.ascontiguousarray(a, np.float32)
        nrm, zdz, og = f(nrm), f(zdz), f(out_grad)
        B, H, W = nrm.shape[:3]
        col = np.zeros((B, H, W, 3), np.float32) if col is None else f(col)
        cg = np.zeros((B, H, W, 3), np.float32)
        self.dn.ref_bilateral_bwd(B, H, W, float(sigma), col.ctypes.data, nrm.ctypes.data, zdz.ctypes.data, og.ctypes.data, cg.ctypes.data)
        return cg

    def env_shade(self, scene, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms, BSDF="pbr", n_samples_x=8,
                  rnd_seed=0, shadow_scale=1.0, grads=None, vis_mode="brute", ray_log=False):
        """Forward -> (diff, spec); with grads=(diff_grad, spec_grad) -> (pos_grad, nrm_grad, kd_grad, ks_grad, light_grad).
        ray_log=True (forward only) appends the directions of the shadow rays the reference traced, [B,H,W,2*n^2,3] in sample-slot
        order (NaN where the pixel is masked)."""
        f = lambda a: np.ascontiguousarray(a, np.float32)
        mask, ro, gb_pos, gb_normal, gb_kd, gb_ks = [f(a) for a in (mask, ro, gb_pos, gb_normal, gb_kd, gb_ks)]
        B, H, W = mask.shape
        view = np.ascontiguousarray(np.broadcast_to(f(gb_view_pos), (B, 1, 1, 3)))
        light, pdf, rows, cols = f(light), f(pdf), f(rows), f(cols)
        perms = np.ascontiguousarray(perms, np.int32)
        assert perms.shape[1] == n_samples_x * n_samples_x
        Hl, Wl = light.shape[:2]
        z4 = lambda: np.zeros((B, H, W, 3), np.float32)
        diff, spec = z4(), z4()
        dg, sg = (f(grads[0]), f(grads[1])) if grads is not None else (z4(), z4())
        pg, ng, kg, sgd, lg = z4(), z4(), z4(), z4(), np.zeros((Hl, Wl, 3), np.float32)
        occ = C.cast(self.orc.lib.orc_occluded1, C.c_void_p)
        self.lib.ref_set_visibility(occ, scene.h, {"brute": 0, "bvh": 1}[vis_mode])
        p = lambda a: a.ctypes.data
        S2 = 2 * n_samples_x * n_samples_x
        if ray_log:
            dirs = np.full((B, H, W, S2, 3), np.nan, np.float32); cnt = np.zeros((B, H, W), np.int32)
            self.lib.ref_set_ray_log(p(dirs), p(cnt), S2)
        self.lib.ref_env_shade(B, H, W, Hl, Wl, perms.shape[0], n_samples_x, BSDF_MODES.index(BSDF), int(rnd_seed) & 0xFFFFFFFF, float(shadow_scale),
                               0 if grads is None else 1, p(mask), p(ro), p(gb_pos), p(gb_normal), p(view), p(gb_kd), p(gb_ks), p(light), p(pdf), p(rows),
                               p(cols), p(perms), p(diff), p(spec), p(dg), p(sg), p(pg), p(ng), p(kg), p(sgd), p(lg))
        if ray_log:
            self.lib.ref_set_ray_log(None, None, 0)
            assert int(cnt.max()) <= S2
            return diff, spec, dirs
        return (diff, spec) if grads is None else (pg, ng, kg, sgd, lg)


def _envshade_struct(real):
    P = C.POINTER
    class S(C.Structure):
        _fields_ = [
            ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Hl", C.c_int32), ("Wl", C.c_int32),
            ("n_perms", C.c_int32), ("N", C.c_int32), ("bsdf", C.c_int32), ("seed", C.c_uint32),
            ("batch_offset", C.c_int32), ("backward", C.c_int32), ("vis_mode", C.c_int32), ("parallel_bwd", C.c_int32), ("shadow_scale", real),
            ("mask", C.c_void_p), ("ro", C.c_void_p), ("pos", C.c_void_p), ("nrm", C.c_void_p), ("view", C.c_void_p),
            ("kd", C.c_void_p), ("ks", C.c_void_p),
            ("light", C.c_void_p), ("pdf", C.c_void_p), ("rows", C.c_void_p), ("cols", C.c_void_p),
            ("perms", C.c_void_p), ("scene", C.c_void_p),
            ("diff", C.c_void_p), ("spec", C.c_void_p), ("diff_grad", C.c_void_p), ("spec_grad", C.c_void_p),
            ("pos_grad", C.c_void_p), ("nrm_grad", C.c_void_p), ("kd_grad", C.c_void_p), ("ks_grad", C.c_void_p),
            ("light_grad", C.c_void_p),
            ("rec_texel", C.c_void_p), ("rec_vis", C.c_void_p), ("counters", C.c_void_p),
            ("s_pos", C.c_void_p), ("s_nrm", C.c_void_p), ("s_kd", C.c_void_p), ("s_ks", C.c_void_p),
        ]
    return S


BSDF_MODES = ["pbr", "diffuse", "white"]     # render/optixutils/ops.py:136


class Scene:
    """Triangle soup + canonical LBVH held by the C side."""
    def __init__(self, orc, verts, tris):
        self.orc = orc
        self.verts = np.ascontiguousarray(verts, dtype=orc.dt).reshape(-1, 3)
        self.tris = np.ascontiguousarray(tris, dtype=np.int32).reshape(-1, 3)
        assert self.tris.shape[0] > 0 and self.verts.shape[0] > 0
        self.T = self.tris.shape[0]
        self.h = orc.lib.orc_scene_create(self.verts.ctypes.data, self.verts.shape[0], self.tris.ctypes.data, self.T)
        orc.lib.orc_lbvh_build(self.h, self.verts.ctypes.data, self.tris.ctypes.data)

    def __del__(self):
        try:
            self.orc.lib.orc_scene_destroy(self.h)
        except Exception:
            pass

    def export_lbvh(self):
        T = self.T
        morton = np.zeros(T, np.uint32); prim = np.zeros(T, np.int32)
        left = np.zeros(max(T - 1, 1), np.int32); right = np.zeros(max(T - 1, 1), np.int32)
        lo = np.zeros((2 * T - 1, 3), self.orc.dt); hi = np.zeros((2 * T - 1, 3), self.orc.dt)
        self.orc.lib.orc_lbvh_export(self.h, morton.ctypes.data, prim.ctypes.data, left.ctypes.data, right.ctypes.data,
                                     lo.ctypes.data, hi.ctypes.data)
        return dict(morton=morton, prim=prim, left=left[:T - 1], right=right[:T - 1], lo=lo, hi=hi)

    def visibility(self, ro, rd, mode="brute", return_counters=False):
        ro = np.ascontiguousarray(ro, self.orc.dt).reshape(-1, 3); rd = np.ascontiguousarray(rd, self.orc.dt).reshape(-1, 3)
        vis = np.zeros(ro.shape[0], np.uint8); cnt = np.zeros(2, np.uint64)
        self.orc.lib.orc_visibility(self.h, 0 if mode == "brute" else 1, ro.shape[0], ro.ctypes.data, rd.ctypes.data,
                                    vis.ctypes.data, cnt.ctypes.data)
        return (vis, cnt) if return_counters else vis

    def closest_hit(self, ro, rd):
        ro = np.ascontiguousarray(ro, self.orc.dt).reshape(-1, 3); rd = np.ascontiguousarray(rd, self.orc.dt).reshape(-1, 3)
        tid = np.zeros(ro.shape[0], np.int32); tuv = np.zeros((ro.shape[0], 3), self.orc.dt)
        self.orc.lib.orc_closest_hit(self.h, ro.shape[0], ro.ctypes.data, rd.ctypes.data, tid.ctypes.data, tuv.ctypes.data)
        return tid, tuv


class Oracle:
    def __init__(self, f64=False):
        build()
        self.f64 = f64
        self.dt = np.float64 if f64 else np.float32
        self.real = C.c_double if f64 else C.c_float
        self.lib = C.CDLL(_lib_path(f64))
        self.lib.orc_scene_create.restype = C.c_void_p
        self.lib.orc_scene_create.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        self.lib.orc_lbvh_build.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        self.lib.orc_scene_destroy.argtypes = [C.c_void_p]
        self.lib.orc_lbvh_export.argtypes = [C.c_void_p] * 7
        self.lib.orc_visibility.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        self.lib.orc_closest_hit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        self.lib.orc_env_shade.argtypes = [C.c_void_p]
        self.lib.orc_hash_pcg.restype = C.c_uint32
        self.lib.orc_hash_pcg.argtypes = [C.c_uint32, C.c_uint32]
        self.lib.orc_rand_pcg.restype = C.c_uint32
        self.lib.orc_rand_pcg.argtypes = [C.c_void_p]
        assert self.lib.orc_sizeof_real() == (8 if f64 else 4)
        self._ES = _envshade_struct(self.real)
        assert self.lib.orc_sizeof_envshade() == C.sizeof(self._ES), "struct layout mismatch"

    # ------------------------------------------------------------------ helpers
    def set_threads(self, n):
        """OpenMP team size of the oracle's parallel loops.  Called explicitly because OMP_NUM_THREADS is only read when libgomp
        initialises (torch has usually loaded it already) and torchrun exports OMP_NUM_THREADS=1.  Returns the size in effect."""
        self.lib.omp_set_num_threads(int(n))
        return int(self.lib.omp_get_max_threads())

    def _a(self, x, shape=None):
        x = np.ascontiguousarray(np.asarray(x, dtype=self.dt))
        if shape is not None:
            x = np.ascontiguousarray(np.broadcast_to(x, shape))
        return x

    def _bc(self, *arrs, chans):
        """Broadcast NHWC arrays over their leading dims (size-1 dims broadcast, tensor.h:32)."""
        arrs = [np.asarray(a, dtype=self.dt) for a in arrs]
        lead = np.broadcast_shapes(*[a.shape[:-1] for a in arrs])
        out = [np.ascontiguousarray(np.broadcast_to(a, lead + (c,))) for a, c in zip(arrs, chans)]
        return lead, out

    def scene(self, verts, tris):
        return Scene(self, verts, tris)

    # ------------------------------------------------------------------ elementwise ops
    def _run(self, name, ins, chans, extra, outs_ch, extra_after_ins=True, dout=None, dout_ch=None):
        allin = list(ins) + ([dout] if dout is not None else [])
        allch = list(chans) + ([dout_ch] if dout is not None else [])
        lead, arrs = self._bc(*allin, chans=allch)
        n = int(np.prod(lead)) if len(lead) else 1
        outs = [np.zeros(lead + (c,), self.dt) for c in outs_ch]
        args = [C.c_int(n)] + [C.c_void_p(a.ctypes.data) for a in arrs[:len(ins)]]
        for e in extra:
            args.append(self.real(e) if isinstance(e, float) else C.c_int(int(e)))
        if dout is not None:
            args.append(C.c_void_p(arrs[-1].ctypes.data))
        args += [C.c_void_p(o.ctypes.data) for o in outs]
        getattr(self.lib, name)(*args)
        return outs[0] if len(outs) == 1 else tuple(outs)

    def lambert(self, nrm, wi):
        return self._run("orc_lambert_fwd", [nrm, wi], [3, 3], [], [1])

    def lambert_bwd(self, nrm, wi, dout):
        return self._run("orc_lambert_bwd", [nrm, wi], [3, 3], [], [3, 3], dout=dout, dout_ch=1)

    def frostbite_diffuse(self, nrm, wi, wo, lr):
        return self._run("orc_frostbite_fwd", [nrm, wi, wo, lr], [3, 3, 3, 1], [], [1])

    def frostbite_diffuse_bwd(self, nrm, wi, wo, lr, dout):
        return self._run("orc_frostbite_bwd", [nrm, wi, wo, lr], [3, 3, 3, 1], [], [3, 3, 3, 1], dout=dout, dout_ch=1)

    def fresnel_shlick(self, f0, f90, cosT):
        return self._run("orc_fresnel_shlick_fwd", [f0, f90, cosT], [3, 3, 1], [], [3])

    def fresnel_shlick_bwd(self, f0, f90, cosT, dout):
        return self._run("orc_fresnel_shlick_bwd", [f0, f90, cosT], [3, 3, 1], [], [3, 3, 1], dout=dout, dout_ch=3)

    def ndf_ggx(self, a2, c):
        return self._run("orc_ndf_ggx_fwd", [a2, c], [1, 1], [], [1])

    def ndf_ggx_bwd(self, a2, c, dout):
        return self._run("orc_ndf_ggx_bwd", [a2, c], [1, 1], [], [1, 1], dout=dout, dout_ch=1)

    def lambda_ggx(self, a2, c):
        return self._run("orc_lambda_ggx_fwd", [a2, c], [1, 1], [], [1])

    def lambda_ggx_bwd(self, a2, c, dout):
        return self._run("orc_lambda_ggx_bwd", [a2, c], [1, 1], [], [1, 1], dout=dout, dout_ch=1)

    def masking_smith(self, a2, ci, co):
        return self._run("orc_masking_smith_fwd", [a2, ci, co], [1, 1, 1], [], [1])

    def masking_smith_bwd(self, a2, ci, co, dout):
        return self._run("orc_masking_smith_bwd", [a2, ci, co], [1, 1, 1], [], [1, 1, 1], dout=dout, dout_ch=1)

    def pbr_specular(self, col, nrm, wo, wi, alpha, min_roughness=0.08):
        return self._run("orc_pbr_specular_fwd", [col, nrm, wo, wi, alpha], [3, 3, 3, 3, 1], [float(min_roughness)], [3])

    def pbr_specular_bwd(self, col, nrm, wo, wi, alpha, dout, min_roughness=0.08):
        return self._run("orc_pbr_specular_bwd", [col, nrm, wo, wi, alpha], [3, 3, 3, 3, 1], [float(min_roughness)],
                         [3, 3, 3, 3, 1], dout=dout, dout_ch=3)

    def pbr_bsdf(self, kd, arm, pos, nrm, view_pos, light_pos, min_roughness=0.08, bsdf="lambert"):
        return self._run("orc_pbr_bsdf_fwd", [kd, arm, pos, nrm, view_pos, light_pos], [3] * 6,
                         [float(min_roughness), 1 if bsdf == "frostbite" else 0], [3])

    def pbr_bsdf_bwd(self, kd, arm, pos, nrm, view_pos, light_pos, dout, min_roughness=0.08, bsdf="lambert"):
        return self._run("orc_pbr_bsdf_bwd", [kd, arm, pos, nrm, view_pos, light_pos], [3] * 6,
                         [float(min_roughness), 1 if bsdf == "frostbite" else 0], [3] * 6, dout=dout, dout_ch=3)

    def prepare_shading_normal(self, pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm, two_sided_shading=True, opengl=True):
        if perturbed_nrm is None:
            perturbed_nrm = np.array([0, 0, 1], self.dt)[None, None, None, :]   # renderutils/ops.py:217-218
        return self._run("orc_prepare_shading_normal_fwd", [pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm],
                         [3] * 6, [int(two_sided_shading), int(opengl)], [3])

    def prepare_shading_normal_bwd(self, pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm, dout, two_sided_shading=True, opengl=True):
        if perturbed_nrm is None:
            perturbed_nrm = np.array([0, 0, 1], self.dt)[None, None, None, :]
        return self._run("orc_prepare_shading_normal_bwd", [pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm],
                         [3] * 6, [int(two_sided_shading), int(opengl)], [3] * 6, dout=dout, dout_ch=3)

    # ------------------------------------------------------------------ light pdf / cdf
    def dirs_to_texels(self, dirs, Hl, Wl):
        """Env texel ((y << 16) | x) of each direction, computed exactly as env_shade records it."""
        d = np.ascontiguousarray(dirs, self.dt).reshape(-1, 3)
        out = np.zeros(d.shape[0], np.int32)
        self.lib.orc_dirs_to_texels(C.c_int(d.shape[0]), C.c_int(Hl), C.c_int(Wl), C.c_void_p(d.ctypes.data), C.c_void_p(out.ctypes.data))
        return out.reshape(np.asarray(dirs).shape[:-1])

    def update_pdf(self, base):
        base = self._a(base); H, W = base.shape[:2]
        pdf = np.zeros((H, W), self.dt); rows = np.zeros(H, self.dt); cols = np.zeros((H, W), self.dt)
        self.lib.orc_update_pdf(C.c_int(H), C.c_int(W), C.c_void_p(base.ctypes.data), C.c_void_p(pdf.ctypes.data),
                                C.c_void_p(rows.ctypes.data), C.c_void_p(cols.ctypes.data))
        return pdf, rows, cols

    # ------------------------------------------------------------------ env shade
    def env_shade(self, scene, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms,
                  BSDF="pbr", n_samples_x=8, rnd_seed=0, shadow_scale=1.0, batch_offset=0, vis_mode="brute",
                  grads=None, records=False, counters=False, parallel_bwd=False, sampling_gbuffer=None):
        """Forward (grads=None) -> (diff, spec[, records][, counters]);
        backward (grads=(diff_grad, spec_grad)) -> (pos_grad, nrm_grad, kd_grad, ks_grad, light_grad).
        Mirrors env_shade_fwd / env_shade_bwd, render/optixutils/c_src/torch_bindings.cpp:123-272."""
        assert scene is None or scene.orc is self, "scene was built by a different Oracle instance (fp32 vs fp64 layouts differ)"
        ro = np.asarray(ro, self.dt)
        B, H, W = ro.shape[:3]
        full = (B, H, W, 3)
        mask = self._a(mask, (B, H, W))
        ro = self._a(ro, full); pos = self._a(gb_pos, full); nrm = self._a(gb_normal, full)
        view = self._a(gb_view_pos, full); kd = self._a(gb_kd, full); ks = self._a(gb_ks, full)
        light = self._a(light); pdf = self._a(pdf); rows = self._a(rows); cols = self._a(cols)
        perms = np.ascontiguousarray(perms, np.int32)
        N = int(n_samples_x); S = N * N
        assert perms.shape[1] == S and rows.ndim == 1
        p = self._ES()
        p.B, p.H, p.W = B, H, W
        p.Hl, p.Wl = light.shape[0], light.shape[1]
        p.n_perms = perms.shape[0]; p.N = N
        p.bsdf = BSDF_MODES.index(BSDF) if isinstance(BSDF, str) else int(BSDF)
        p.seed = int(rnd_seed) & 0xFFFFFFFF
        p.batch_offset = int(batch_offset)
        p.vis_mode = 2 if scene is None else {"brute": 0, "bvh": 1, "none": 2}[vis_mode]
        p.shadow_scale = float(shadow_scale)
        p.parallel_bwd = int(parallel_bwd)
        keep = [mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, perms]
        p.mask, p.ro, p.pos, p.nrm, p.view, p.kd, p.ks = [a.ctypes.data for a in (mask, ro, pos, nrm, view, kd, ks)]
        p.light, p.pdf, p.rows, p.cols, p.perms = [a.ctypes.data for a in (light, pdf, rows, cols, perms)]
        p.scene = scene.h if scene is not None else None
        if sampling_gbuffer is not None:       # test-only: (pos, nrm, kd, ks) used for the sampling decisions
            sg_ = [self._a(x, full) for x in sampling_gbuffer]
            keep += sg_
            p.s_pos, p.s_nrm, p.s_kd, p.s_ks = [a.ctypes.data for a in sg_]
        cnt = np.zeros(3, np.uint64); p.counters = cnt.ctypes.data
        rec_t = rec_v = None
        if records:
            rec_t = np.full((B, H, W, 2 * S), -1, np.int32); rec_v = np.full((B, H, W, 2 * S), 255, np.uint8)
            p.rec_texel = rec_t.ctypes.data; p.rec_vis = rec_v.ctypes.data
        if grads is None:
            diff = np.zeros(full, self.dt); spec = np.zeros(full, self.dt)
            p.backward = 0; p.diff = diff.ctypes.data; p.spec = spec.ctypes.data
            self.lib.orc_env_shade(C.byref(p))
            out = [diff, spec]
            if records:
                out.append((rec_t, rec_v))
            if counters:
                out.append(cnt)
            return tuple(out)
        dg = self._a(grads[0], full); sg = self._a(grads[1], full)
        pg, ng, kg, sgr = (np.zeros(full, self.dt) for _ in range(4))
        lg = np.zeros(light.shape, self.dt)
        p.backward = 1
        p.diff_grad, p.spec_grad = dg.ctypes.data, sg.ctypes.data
        p.pos_grad, p.nrm_grad, p.kd_grad, p.ks_grad, p.light_grad = [a.ctypes.data for a in (pg, ng, kg, sgr, lg)]
        self.lib.orc_env_shade(C.byref(p))
        del keep
        return pg, ng, kg, sgr, lg

    # ------------------------------------------------------------------ denoiser
    def bilateral_fwd(self, col, nrm, zdz, sigma):
        """out [B,H,W,4] = (sum w*col, max(sum w, 1e-4)); denoising.cu:14-72."""
        col = self._a(col); nrm = self._a(nrm); zdz = self._a(zdz)
        B, H, W = col.shape[:3]
        out = np.zeros((B, H, W, 4), self.dt)
        self.lib.orc_bilateral_fwd(C.c_int(B), C.c_int(H), C.c_int(W), C.c_void_p(col.ctypes.data), C.c_void_p(nrm.ctypes.data),
                                   C.c_void_p(zdz.ctypes.data), self.real(sigma), C.c_void_p(out.ctypes.data))
        return out

    def bilateral_bwd(self, nrm, zdz, sigma, out_grad):
        nrm = self._a(nrm); zdz = self._a(zdz); out_grad = self._a(out_grad)
        B, H, W = nrm.shape[:3]
        cg = np.zeros((B, H, W, 3), self.dt)
        self.lib.orc_bilateral_bwd(C.c_int(B), C.c_int(H), C.c_int(W), C.c_void_p(nrm.ctypes.data), C.c_void_p(zdz.ctypes.data),
                                   self.real(sigma), C.c_void_p(out_grad.ctypes.data), C.c_void_p(cg.ctypes.data))
        return cg

    def bilateral_denoiser(self, col, nrm, zdz, sigma):
        """render/optixutils/ops.py:139-141"""
        o = self.bilateral_fwd(col, nrm, zdz, sigma)
        return o[..., 0:3] / o[..., 3:4]

    # ------------------------------------------------------------------ row f3: image loss, xfm
    _LOSSES = {"l1": 0, "mse": 1, "relmse": 2, "smape": 3, "n2n": 4}

    def image_loss(self, img, target, loss="l1", tonemapper="none"):
        """renderutils/ops.py:476-498: mean over pixels of mean_c(loss)."""
        lead, (a, b) = self._bc(img, target, chans=[3, 3])
        n = int(np.prod(lead)); px = np.zeros(n, self.dt)
        self.lib.orc_image_loss_fwd(C.c_int(n), C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), C.c_int(self._LOSSES[loss]),
                                    C.c_int(1 if tonemapper == "log_srgb" else 0), C.c_void_p(px.ctypes.data))
        return px.sum(dtype=np.float64) / n

    def image_loss_bwd(self, img, target, loss="l1", tonemapper="none", dout=1.0):
        lead, (a, b) = self._bc(img, target, chans=[3, 3])
        n = int(np.prod(lead)); dpx = np.full(n, dout / n, self.dt)
        gi = np.zeros(lead + (3,), self.dt); gt = np.zeros(lead + (3,), self.dt)
        self.lib.orc_image_loss_bwd(C.c_int(n), C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), C.c_int(self._LOSSES[loss]),
                                    C.c_int(1 if tonemapper == "log_srgb" else 0), C.c_void_p(dpx.ctypes.data), C.c_void_p(gi.ctypes.data),
                                    C.c_void_p(gt.ctypes.data))
        return gi, gt

    def xfm(self, points, matrix, is_points=True):
        pts = self._a(points); m = self._a(matrix)
        B, V = m.shape[0], pts.shape[1]
        out = np.zeros((B, V, 4 if is_points else 3), self.dt)
        self.lib.orc_xfm_fwd(C.c_int(B), C.c_int(pts.shape[0]), C.c_int(V), C.c_void_p(pts.ctypes.data), C.c_void_p(m.ctypes.data), C.c_int(int(is_points)),
                             C.c_void_p(out.ctypes.data))
        return out

    def xfm_bwd(self, matrix, dout, is_points=True):
        m = self._a(matrix); g = self._a(dout)
        B, V = g.shape[0], g.shape[1]
        out = np.zeros((B, V, 3), self.dt)
        self.lib.orc_xfm_bwd(C.c_int(B), C.c_int(V), C.c_void_p(m.ctypes.data), C.c_void_p(g.ctypes.data), C.c_int(int(is_points)), C.c_void_p(out.ctypes.data))
        return out

    # ------------------------------------------------------------------ det math (fp32 only)
    def det_sincos(self, a):
        a = np.ascontiguousarray(a, np.float32); s = np.zeros_like(a); c = np.zeros_like(a)
        self.lib.orc_det_sincos(C.c_int(a.size), C.c_void_p(a.ctypes.data), C.c_void_p(s.ctypes.data), C.c_void_p(c.ctypes.data))
        return s, c

    def det_atan2(self, y, x):
        y = np.ascontiguousarray(y, np.float32); x = np.ascontiguousarray(x, np.float32); o = np.zeros_like(y)
        self.lib.orc_det_atan2(C.c_int(y.size), C.c_void_p(y.ctypes.data), C.c_void_p(x.ctypes.data), C.c_void_p(o.ctypes.data))
        return o

    def det_acos(self, x):
        x = np.ascontiguousarray(x, np.float32); o = np.zeros_like(x)
        self.lib.orc_det_acos(C.c_int(x.size), C.c_void_p(x.ctypes.data), C.c_void_p(o.ctypes.data))
        return o
