"""Drop-in replacement for render/optixutils/ops.py (reference lines cited per function).

Same names, argument order and meaning; differences are deliberate fixes listed in SURVEY.md
appendix A: nothing is JIT-compiled at import, CUDA errors raise RuntimeError, no host
synchronisation, the BVH build runs on the current stream, no OptiX / NVRTC / RT cores.
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib as L

_BSDF_MODES = ['pbr', 'diffuse', 'white']      # ops.py:136 -- order matters, it is the kernel's enum
# What the forward pass records for the backward pass when the seed is shared (rnd_seed is not None):
#   "rays": the evaluated rays themselves (direction, MIS weight, env texel: 20 B per sample slot = 2.5 KB/pixel at n_samples_x = 8);
#           backward = adjoint BSDF + gradient scatter only (no sampling, no traversal);
#   "bits": 1 visibility bit per sample (16 B/pixel); backward re-generates the samples but skips the traversal;
#   None  : nothing; backward re-traces like the reference (torch_bindings.cpp:266-267).
# "rays" falls back to "bits" when the record (B*H*W * 2N^2 * 20 B: 5.4 GB at 8 x 512^2, N = 8; 13.1 GB at 8 x 800^2) would exceed
# RAY_RECORD_MAX_BYTES or RAY_RECORD_MAX_FREE_FRACTION of the device memory that is free at call time (nvdiffrast / tiny-cuda-nn
# share the GPU in a real run; the reference itself stores nothing and re-traces).
HIT_RECORD_REPLAY = "rays"
RAY_RECORD_MAX_BYTES = 32 << 30
RAY_RECORD_MAX_FREE_FRACTION = 0.5


_fits_cache = {}


def _ray_record_fits(nbytes, device):
    if nbytes > RAY_RECORD_MAX_BYTES:
        return False
    key = (str(device), int(nbytes))
    if torch.cuda.is_current_stream_capturing():       # no memory queries while a CUDA graph is being captured: reuse the eager decision
        return _fits_cache.get(key, True)
    _fits_cache[key] = _ray_record_fits_now(nbytes, device)
    return _fits_cache[key]


def _ray_record_fits_now(nbytes, device):
    free, _total = torch.cuda.mem_get_info(device)
    # memory cached by torch's allocator is reusable for the record even though the driver reports it as used
    free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
    return nbytes <= RAY_RECORD_MAX_FREE_FRACTION * free


def _f32(t, name):
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32 (got %s)" % (name, t.dtype))
    return t


# ----------------------------------------------------------------------------------------------
# Context: replaces OptiXContext / OptiXStateWrapper (ops.py:125-128)
# ----------------------------------------------------------------------------------------------
class OptiXContext:
    """Opaque per-scene state owning the acceleration structure.  `cpp_wrapper` is kept as the
    attribute name the reference's callers see (ops.py:128); here it is the C-ABI context handle."""

    def __init__(self):
        h = C.c_void_p()
        L.check(L.lib().mcs_ctx_create(C.byref(h)), "mcs_ctx_create")
        self.cpp_wrapper = h
        self._geom = None        # keeps verts/tris alive: the build is asynchronous
        self._version = 0        # bumped by every optix_build_bvh (guards the visibility-record replay)

    def __del__(self):
        try:
            if getattr(self, "cpp_wrapper", None) is not None and self.cpp_wrapper.value:
                torch.cuda.synchronize()
                L.lib().mcs_ctx_destroy(self.cpp_wrapper)
                self.cpp_wrapper = None
        except Exception:
            pass


def optix_build_bvh(optix_ctx, verts, tris, rebuild):
    """ops.py:130-133.  verts fp32 [V,3], tris int32 [T,3] (CUDA).  rebuild=0 refits boxes only."""
    assert tris.shape[0] > 0, "Got empty training triangle mesh (unrecoverable discontinuity)"
    assert verts.shape[0] > 0, "Got empty training triangle mesh (unrecoverable discontinuity)"
    L.require_cuda(verts, tris)
    v = _f32(verts, "verts").detach().reshape(-1, 3).contiguous()      # detached: the context must not keep the caller's autograd graph alive
    if tris.dtype != torch.int32:
        raise RuntimeError("tris must be int32 (the reference's callers do .int(), geometry/dlmesh.py:50)")
    t = tris.reshape(-1, 3).contiguous()
    optix_ctx._geom = (v, t)
    optix_ctx._version += 1
    L.check(L.lib().mcs_bvh_build(optix_ctx.cpp_wrapper, v.data_ptr(), v.shape[0], t.data_ptr(), t.shape[0], int(rebuild), L.stream_ptr()),
            "optix_build_bvh")


def _split_seed(rnd_seed):
    """(host uint32 seed, device pointer or None).  `rnd_seed` may be a 1-element CUDA int32 tensor: the kernel then reads the seed
    from device memory when it RUNS (mcshade.h: seed_offset_dev), so a CUDA-graph-captured training step can advance its seed with
    an in-graph `seed += 1` the way render.py:116 bumps the host counter."""
    if isinstance(rnd_seed, torch.Tensor):
        if not (rnd_seed.is_cuda and rnd_seed.dtype == torch.int32 and rnd_seed.numel() == 1):
            raise RuntimeError("rnd_seed tensor must be a 1-element CUDA int32 tensor")
        return 0, rnd_seed.data_ptr()
    return int(rnd_seed) & 0xFFFFFFFF, None


def _env_descs(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms):
    L.require_cuda(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms)
    for n, t in (("mask", mask), ("ro", ro), ("gb_pos", gb_pos), ("gb_normal", gb_normal), ("gb_view_pos", gb_view_pos), ("gb_kd", gb_kd),
                 ("gb_ks", gb_ks), ("light", light), ("pdf", pdf), ("rows", rows), ("cols", cols)):
        _f32(t, n)
    if perms.dtype != torch.int32:
        raise RuntimeError("perms must be int32")
    d = [L.nhw1(mask), L.nhwc(ro), L.nhwc(gb_pos), L.nhwc(gb_normal), L.nhwc(gb_view_pos), L.nhwc(gb_kd), L.nhwc(gb_ks),
         L.view_hwc(light), L.view_hw(pdf), L.view_h(rows), L.view_hw(cols), L.view_perms(perms)]
    return d


class _optix_env_shade_func(torch.autograd.Function):
    """ops.py:78-105"""
    _random_perm = {}

    @staticmethod
    def get_perms(n_samples_x, device):
        key = (n_samples_x, str(device))
        if key not in _optix_env_shade_func._random_perm:
            # (32k) tables with random permutations to decorrelate BSDF and light strata (ops.py:84-86)
            _optix_env_shade_func._random_perm[key] = torch.argsort(
                torch.rand(32768, n_samples_x * n_samples_x, device=device), dim=-1).int()
        return _optix_env_shade_func._random_perm[key]

    @staticmethod
    def forward(ctx, optix_ctx, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, BSDF, n_samples_x, rnd_seed,
                shadow_scale, perms, batch_offset):
        _rnd_seed = np.random.randint(2**31) if rnd_seed is None else rnd_seed
        if perms is None:
            perms = _optix_env_shade_func.get_perms(n_samples_x, ro.device)
        d = _env_descs(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms)
        B, H, W = ro.shape[0], ro.shape[1], ro.shape[2]
        diff = torch.empty(B, H, W, 3, dtype=torch.float32, device=ro.device)
        spec = torch.empty(B, H, W, 3, dtype=torch.float32, device=ro.device)
        # Visibility record (1 bit per sample, 16 B/pixel at n_samples_x = 8): with a fixed seed the backward pass traces exactly the
        # rays of the forward pass, so it can replay the record instead of re-tracing (the reference re-traces, torch_bindings.cpp:266).
        # Not possible in decorrelated mode (rnd_seed=None draws a different seed for backward, ops.py:83,100).
        need_grad = any(t.requires_grad for t in (gb_pos, gb_normal, gb_kd, gb_ks, light))
        hit = rec_cnt = rec_rays = None
        slots = 2 * n_samples_x * n_samples_x
        mode = HIT_RECORD_REPLAY if (rnd_seed is not None and need_grad) else None
        if mode == "rays" and not _ray_record_fits(B * H * W * (slots * 20 + 4), ro.device):
            mode = "bits"
        if mode == "rays":
            rec_cnt = torch.empty(B, H, W, dtype=torch.int32, device=ro.device)
            rec_rays = torch.empty(B, H, W, 5, slots, dtype=torch.float32, device=ro.device)
        elif mode == "bits":
            hit = torch.empty(B, H, W, (slots + 31) // 32, dtype=torch.int32, device=ro.device)
        seed_host, seed_dev = _split_seed(_rnd_seed)
        L.check(L.lib().mcs_env_shade_fwd(optix_ctx.cpp_wrapper, *[C.byref(x) for x in d], int(BSDF), int(n_samples_x),
                                          seed_host, seed_dev, float(shadow_scale), int(batch_offset),
                                          diff.data_ptr(), spec.data_ptr(), hit.data_ptr() if hit is not None else None,
                                          rec_cnt.data_ptr() if rec_cnt is not None else None, rec_rays.data_ptr() if rec_rays is not None else None,
                                          slots, L.stream_ptr()),
                "optix_env_shade (forward)")
        ctx.rec = (rec_cnt, rec_rays, slots)
        ctx.save_for_backward(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms)
        ctx.hit = hit
        ctx.bvh_version = optix_ctx._version
        ctx.optix_ctx = optix_ctx
        ctx.BSDF = BSDF
        ctx.n_samples_x = n_samples_x
        ctx.rnd_seed = rnd_seed
        ctx.shadow_scale = shadow_scale
        ctx.batch_offset = batch_offset
        return diff, spec

    @staticmethod
    def backward(ctx, diff_grad, spec_grad):
        optix_ctx = ctx.optix_ctx
        # decorrelated mode draws an independent seed for the backward pass (ops.py:100)
        _rnd_seed = np.random.randint(2**31) if ctx.rnd_seed is None else ctx.rnd_seed
        mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms = ctx.saved_tensors
        d = _env_descs(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms)
        B, H, W = ro.shape[0], ro.shape[1], ro.shape[2]
        dev = ro.device
        g = [torch.empty(B, H, W, 3, dtype=torch.float32, device=dev) for _ in range(4)]
        light_grad = torch.empty(light.shape[0], light.shape[1], 3, dtype=torch.float32, device=dev)
        dg, sg = L.nhwc(diff_grad.float()), L.nhwc(spec_grad.float())
        # replay is only valid against the acceleration structure the forward pass traced (the reference would re-trace whatever
        # BVH the context holds at backward time); if the context was rebuilt in between, fall back to re-tracing
        hit = ctx.hit if (ctx.hit is not None and ctx.bvh_version == optix_ctx._version) else None
        rec_cnt, rec_rays, slots = ctx.rec
        if rec_cnt is not None and ctx.bvh_version == optix_ctx._version:
            dsc = [L.nhwc(gb_pos), L.nhwc(gb_normal), L.nhwc(gb_view_pos), L.nhwc(gb_kd), L.nhwc(gb_ks), L.view_hwc(light)]
            L.check(L.lib().mcs_env_shade_bwd_replay(*[C.byref(x) for x in dsc], int(ctx.BSDF), int(ctx.n_samples_x), float(ctx.shadow_scale),
                                                     C.byref(dg), C.byref(sg), rec_cnt.data_ptr(), rec_rays.data_ptr(), int(slots),
                                                     g[0].data_ptr(), g[1].data_ptr(), g[2].data_ptr(), g[3].data_ptr(), light_grad.data_ptr(),
                                                     L.stream_ptr()), "optix_env_shade (backward, ray-record replay)")
            return (None, None, None, g[0], g[1], None, g[2], g[3], light_grad, None, None, None, None, None, None, None, None, None)
        # (a device seed tensor must still hold the forward pass's value here: advance it BEFORE the forward call, not after)
        seed_host, seed_dev = _split_seed(_rnd_seed)
        L.check(L.lib().mcs_env_shade_bwd(optix_ctx.cpp_wrapper, *[C.byref(x) for x in d], int(ctx.BSDF), int(ctx.n_samples_x),
                                          seed_host, seed_dev, float(ctx.shadow_scale), int(ctx.batch_offset),
                                          C.byref(dg), C.byref(sg), g[0].data_ptr(), g[1].data_ptr(), g[2].data_ptr(), g[3].data_ptr(),
                                          light_grad.data_ptr(), hit.data_ptr() if hit is not None else None, L.stream_ptr()),
                "optix_env_shade (backward)")
        # same gradient slots as ops.py:105 (no gradient for ro / view_pos / pdf / rows / cols)
        return (None, None, None, g[0], g[1], None, g[2], g[3], light_grad, None, None, None, None, None, None, None, None, None)


def optix_env_shade(optix_ctx, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, BSDF='pbr', n_samples_x=8,
                    rnd_seed=None, shadow_scale=1.0, perms=None, batch_offset=0):
    """ops.py:135-137.  Extra keyword-only-in-spirit arguments (defaults reproduce the reference):
    perms        -- inject the [P, n^2] int32 permutation table (the reference draws it once from the unseeded CUDA RNG)
    batch_offset -- index of this rank's first view in the global batch (data-parallel RNG parity, kernel.cu:504)"""
    iBSDF = _BSDF_MODES.index(BSDF)
    return _optix_env_shade_func.apply(optix_ctx, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, iBSDF,
                                       n_samples_x, rnd_seed, shadow_scale, perms, batch_offset)


def env_shade_records(optix_ctx, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms, BSDF='pbr',
                      n_samples_x=8, rnd_seed=0, shadow_scale=1.0, batch_offset=0):
    """Parity hook: forward pass + per-ray records (env texel, visibility).  See mcs_env_shade_records."""
    d = _env_descs(mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms)
    B, H, W = ro.shape[0], ro.shape[1], ro.shape[2]
    S2 = 2 * n_samples_x * n_samples_x
    diff = torch.empty(B, H, W, 3, dtype=torch.float32, device=ro.device)
    spec = torch.empty(B, H, W, 3, dtype=torch.float32, device=ro.device)
    rec_t = torch.full((B, H, W, S2), -1, dtype=torch.int32, device=ro.device)
    rec_v = torch.full((B, H, W, S2), 255, dtype=torch.uint8, device=ro.device)
    seed_host, seed_dev = _split_seed(rnd_seed)
    L.check(L.lib().mcs_env_shade_records(optix_ctx.cpp_wrapper, *[C.byref(x) for x in d], _BSDF_MODES.index(BSDF), int(n_samples_x),
                                          seed_host, seed_dev, float(shadow_scale), int(batch_offset), diff.data_ptr(), spec.data_ptr(),
                                          rec_t.data_ptr(), rec_v.data_ptr(), L.stream_ptr()), "env_shade_records")
    return diff, spec, rec_t, rec_v


# ----------------------------------------------------------------------------------------------
# Ray queries outside the fused kernel (parity tests, synthetic G-buffer producer)
# ----------------------------------------------------------------------------------------------
def trace_visibility(optix_ctx, ro, rd):
    """uint8 [n]: 1 if the ray (origin ro[n,3], direction rd[n,3], t in (0,1e16)) hits nothing."""
    L.require_cuda(ro, rd)
    ro = _f32(ro, "ro").reshape(-1, 3).contiguous(); rd = _f32(rd, "rd").reshape(-1, 3).contiguous()
    vis = torch.empty(ro.shape[0], dtype=torch.uint8, device=ro.device)
    L.check(L.lib().mcs_trace_visibility(optix_ctx.cpp_wrapper, ro.data_ptr(), rd.data_ptr(), ro.shape[0], vis.data_ptr(), L.stream_ptr()),
            "trace_visibility")
    return vis


def trace_closest(optix_ctx, ro, rd):
    """(tri_id int32 [n] (-1 = miss), tuv fp32 [n,3] = (t, u, v))"""
    L.require_cuda(ro, rd)
    ro = _f32(ro, "ro").reshape(-1, 3).contiguous(); rd = _f32(rd, "rd").reshape(-1, 3).contiguous()
    tid = torch.empty(ro.shape[0], dtype=torch.int32, device=ro.device)
    tuv = torch.empty(ro.shape[0], 3, dtype=torch.float32, device=ro.device)
    L.check(L.lib().mcs_trace_closest(optix_ctx.cpp_wrapper, ro.data_ptr(), rd.data_ptr(), ro.shape[0], tid.data_ptr(), tuv.data_ptr(),
                                      L.stream_ptr()), "trace_closest")
    return tid, tuv


def bvh_export(optix_ctx):
    """Binary LBVH arrays (sorted Morton keys, prim ids, children, padded boxes) for structural parity tests."""
    T = optix_ctx._geom[1].shape[0]
    dev = optix_ctx._geom[0].device
    morton = torch.empty(T, dtype=torch.int32, device=dev); prim = torch.empty(T, dtype=torch.int32, device=dev)
    left = torch.empty(max(T - 1, 1), dtype=torch.int32, device=dev); right = torch.empty(max(T - 1, 1), dtype=torch.int32, device=dev)
    lo = torch.empty(2 * T - 1, 3, dtype=torch.float32, device=dev); hi = torch.empty(2 * T - 1, 3, dtype=torch.float32, device=dev)
    L.check(L.lib().mcs_bvh_export(optix_ctx.cpp_wrapper, morton.data_ptr(), prim.data_ptr(), left.data_ptr(), right.data_ptr(), lo.data_ptr(),
                                   hi.data_ptr(), L.stream_ptr()), "bvh_export")
    return dict(morton=morton, prim=prim, left=left[:T - 1], right=right[:T - 1], lo=lo, hi=hi)


# ----------------------------------------------------------------------------------------------
# Bilateral denoiser (ops.py:107-119, 139-141)
# ----------------------------------------------------------------------------------------------
class _bilateral_denoiser_func(torch.autograd.Function):
    @staticmethod
    def forward(ctx, col, nrm, zdz, sigma):
        L.require_cuda(col, nrm, zdz)
        ctx.save_for_backward(nrm, zdz)
        ctx.sigma = sigma
        B, H, W = col.shape[0], col.shape[1], col.shape[2]
        out = torch.empty(B, H, W, 4, dtype=torch.float32, device=col.device)
        c, n, z = L.nhwc(_f32(col, "col")), L.nhwc(_f32(nrm, "nrm")), L.nhwc(_f32(zdz, "zdz"))
        L.check(L.lib().mcs_bilateral_fwd(C.byref(c), C.byref(n), C.byref(z), float(sigma), out.data_ptr(), L.stream_ptr()), "bilateral_denoiser (forward)")
        return out

    @staticmethod
    def backward(ctx, out_grad):
        nrm, zdz = ctx.saved_tensors
        B, H, W = nrm.shape[0], nrm.shape[1], nrm.shape[2]
        col_grad = torch.empty(B, H, W, 3, dtype=torch.float32, device=nrm.device)
        n, z, g = L.nhwc(nrm), L.nhwc(zdz), L.nhwc(out_grad.float())
        L.check(L.lib().mcs_bilateral_bwd(C.byref(n), C.byref(z), float(ctx.sigma), C.byref(g), col_grad.data_ptr(), L.stream_ptr()),
                "bilateral_denoiser (backward)")
        return col_grad, None, None, None      # no gradient for nrm / zdz (ops.py:119)


def bilateral_denoiser(col, nrm, zdz, sigma):
    """ops.py:139-141"""
    col_w = _bilateral_denoiser_func.apply(col, nrm, zdz, sigma)
    return col_w[..., 0:3] / col_w[..., 3:4]


class _bilateral_denoiser2_func(torch.autograd.Function):
    """Two signals, one set of guides (render.py:120-121 filters diffuse and specular identically)."""
    @staticmethod
    def forward(ctx, colA, colB, nrm, zdz, sigma):
        L.require_cuda(colA, colB, nrm, zdz)
        ctx.save_for_backward(nrm, zdz)
        ctx.sigma = sigma
        B, H, W = colA.shape[0], colA.shape[1], colA.shape[2]
        outA = torch.empty(B, H, W, 4, dtype=torch.float32, device=colA.device)
        outB = torch.empty(B, H, W, 4, dtype=torch.float32, device=colA.device)
        a, b, n, z = L.nhwc(_f32(colA, "colA")), L.nhwc(_f32(colB, "colB")), L.nhwc(_f32(nrm, "nrm")), L.nhwc(_f32(zdz, "zdz"))
        L.check(L.lib().mcs_bilateral_fwd2(C.byref(a), C.byref(b), C.byref(n), C.byref(z), float(sigma), outA.data_ptr(), outB.data_ptr(),
                                           L.stream_ptr()), "bilateral_denoiser2 (forward)")
        return outA, outB

    @staticmethod
    def backward(ctx, gA, gB):
        nrm, zdz = ctx.saved_tensors
        B, H, W = nrm.shape[0], nrm.shape[1], nrm.shape[2]
        cA = torch.empty(B, H, W, 3, dtype=torch.float32, device=nrm.device)
        cB = torch.empty(B, H, W, 3, dtype=torch.float32, device=nrm.device)
        n, z, a, b = L.nhwc(nrm), L.nhwc(zdz), L.nhwc(gA.float()), L.nhwc(gB.float())
        L.check(L.lib().mcs_bilateral_bwd2(C.byref(n), C.byref(z), float(ctx.sigma), C.byref(a), C.byref(b), cA.data_ptr(), cB.data_ptr(),
                                           L.stream_ptr()), "bilateral_denoiser2 (backward)")
        return cA, cB, None, None, None


def bilateral_denoiser2(colA, colB, nrm, zdz, sigma):
    """Fused equivalent of (bilateral_denoiser(colA, ...), bilateral_denoiser(colB, ...))."""
    a, b = _bilateral_denoiser2_func.apply(colA, colB, nrm, zdz, sigma)
    return a[..., 0:3] / a[..., 3:4], b[..., 0:3] / b[..., 3:4]


# ----------------------------------------------------------------------------------------------
# Tail of render.shade() (render/render.py:119-131), row f3: denoiser normalisation + demodulated recombination in one launch
# ----------------------------------------------------------------------------------------------
class _shade_combine_func(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a4, b4, kd, ks, pbr):
        L.require_cuda(a4, b4, kd, ks)
        a4, b4, kd, ks = _f32(a4, "a4"), _f32(b4, "b4"), _f32(kd, "kd"), _f32(ks, "ks")
        ctx.save_for_backward(a4, b4, kd, ks)
        ctx.pbr = int(pbr)
        out = torch.empty(*a4.shape[:3], 3, dtype=torch.float32, device=a4.device)
        L.check(L.lib().mcs_shade_combine_fwd(C.byref(L.nhwc(a4)), C.byref(L.nhwc(b4)), C.byref(L.nhwc(kd)), C.byref(L.nhwc(ks)), ctx.pbr, out.data_ptr(),
                                              L.stream_ptr()), "shade_combine (forward)")
        return out

    @staticmethod
    def backward(ctx, dout):
        a4, b4, kd, ks = ctx.saved_tensors
        shp = a4.shape[:3]
        d_a4 = torch.empty(*shp, 4, dtype=torch.float32, device=a4.device); d_kd = torch.empty(*shp, 3, dtype=torch.float32, device=a4.device)
        d_b4 = torch.empty(*shp, 4, dtype=torch.float32, device=a4.device) if ctx.pbr else None
        d_ks = torch.empty(*shp, 3, dtype=torch.float32, device=a4.device) if ctx.pbr else None
        g = _f32(dout, "dout")
        L.check(L.lib().mcs_shade_combine_bwd(C.byref(L.nhwc(a4)), C.byref(L.nhwc(b4)), C.byref(L.nhwc(kd)), C.byref(L.nhwc(ks)), ctx.pbr, C.byref(L.nhwc(g)),
                                              d_a4.data_ptr(), d_b4.data_ptr() if ctx.pbr else d_a4.data_ptr(), d_kd.data_ptr(),
                                              d_ks.data_ptr() if ctx.pbr else d_kd.data_ptr(), L.stream_ptr()), "shade_combine (backward)")
        return d_a4, d_b4, d_kd, d_ks, None


def shade_combine(diffuse_w, specular_w, kd, ks, BSDF='pbr'):
    """diffuse_w / specular_w: RAW [B,H,W,4] bilateral outputs (rgb weighted sum, weight) as returned by the `_func.apply` of the
    denoiser, kd / ks [B,H,W,3] full-size tensors.  Returns the shaded colour of render.py:123-127 for 'pbr' ('diffuse' / 'white':
    diffuse only, specular_w / ks unused)."""
    pbr = BSDF == 'pbr'
    if not pbr:
        specular_w, ks = diffuse_w, kd
    return _shade_combine_func.apply(diffuse_w, specular_w, kd, ks, pbr)


def denoise_and_combine(diffuse, specular, nrm, zdz, sigma, kd, ks, BSDF='pbr'):
    """render.py:119-127 in two launches: the fused two-signal bilateral filter, then normalisation + recombination."""
    a, b = _bilateral_denoiser2_func.apply(diffuse, specular, nrm, zdz, sigma)
    return shade_combine(a, b, kd, ks, BSDF)
