#!/usr/bin/env python
"""bench.py -- hot-path benchmark (BASELINE.json metric: Mrays/s + train iters/s @512x512, 64 spp).

One "step" = one training iteration's worth of the hot path on one batch of synthetic views:
    update_pdf -> LBVH rebuild -> prepare_shading_normal -> env_shade fwd (2*N^2 shadow rays / covered pixel)
    -> fused bilateral denoise (diffuse + specular) -> recombine + fused log-sRGB L1 image loss -> full backward
    (denoise bwd, env_shade bwd re-tracing all rays, shading-normal bwd, texture scatter)
    -> [N > 1: one NCCL all-reduce over the flat parameter-gradient bucket].
value = shadow rays processed per second over the whole job (fwd + bwd rays, all ranks), in Mrays/s;
a ray is counted the way the reference traces it: covered pixels x 2 N^2 per pass (SURVEY.md section 8d).

Usage:  python bench.py --gpus N --steps K --warmup W          (torchrun for N > 1)
        python bench.py --impl reference ...                    (CPU oracle arm)
        python bench.py ... --dump-outputs DIR                  (also save the last timed step's outputs as DIR/<name>.npy)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True         # the benchmark may run from a read-only tree: no __pycache__ next to the sources

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD = dict(name="spot_metal-like synthetic (BASELINE configs[2]): 8 views x 512x512, n_samples_x=8 (64 spp, 128 shadow rays/px), "
                     "procedural 7168-tri blob+ring mesh, 256x256 trainable probe, bilateral denoiser sigma=2",
                views_per_gpu=8, res=512, n_samples_x=8, mesh="blob+torus", mesh_level=4, light_res=256, tex_res=1024, sigma=2.0,
                ref_light_hw=(1024, 2048), global_batch_strong=8)


# ------------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  nvidia-smi needs a few hundred ms to
    start, so the poller is started before the warm-up steps and every sample is time-stamped; the summary uses the samples that fall
    inside the timed window (and says so), falling back to the samples taken under the warm-up load if the window caught < 2."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop, self.th, self.proc = index, [], False, None, None
        self.t_load = self.t0 = self.t1 = None

    def _run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self.stop:
                    break
                if line.strip():
                    self.samples.append((time.time(), [x.strip() for x in line.strip().split(",")]))
        except Exception:
            pass

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True); self.th.start(); self.t_load = time.time(); return self

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def close(self):
        self.stop = True
        try:
            self.proc.terminate()
        except Exception:
            pass
        if self.th is not None:
            self.th.join(timeout=6)

    def summary(self):
        inside = [s for t, s in self.samples if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e30)]
        window = "timed region"
        if len(inside) < 2:
            inside = [s for t, s in self.samples if t >= (self.t_load or 0) + 0.5 and t <= (self.t1 or 1e30)]
            window = "warm-up + timed region (timed region shorter than two 50 ms samples)"
        sm = [float(s[0]) for s in inside if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in inside if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in inside if len(s) >= 6 for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm),
                "window": window}


# ------------------------------------------------------------------------------------------------
def build_scene_numpy(wl, rank):
    from nvdiffrecmc_b200 import synth
    v, f = synth.scene_mesh(wl["mesh"], level=wl["mesh_level"], seed=5)
    vn = synth.vertex_normals(v, f)
    return v, f, vn


def view_pose(gi):
    """Camera of global candidate view `gi` (same on every rank)."""
    ang = float(np.random.default_rng(4).uniform(0, 2 * np.pi, size=4096)[gi])
    return ang, -0.4 + 0.3 * np.sin(gi)


def deal_views(cover, world, per_rank):
    """Global batch order = greedy (largest first, least-loaded rank) deal of the candidate views by covered pixels, so that every rank's contiguous slice
    [r*per_rank, (r+1)*per_rank) carries the same number of shadow rays to within ~1 % (VERDICT r1 item 5: with per-view static
    sharding the slowest rank set the step time at the all-reduce).  The ORDER of a batch is free -- the reference's batch is whatever
    the DataLoader collates (train.py:371) -- so batch_offset = rank * per_rank keeps the single-process RNG stream (kernel.cu:504)."""
    order = np.argsort(-np.asarray(cover), kind="stable")
    slots, load = [[] for _ in range(world)], [0] * world
    for gi in order:                                   # longest-processing-time-first with a capacity of per_rank views per rank
        r = min((k for k in range(world) if len(slots[k]) < per_rank), key=lambda k: (load[k], k))
        slots[r].append(int(gi)); load[r] += int(cover[gi])
    return [gi for r in range(world) for gi in slots[r]]


class GpuWorkload:
    """All device-resident state of one rank: `views` views of the global batch starting at global slot `offset`."""

    def __init__(self, wl, rank, world, dev, views=None, light_init="random", global_views=None):
        import torch
        import nvdiffrecmc_b200.optixutils as ou
        from nvdiffrecmc_b200 import parallel, synth
        from nvdiffrecmc_b200.light import EnvironmentLight
        from nvdiffrecmc_b200.denoiser import BilateralDenoiser
        self.torch, self.ou, self.wl, self.dev, self.rank, self.world = torch, ou, wl, dev, rank, world
        B = self.B = views if views is not None else wl["views_per_gpu"]
        res, N = wl["res"], wl["n_samples_x"]
        self.offset = rank * B
        v, f, vn = build_scene_numpy(wl, rank)
        self.mesh = (v, f)
        self.verts = torch.tensor(v, device=dev); self.tris = torch.tensor(f, device=dev)
        self.ctx = ou.OptiXContext()
        ou.optix_build_bvh(self.ctx, self.verts, self.tris, rebuild=1)

        def primary(gi, r):
            ang, tilt = view_pose(gi)
            campos, ro, rd = synth.primary_rays(synth.orbit_view(ang, tilt=tilt), r)
            tid, tuv = ou.trace_closest(self.ctx, torch.tensor(ro.reshape(-1, 3), device=dev), torch.tensor(rd.reshape(-1, 3), device=dev))
            return campos, tid.cpu().numpy().reshape(r, r), tuv.cpu().numpy().reshape(r, r, 3)

        # global batch = world*B views, ordered by a coverage-balanced deal (identical on every rank: 64^2 primary rays per candidate)
        n_glob = world * B
        if global_views is None:
            cover = [int((primary(gi, 64)[1] >= 0).sum()) for gi in range(n_glob)]
            global_views = deal_views(cover, world, B)
        self.global_views = list(global_views)
        mine = self.global_views[rank * B:(rank + 1) * B]
        # G-buffer: primary rays through our own BVH (SURVEY f2)
        gb = []
        for gi in mine:
            campos, tid, tuv = primary(gi, res)
            gb.append(synth.assemble_gbuffer(v, f, vn, tid, tuv, campos, seed=100 + gi))
        st = lambda k: np.stack([g[k] for g in gb])
        self.host = dict(mask=st("mask"), pos=st("pos"), smooth_nrm=st("smooth_nrm"), tangent=st("tangent"), geom_nrm=st("geom_nrm"),
                         view=st("view_pos").reshape(B, 1, 1, 3), depth=st("depth"))
        # texel index of each pixel into the trainable kd / ks textures (stand-in for dr.texture: nearest texel of a hashed uv)
        tr = wl["tex_res"]
        self.host["texel"] = np.stack([np.random.default_rng(1000 + gi).integers(0, tr * tr, size=(res, res)) for gi in mine]).astype(np.int64)
        self.pinned = {k: torch.tensor(a).pin_memory() for k, a in self.host.items()}
        self.gb = {k: t.to(dev) for k, t in self.pinned.items()}
        self.covered = int((self.host["mask"] > 0).sum())
        self.rays_per_pass = self.covered * 2 * N * N
        # trainable parameters: light probe + kd / ks textures in ONE flat bucket (parallel.GradBucket: parameters are views of
        # `flat`, their .grad views of `flat_grad`; a single all-reduce per step, hooked in front of optimizer.step)
        g = torch.Generator(device="cpu").manual_seed(2)
        lr_ = wl["light_res"]
        self.bucket = parallel.GradBucket([(lr_, lr_, 3), (tr * tr, 3), (tr * tr, 3)], dev)
        self.light_base, self.kd_tex, self.ks_tex = self.bucket.params
        self.n_light = n_light = lr_ * lr_ * 3
        n_tex = tr * tr * 3
        with torch.no_grad():
            if light_init == "hdr":      # the probe the optimisation converges to: the HDR environment box-filtered to the trainable resolution
                hdr = synth.hdr_light(wl["ref_light_hw"][0], wl["ref_light_hw"][1], seed=7)
                fy, fx = hdr.shape[0] // lr_, hdr.shape[1] // lr_
                self.light_base.copy_(torch.tensor(hdr[:lr_ * fy, :lr_ * fx].reshape(lr_, fy, lr_, fx, 3).mean((1, 3))).to(dev))
            else:                        # create_trainable_env_rnd, render/light.py:98-101 (train.py:536,612): U[0.25, 0.75)
                self.light_base.copy_((torch.rand(n_light, generator=g) * 0.5 + 0.25).view(lr_, lr_, 3).to(dev))
            self.kd_tex.copy_(torch.rand(n_tex, generator=g).view(tr * tr, 3).to(dev))
            ks0 = torch.rand(tr * tr, 3, generator=g); ks0[:, 0] = 0; ks0[:, 1] = 0.1 + 0.9 * ks0[:, 1]
            self.ks_tex.copy_(ks0.to(dev))
        self.flat, self.flat_grad = self.bucket.flat, self.bucket.flat_grad
        # torch.optim.Adam as in train.py:401-409; capturable so that the whole step can live in one CUDA graph
        self.optimizer = parallel.hook_optimizer(torch.optim.Adam(self.bucket.params, lr=wl.get("lr", 0.01), fused=True, capturable=True), self.bucket)
        self.lgt = EnvironmentLight(self.light_base)
        # the dataset side of a training iteration (dataset/dataset_mesh.py:95-110): every target image is rendered by the same hot
        # path, forward only, from the reference material (data/spot/metal.mtl: ks = (0, 0.2, 1)) under the native-resolution HDR probe
        with torch.no_grad():
            self.ref_lgt = EnvironmentLight(torch.tensor(synth.hdr_light(wl["ref_light_hw"][0], wl["ref_light_hw"][1], seed=7), device=dev))
            self.ref_kd = torch.rand(tr * tr, 3, generator=g).to(dev)
            self.ref_ks = torch.tensor([0.0, 0.2, 1.0], device=dev).expand(tr * tr, 3).contiguous()
        self.denoiser = BilateralDenoiser(influence=wl["sigma"] / 2.0)
        self.perms = torch.tensor(synth.make_perms(N, seed=3), device=dev)
        self.seed = torch.zeros(1, dtype=torch.int32, device=dev)        # render.py:19 `rnd_seed`, kept on the device (graph-capturable)
        self.bytes_h2d = sum(t.numel() * t.element_size() for t in self.pinned.values())
        self.graph = None
        self.last = {}

    def upload(self):
        for k, t in self.pinned.items():
            self.gb[k].copy_(t, non_blocking=True)

    # ---- one shade() call: render/render.py:99-131 ------------------------------------------------------------------------
    def shade(self, kd_tex, ks_tex, lgt, timers=None, keep=False, tag="fwd"):
        torch, ou, wl, gb = self.torch, self.ou, self.wl, self.gb
        import nvdiffrecmc_b200.renderutils as ru
        from nvdiffrecmc_b200.denoiser import _safe_normalize
        from nvdiffrecmc_b200.raster import texel_fetch
        N = wl["n_samples_x"]
        kd = texel_fetch(kd_tex, gb["texel"])                                        # material look-up (stand-in for dr.texture, nearest)
        ks = texel_fetch(ks_tex, gb["texel"])
        nrm = ru.prepare_shading_normal(gb["pos"], gb["view"], None, gb["smooth_nrm"], gb["tangent"], gb["geom_nrm"], two_sided_shading=True,
                                        opengl=True)                                 # render.py:99
        ro = gb["pos"] + nrm * 0.001                                                 # render.py:110
        self.seed += 1                                                               # render.py:116 (bumped on EVERY shade call, quirk 12)
        if timers is not None:
            timers[tag + "0"].record()
        diff, spec = ou.optix_env_shade(self.ctx, gb["mask"], ro, gb["pos"], nrm, gb["view"], kd, ks, lgt.base, lgt._pdf,
                                        lgt.rows[:, 0], lgt.cols, BSDF='pbr', n_samples_x=N, rnd_seed=self.seed, shadow_scale=1.0,
                                        perms=self.perms, batch_offset=self.offset)  # render.py:113-115
        if timers is not None:
            timers[tag + "1"].record()
        if keep:
            self.last = dict(ro=ro, nrm=nrm, kd=kd, ks=ks, diff=diff, spec=spec)
        zdz = torch.stack([gb["depth"], torch.full_like(gb["depth"], 0.01)], -1)
        return ou.denoise_and_combine(diff, spec, _safe_normalize(nrm), zdz, self.denoiser.sigma, kd, ks)   # render.py:119-127 (+ denoiser.py:28)

    def forward_backward(self, timers=None, keep=False):
        """dataset-side reference render (forward only, HDR probe) -> update_pdf -> LBVH rebuild -> shade() -> image loss -> backward."""
        torch, ou = self.torch, self.ou
        import nvdiffrecmc_b200.renderutils as ru
        if timers is not None:
            timers["ref0"].record()
        with torch.no_grad():
            target = self.shade(self.ref_kd, self.ref_ks, self.ref_lgt, timers, tag="rfwd")   # dataset_mesh.py:108-110 ('img' of the batch)
        if timers is not None:
            timers["ref1"].record()
        self.lgt.update_pdf()                                                        # train.py:422
        ou.optix_build_bvh(self.ctx, self.verts, self.tris, rebuild=1)               # dlmesh.py:50 (every iteration)
        shaded = self.shade(self.kd_tex, self.ks_tex, self.lgt, timers, keep)
        loss = ru.image_loss(shaded, target, loss='l1', tonemapper='log_srgb')       # train.py:57-58 ('logl1', the default loss)
        if timers is not None:
            timers["bwd0"].record()
        loss.backward()
        if timers is not None:
            timers["bwd1"].record()
        return loss

    def step(self, timers=None, keep=False):
        """One training iteration of the hot path (SURVEY 8d): forward_backward -> [N > 1: ONE all-reduce] -> Adam -> clamps.
        Returns the loss (device)."""
        torch = self.torch
        self.optimizer.zero_grad()                                                   # train.py:407-411 (routed to the bucket: one memset)
        loss = self.forward_backward(timers, keep)
        self.optimizer.step()                                                        # train.py:452; pre-hook: ONE all-reduce (SURVEY 8e)
        with torch.no_grad():
            self.flat[:self.n_light].clamp_(min=0.0)                                 # light.clamp_(min=0), train.py:460
            self.flat[self.n_light:].clamp_(0.0, 1.0)                                # material kd / ks ranges
        return loss

    # ---- the same step as ONE CUDA graph (SURVEY f3: launch-bound regime at batch/8 per GPU) -------------------------------------
    def capture(self):
        """Capture step() -- kernels, memsets, the NCCL all-reduce and the fused Adam -- into a CUDA graph.  Everything on the path is
        stream-ordered and allocation-free in steady state; the seed lives on the device.  Returns None on success, else the reason."""
        torch = self.torch
        try:
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(device=self.dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                      # warm the private pool / lazy initialisations on the capture stream
                    self.step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self.graph_loss = self.step()
            self.graph = g
            return None
        except Exception as e:                          # noqa: BLE001 -- reported in the JSON line, the bench falls back to eager
            self.graph = None
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
            return "%s: %s" % (type(e).__name__, str(e).splitlines()[0][:200])

    def run(self):
        if self.graph is not None:
            self.graph.replay()
            self.loss = self.graph_loss
        else:
            self.loss = self.step()
        return self.loss

    def dump_outputs(self, out_dir):
        """Save what the last run() handed its caller -- the loss, the updated trainable parameters (light probe, kd / ks textures)
        and their gradients -- as float32 `out_dir/<name>.npy` (~52 MB for the default workload)."""
        os.makedirs(out_dir, exist_ok=True)
        arrays = {"loss": self.loss.detach().reshape(1)}
        for i, (name, p) in enumerate(zip(("light", "kd_tex", "ks_tex"), self.bucket.params)):
            arrays[name] = p.detach()
            arrays[name + "_grad"] = self.flat_grad[self.bucket.offsets[i]:self.bucket.offsets[i + 1]].view(p.shape)
        for name, t in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def time_env_kernels(w, reps=20, warm=5, full=False, shadow_scale=1.0):
    """CUDA-event time of the fused env_shade forward launch (with the ray record, as the training step issues it) and of the
    replay backward launch ALONE: the C-ABI entry points are called directly on preallocated buffers, events on the launching
    stream (torch's current stream) immediately around each launch, so no allocator or autograd time is inside the brackets.
    Median of `reps` after `warm` untimed launches (SURVEY 8d: median of >= 20 after 5 warm-ups); a new seed (new rays) per launch."""
    import ctypes as C
    import torch
    import nvdiffrecmc_b200.renderutils as ru
    from nvdiffrecmc_b200 import _lib as L
    from nvdiffrecmc_b200.optixutils import ops
    gb, wl = w.gb, w.wl
    N = wl["n_samples_x"]
    with torch.no_grad():
        nrm = ru.prepare_shading_normal(gb["pos"], gb["view"], None, gb["smooth_nrm"], gb["tangent"], gb["geom_nrm"])
        ro = gb["pos"] + nrm * 0.001
        kd = w.kd_tex.detach()[gb["texel"]].contiguous(); ks = w.ks_tex.detach()[gb["texel"]].contiguous()
        light = w.lgt.base.detach().contiguous()
    B, H, W_ = ro.shape[:3]
    dev = ro.device
    slots = 2 * N * N
    d = ops._env_descs(gb["mask"], ro, gb["pos"], nrm, gb["view"], kd, ks, light, w.lgt._pdf, w.lgt.rows[:, 0], w.lgt.cols, w.perms)
    diff = torch.empty(B, H, W_, 3, device=dev); spec = torch.empty_like(diff)
    rec_cnt = torch.empty(B, H, W_, dtype=torch.int32, device=dev)
    rec_rays = torch.empty(B, H, W_, 5, slots, device=dev)
    g = [torch.empty(B, H, W_, 3, device=dev) for _ in range(4)]
    lg = torch.empty(light.shape[0], light.shape[1], 3, device=dev)
    gd = torch.ones_like(diff); gs = torch.ones_like(spec)
    dsc = [L.nhwc(gb["pos"]), L.nhwc(nrm), L.nhwc(gb["view"]), L.nhwc(kd), L.nhwc(ks), L.view_hwc(light)]
    dg, sg = L.nhwc(gd), L.nhwc(gs)
    lib, sp = L.lib(), L.stream_ptr()
    fw, bw = [], []
    for r in range(reps + warm):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        L.check(lib.mcs_env_shade_fwd(w.ctx.cpp_wrapper, *[C.byref(x) for x in d], 0, N, 1000 + r, None, float(shadow_scale), int(w.offset), diff.data_ptr(), spec.data_ptr(),
                                      None, rec_cnt.data_ptr(), rec_rays.data_ptr(), slots, sp), "optix_env_shade (forward)")
        e[1].record()
        e[2].record()
        L.check(lib.mcs_env_shade_bwd_replay(*[C.byref(x) for x in dsc], 0, N, float(shadow_scale), C.byref(dg), C.byref(sg), rec_cnt.data_ptr(), rec_rays.data_ptr(), slots,
                                             g[0].data_ptr(), g[1].data_ptr(), g[2].data_ptr(), g[3].data_ptr(), lg.data_ptr(), sp),
                "optix_env_shade (backward, ray-record replay)")
        e[3].record()
        torch.cuda.synchronize()
        if r >= warm:
            fw.append(e[0].elapsed_time(e[1])); bw.append(e[2].elapsed_time(e[3]))
    if full:
        return fw, bw
    return float(np.median(fw)), float(np.median(bw))


def verify_launch(w, seed=12345):
    """--verify (on by default, outside every timed region): parity of the bench's OWN launch configuration with the CPU oracle.
    The product runs the full [views, res, res] launch (forward, records, backward through the public op); the oracle recomputes view
    0's 64 x 64 centre crop plus ~2 k random covered pixels of all views (tests/parity_check.py).  Integer records must agree bit
    for bit; radiance and the five gradients within 1e-4 relative L2 (kernel.cu:463-542)."""
    import torch
    import nvdiffrecmc_b200.renderutils as ru
    from common import oracle
    from parity_check import env_shade_parity, select_pixels
    gb, wl = w.gb, w.wl
    N = wl["n_samples_x"]
    t0 = time.time()
    with torch.no_grad():
        nrm = ru.prepare_shading_normal(gb["pos"], gb["view"], None, gb["smooth_nrm"], gb["tangent"], gb["geom_nrm"], two_sided_shading=True, opengl=True)
        nrm = (nrm * (gb["mask"][..., None] > 0)).contiguous()
        ro = (gb["pos"] + nrm * 0.001).contiguous()
        kd = w.kd_tex.detach()[gb["texel"]].contiguous(); ks = w.ks_tex.detach()[gb["texel"]].contiguous()
        w.lgt.update_pdf()
        dev_in = dict(mask=gb["mask"], ro=ro, pos=gb["pos"], nrm=nrm, view=gb["view"], kd=kd, ks=ks, light=w.lgt.base.detach().contiguous(),
                      pdf=w.lgt._pdf, rows=w.lgt.rows[:, 0].contiguous(), cols=w.lgt.cols)
        # the non-recording forward launch exactly as step() issues it (MODE 0 + ray record)
        lt = dev_in["light"].clone().requires_grad_(True)
    d0, s0 = w.ou.optix_env_shade(w.ctx, gb["mask"], ro, gb["pos"], nrm, gb["view"], kd, ks, lt, dev_in["pdf"], dev_in["rows"], dev_in["cols"],
                                  BSDF='pbr', n_samples_x=N, rnd_seed=seed, shadow_scale=1.0, perms=w.perms, batch_offset=w.offset)
    o = oracle()
    scene = o.scene(*w.mesh)
    mask = gb["mask"].cpu().numpy()
    sel = select_pixels(mask, crop=64, n_random=2048, seed=7)
    r = env_shade_parity(w.ctx, scene, dev_in, w.perms, N, sel, bsdf="pbr", seed=seed, batch_offset=w.offset, bench_fwd=(d0.detach(), s0.detach()))
    r["launch"] = "%d x %d x %d, n_samples_x=%d, batch_offset=%d" % (w.B, wl["res"], wl["res"], N, w.offset)
    r["tolerance_rel_l2"] = 1e-4
    r["ok"] = bool(r["texel_mismatch"] == 0 and r["vis_mismatch"] == 0 and r["max_rel_l2"] <= 1e-4)
    r["seconds"] = round(time.time() - t0, 1)
    return r


def traced_fraction(w):
    """Share of the logical rays (covered px x 2N^2) that the kernel actually traces, and that are visible: rays with n.wi <= 0
    contribute exactly zero and are skipped (rec_vis == 2).  Counted on the full launch with the records entry point."""
    import torch
    import nvdiffrecmc_b200.renderutils as ru
    from nvdiffrecmc_b200.optixutils.ops import env_shade_records
    gb, wl = w.gb, w.wl
    N = wl["n_samples_x"]
    with torch.no_grad():
        nrm = ru.prepare_shading_normal(gb["pos"], gb["view"], None, gb["smooth_nrm"], gb["tangent"], gb["geom_nrm"])
        ro = gb["pos"] + nrm * 0.001
        kd = w.kd_tex.detach()[gb["texel"]]; ks = w.ks_tex.detach()[gb["texel"]]
        d, s, rt, rv = env_shade_records(w.ctx, gb["mask"], ro, gb["pos"], nrm, gb["view"], kd, ks, w.lgt.base.detach(), w.lgt._pdf,
                                         w.lgt.rows[:, 0], w.lgt.cols, w.perms, n_samples_x=N, rnd_seed=0, batch_offset=w.offset)
        cov = gb["mask"] > 0
        n_cov = int(cov.sum()) * 2 * N * N
        traced = int(((rv != 2) & cov[..., None]).sum()); visible = int(((rv == 1) & cov[..., None]).sum())
    return traced / max(n_cov, 1), visible / max(n_cov, 1)


def traversal_counts(wl, sample_res=64):
    """n_nodes / n_tris per ray of the CANONICAL CPU traversal (oracle LBVH, SURVEY 8d) on a pixel subsample of view 0."""
    from common import oracle
    from nvdiffrecmc_b200 import synth
    o = oracle()
    v, f, vn = build_scene_numpy(wl, 0)
    scene = o.scene(v, f)
    ang, tilt = view_pose(0)
    campos, ro, rd = synth.primary_rays(synth.orbit_view(ang, tilt=tilt), sample_res)
    tid, tuv = scene.closest_hit(ro.reshape(-1, 3), rd.reshape(-1, 3))
    g = synth.assemble_gbuffer(v, f, vn, tid.reshape(sample_res, sample_res), tuv.reshape(sample_res, sample_res, 3), campos, seed=100)
    view = g["view_pos"].reshape(1, 1, 1, 3)
    nrm = o.prepare_shading_normal(g["pos"][None], view, None, g["smooth_nrm"][None], g["tangent"][None], g["geom_nrm"][None])
    ro_s = g["pos"][None] + nrm * np.float32(0.001)
    light = synth.random_light(wl["light_res"], seed=2)
    pdf, rows, cols = o.update_pdf(light)
    N = wl["n_samples_x"]
    perms = synth.make_perms(N, seed=3, rows=1024)
    t0 = time.time()
    d, s, cnt = o.env_shade(scene, g["mask"][None], ro_s, g["pos"][None], nrm, view, g["kd"][None], g["ks"][None], light, pdf, rows, cols, perms,
                            n_samples_x=N, rnd_seed=0, vis_mode="bvh", counters=True)
    dt = time.time() - t0
    rays = float(cnt[0])
    return dict(nodes_per_ray=float(cnt[1]) / rays, tris_per_ray=float(cnt[2]) / rays, rays=int(rays), seconds=dt,
                sample="candidate view 0 at %dx%d, n_samples_x=%d" % (sample_res, sample_res, N))


# ------------------------------------------------------------------------------------------------
def cpu_reference(o):
    """(object with env_shade / bilateral_fwd / bilateral_bwd, kind): the reference's own raygen program and denoiser kernels compiled for
    the host (oracle/_ref, built where /root/reference exists and shipped as a prebuilt library) when available, else the oracle port."""
    try:
        from oracle import Reference
        return Reference(o), "reference"
    except Exception:
        return o, "port"


def cpu_reference_step(o, case, N, sigma, seed, env_shade=None):
    """The same hot-path step on the host CPUs (all OpenMP threads): env_shade forward + backward through `env_shade` (the compiled
    reference or the oracle port), LBVH rebuild / shading normal / denoiser / update_pdf through the oracle port."""
    c = case
    impl = env_shade if env_shade is not None else o
    es = impl.env_shade
    scene = o.scene(c["verts"], c["tris"])                                       # LBVH rebuild every iteration
    nrm = o.prepare_shading_normal(c["pos"], c["view"], None, c["smooth_nrm"], c["tangent"], c["geom_nrm"])
    ro = (c["pos"] + nrm * np.float32(0.001)).astype(np.float32)
    zdz = np.stack([c["depth"], np.full_like(c["depth"], 0.01)], -1)
    nn = nrm / np.maximum(np.linalg.norm(nrm, axis=-1, keepdims=True), 1e-20)
    if "ref_light" in c:                                                          # dataset-side reference render (dataset_mesh.py:108-110)
        rargs = (scene, c["mask"], ro, c["pos"], nrm, c["view"], c["ref_kd"], c["ref_ks"], c["ref_light"], c["ref_pdf"], c["ref_rows"], c["ref_cols"],
                 c["perms"])
        rd_, rs_ = es(*rargs, n_samples_x=N, rnd_seed=seed + 7919, vis_mode="bvh")
        impl.bilateral_fwd(rd_, nn, zdz, sigma); impl.bilateral_fwd(rs_, nn, zdz, sigma)
    pdf, rows, cols = o.update_pdf(c["light"])
    args = (scene, c["mask"], ro, c["pos"], nrm, c["view"], c["kd"], c["ks"], c["light"], pdf, rows, cols, c["perms"])
    d, s = es(*args, n_samples_x=N, rnd_seed=seed, vis_mode="bvh")
    fd, fs = impl.bilateral_fwd(d, nn, zdz, sigma), impl.bilateral_fwd(s, nn, zdz, sigma)
    gd = np.concatenate([np.ones_like(d) / fd[..., 3:], np.zeros_like(fd[..., 3:])], -1)
    cd, cs = impl.bilateral_bwd(nn, zdz, sigma, gd), impl.bilateral_bwd(nn, zdz, sigma, gd)
    if impl is o:
        g = es(*args, n_samples_x=N, rnd_seed=seed, vis_mode="bvh", grads=(cd, cs), parallel_bwd=True)
    else:
        g = es(*args, n_samples_x=N, rnd_seed=seed, vis_mode="bvh", grads=(cd, cs))
    o.prepare_shading_normal_bwd(c["pos"], c["view"], None, c["smooth_nrm"], c["tangent"], c["geom_nrm"], g[1])
    return float(d.sum())


def cpu_case(o, wl, res_s):
    """Bounded sample of the bench workload for the CPU legs: 1 view at res_s^2 of the same mesh / probes / n_samples_x."""
    from common import make_case
    from nvdiffrecmc_b200 import synth
    N = wl["n_samples_x"]
    case = make_case(res=res_s, B=1, N=N, mesh=wl["mesh"], level=wl["mesh_level"], light="random", light_hw=(wl["light_res"], wl["light_res"]),
                     perm_rows=4096)
    hdr = synth.hdr_light(wl["ref_light_hw"][0], wl["ref_light_hw"][1], seed=7)
    case["ref_light"] = hdr
    case["ref_pdf"], case["ref_rows"], case["ref_cols"] = o.update_pdf(hdr)        # the dataset's probe: pdf built once at load (light.py:82-84)
    case["ref_kd"] = np.random.default_rng(11).uniform(0, 1, size=case["kd"].shape).astype(np.float32) * (case["mask"][..., None] > 0)
    case["ref_ks"] = (np.broadcast_to(np.float32([0.0, 0.2, 1.0]), case["ks"].shape) * (case["mask"][..., None] > 0)).astype(np.float32)
    return case


REF_SAMPLE_RES = 128


def make_config(wl, views, world):
    """`config` of the JSON line -- identical for the product arm and the `--impl reference` arm (everything in it follows from the
    workload definition; measured quantities go to `workload_measured`)."""
    N, res, lr, tr = wl["n_samples_x"], wl["res"], wl["light_res"], wl["tex_res"]
    bucket_mb = (lr * lr * 3 + 2 * tr * tr * 3) * 4 / 1e6
    gbuf_mb = views * (res * res * 64 + 12) / 1e6          # mask 4 + pos / smooth_nrm / tangent / geom_nrm 12 each + depth 4 + texel index 8 B per pixel
    return {"workload": wl["name"], "views_per_gpu": views, "global_views": views * world, "res": res, "n_samples_x": N,
            "rays_per_covered_pixel": 2 * N * N,
            "step": "dataset reference render (fwd only, %dx%d HDR probe, metal material; dataset_mesh.py:108-110) -> update_pdf -> LBVH rebuild -> "
                    "shade (texel fetch, shading normal, env_shade, fused denoise + recombine) -> log-sRGB L1 loss -> backward -> all-reduce -> Adam + clamps"
                    % (wl["ref_light_hw"][0], wl["ref_light_hw"][1]),
            "trainable_probe": "%dx%d U[0.25,0.75) (create_trainable_env_rnd, light.py:98-101); the HDR-initialised probe is in `hdr_probe`" % (lr, lr),
            "parallelism": "dp%d over views (coverage-balanced deal of the global batch), one NCCL all-reduce of the flat gradient bucket (%.1f MB) via "
                           "parallel.GradBucket + hook_optimizer" % (world, bucket_mb),
            "l2_policy": "per-step inputs (G-buffer %.0f MB + intermediates) exceed the 126 MB L2" % gbuf_mb,
            "reference_arm_sampling": "`--impl reference` times the same step on the host cores on a BOUNDED SAMPLE of this workload (1 view at %dx%d of the "
                                      "same scene, probes, n_samples_x, sigma) and reports the size-normalised Mrays/s; its ms_per_step is per sample step"
                                      % (REF_SAMPLE_RES, REF_SAMPLE_RES)}


PASSES = 3      # env_shade passes per training iteration as the reference runs it: dataset reference render (fwd), shade fwd, shade bwd (re-trace)


def host_cores():
    """CPU threads this process may actually use (cgroup / affinity aware), also exported to OpenMP."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:                                   # cgroup v2 cpu quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(n)          # torchrun exports 1; the oracle legs also call Oracle.set_threads(n)
    return n


REF_ARM_NOTE = {
    "reference": "env_shade forward + backward and the bilateral denoiser forward + backward = the reference's own kernels (render/optixutils/c_src/"
                 "envsampling/kernel.cu with bsdf.h, math_utils.h; denoising.cu) compiled for the host cores (oracle/_ref, OpenMP over pixels), shadow "
                 "rays answered by the oracle's LBVH (OptiX itself is closed source and needs an RT driver); shading normal / update_pdf / LBVH build "
                 "= oracle C port",
    "port": "CPU oracle port of kernel.cu/denoising.cu/normal.cu (oracle/_ref not available on this machine; OptiX needs libnvoptix + RT driver)",
}


SM_COUNT, SMSP_PER_SM, LANES = 148, 4, 32


def config_key(wl, views):
    return "%dx%dx%d_n%d_%s%s_light%d" % (views, wl["res"], wl["res"], wl["n_samples_x"], wl["mesh"], wl["mesh_level"], wl["light_res"])


def dominant_kernel_profile(wl, views):
    """Committed ncu --set full capture of env_shade_kernel<0> FOR THIS CONFIG (profiles/r02_dominant_kernel.json, written by
    tools/ncu_summary.py from the .ncu-rep of `tools/kbench.py`): thread-instructions, warp-instructions, DRAM bytes per launch and the
    rays of the captured launch.  None when no capture of this exact configuration is committed -- never a number from another config."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_dominant_kernel.json")) as f:
            return json.load(f)["configs"].get(config_key(wl, views))
    except Exception:
        return None


def run_reference(args, wl):
    """--impl reference: the reference's algorithm on the host CPUs (compiled reference kernels / oracle port; OptiX cannot run here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    from common import oracle
    o = oracle()
    cores = o.set_threads(cores)
    es, kind = cpu_reference(o)
    N, res_s = wl["n_samples_x"], REF_SAMPLE_RES
    case = cpu_case(o, wl, res_s)
    covered = int((case["mask"] > 0).sum())
    rays_step = covered * 2 * N * N * PASSES
    for i in range(args.warmup):
        cpu_reference_step(o, case, N, wl["sigma"], i, es)
    t0 = time.time()
    for i in range(args.steps):
        cpu_reference_step(o, case, N, wl["sigma"], 100 + i, es)
    dt = (time.time() - t0) / args.steps
    val = rays_step / dt / 1e6
    sample = "1 view at %dx%d of the same scene (same mesh, probes, n_samples_x=%d, sigma=%g): %d rays/step" % (res_s, res_s, N, wl["sigma"], rays_step)
    emit({
        "impl": "reference", "metric": "shadow_rays_per_second_train_step", "value": round(val, 4), "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(wl, wl["views_per_gpu"], max(int(args.gpus), 1)),
        "reference_arm": REF_ARM_NOTE[kind],
        "reference_sample": "BOUNDED SAMPLE, not the full workload: " + sample + "; Mrays/s is size-normalised, ms_per_step is per SAMPLE step",
        "cpu_baseline": {"value": round(val, 4), "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(val, 4), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "iters_per_s_on_sample": round(1.0 / dt, 4),
    })


# ------------------------------------------------------------------------------------------------
_STDOUT_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner when NCCL_DEBUG is set, torchrun
    notices), so everything but the final line is routed to stderr at the file-descriptor level."""
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)


def finish(world):
    """End the run.  One process: return, so the interpreter shuts down normally (exit handlers run, libraries are unloaded).
    Several ranks: leave without tearing down NCCL communicators / captured graphs -- with the all-reduce captured inside CUDA graphs,
    `destroy_process_group()` was observed to block for minutes after the result line had been printed (rank 0 works alone on the
    parity / CPU legs long after the other ranks are done).  All results are flushed; the OS reclaims the rest."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)


def emit(obj):
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(obj))
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(2, 1)                  # whatever is printed while the process shuts down stays off the result line's stream


def timed_loop(w, steps, barrier, torch):
    """EXACTLY `steps` steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        w.run()
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def max_over_ranks(ms, world, dev, torch, dist):
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def sum_over_ranks(x, world, dev, torch, dist):
    t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t)


def dp_gradient_check(ws, wl, rank, world, dev, torch, dist):
    """N > 1 (VERDICT r1 item 6): the all-reduced gradient bucket of the data-parallel step equals the single-process gradient of the
    CONCATENATED global batch (contract: image loss = mean over B*H*W, renderutils/ops.py:494; equal shards => mean of local means).
    Every rank runs forward + backward on its shard with the same seed and parameters and all-reduces through parallel.GradBucket;
    rank 0 then renders all views alone.  Light-gradient and texture-scatter atomics reorder, hence 1e-5, not bit-equality."""
    seed0 = 4242
    ws.seed.fill_(seed0)
    ws.bucket.zero_grad()
    loss = ws.forward_backward()
    ws.bucket.all_reduce_mean()
    torch.cuda.synchronize()
    got = ws.flat_grad.clone()
    out = None
    if rank == 0:
        full = GpuWorkload(wl, 0, 1, dev, views=ws.B * world, global_views=ws.global_views)
        with torch.no_grad():
            full.flat.copy_(ws.flat)
        full.seed.fill_(seed0)
        full.bucket.zero_grad()
        full.forward_backward()
        full.bucket.sync_views()
        torch.cuda.synchronize()
        ref = full.flat_grad
        nl, nt = ws.n_light, (ws.flat.numel() - ws.n_light) // 2
        rl = lambda a, b: float((a - b).double().norm() / b.double().norm().clamp_min(1e-30))
        out = {"global_batch": ws.B * world, "views_per_rank": ws.B,
               "rel_l2": {"light": float("%.3e" % rl(got[:nl], ref[:nl])), "kd_tex": float("%.3e" % rl(got[nl:nl + nt], ref[nl:nl + nt])),
                          "ks_tex": float("%.3e" % rl(got[nl + nt:], ref[nl + nt:]))}, "tolerance": 1e-5}
        out["ok"] = bool(max(out["rel_l2"].values()) <= 1e-5)
        del full
    if world > 1:
        dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mcshade", choices=["mcshade", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: views_per_gpu fixed (default, the driver's scaling run); strong: global batch fixed at 8 views. The default line carries "
                         "the strong-scaling numbers as a sub-record either way")
    ap.add_argument("--no-verify", action="store_true", help="skip the parity leg (on by default, outside the timed regions)")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of replaying one CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling and HDR-probe sub-records (debug)")
    ap.add_argument("--views", type=int, default=None, help="override views per GPU (debug)")
    ap.add_argument("--res", type=int, default=None, help="override resolution (debug)")
    ap.add_argument("--n", type=int, default=None, help="override n_samples_x (debug)")
    ap.add_argument("--mesh", default=None, help="override mesh: blob | blob+torus | full | bob-like | grid1m (debug)")
    ap.add_argument("--level", type=int, default=None, help="override icosphere subdivision level (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save the loss, parameters and gradients of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the outputs of the GPU step; the reference arm has none to save")
    quiet_stdout()
    wl = dict(WORKLOAD)
    if args.views:
        wl["views_per_gpu"] = args.views
    if args.res:
        wl["res"] = args.res
    if args.n:
        wl["n_samples_x"] = args.n
    if args.mesh:
        wl["mesh"] = args.mesh
    if args.level is not None:
        wl["mesh_level"] = args.level
    if args.views or args.res or args.n or args.mesh or args.level is not None:
        wl["name"] = "DEBUG OVERRIDE of " + wl["name"]
    if args.impl == "reference":
        return run_reference(args, wl)

    os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")     # the NCCL watchdog must not query events while a graph is captured
    import torch
    import torch.distributed as dist
    from nvdiffrecmc_b200 import _lib
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback for the product path)"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()
    N = wl["n_samples_x"]
    gbs = wl["global_batch_strong"]
    strong_ok = gbs % world == 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(w, steps, warmup, use_graph):
        """warm-up (eager) -> optional graph capture -> timed loop.  Returns (ms over `steps`, launches per step, graph status)."""
        _lib.LAUNCHES.clear()
        w.step()
        per_step = sum(_lib.LAUNCHES.values())
        for _ in range(max(warmup - 1, 0)):
            w.step()
        barrier()
        status = "disabled (--no-graph)"
        if use_graph:
            why = w.capture()
            # every rank must agree, or the ranks would issue different collectives
            bad = sum_over_ranks(0.0 if why is None else 1.0, world, dev, torch, dist)
            if bad > 0:
                w.graph = None
                status = "capture failed -> eager: %s" % (why or "on another rank")
            else:
                status = "one graph per step (kernels + memsets + NCCL all-reduce + fused Adam)" if world > 1 else "one graph per step (kernels + memsets + fused Adam)"
                for _ in range(2):
                    w.run()
        barrier()
        ms = timed_loop(w, steps, barrier, torch)
        return max_over_ranks(ms, world, dev, torch, dist), per_step, status

    # ---- main measurement: device-resident throughput (value) ---------------------------------
    main_views = wl["views_per_gpu"] if args.scaling == "weak" else gbs // world
    assert args.scaling == "weak" or strong_ok, "strong scaling needs a world size that divides the global batch of %d" % gbs
    w = GpuWorkload(wl, rank, world, dev, views=main_views)
    torch.cuda.synchronize()
    clk = ClockSampler(local).start()
    _lib.LAUNCHES.clear()
    w.step()
    launches_per_step = sum(_lib.LAUNCHES.values())
    for _ in range(args.warmup - 1):
        w.step()
    barrier()
    graph_status = "disabled (--no-graph)"
    if not args.no_graph:
        why = w.capture()
        bad = sum_over_ranks(0.0 if why is None else 1.0, world, dev, torch, dist)
        if bad > 0:
            w.graph = None
            graph_status = "capture failed -> eager: %s" % (why or "on another rank")
        else:
            graph_status = "one CUDA graph per step (all kernels, memsets, %sfused Adam)" % ("the NCCL all-reduce, " if world > 1 else "")
            for _ in range(2):
                w.run()
    barrier()
    clk.begin()
    ms = timed_loop(w, args.steps, barrier, torch)
    clk.end()
    clk.close()
    if args.dump_outputs and rank == 0:
        w.dump_outputs(args.dump_outputs)
    ms_step = max_over_ranks(ms, world, dev, torch, dist) / args.steps
    rays_pass_all = sum_over_ranks(w.rays_per_pass, world, dev, torch, dist)
    rays_min = -max_over_ranks(-float(w.rays_per_pass), world, dev, torch, dist)
    rays_max = max_over_ranks(float(w.rays_per_pass), world, dev, torch, dist)
    total_rays_step = rays_pass_all * PASSES
    value = total_rays_step / (ms_step * 1e-3) / 1e6
    launches = launches_per_step * args.steps

    # ---- breakdown: a few EAGER steps with events between the phases (not part of `value`) -----
    names = ["ref0", "ref1", "rfwd0", "rfwd1", "fwd0", "fwd1", "bwd0", "bwd1"]
    timers = [{n: torch.cuda.Event(enable_timing=True) for n in names} for _ in range(3)]
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w.step()                      # graph capture emptied the allocator cache: let the eager path re-acquire its blocks first
    barrier()
    es0.record()
    for t in timers:
        w.step(t)
    es1.record()
    barrier()
    eager_ms_step = max_over_ranks(es0.elapsed_time(es1), world, dev, torch, dist) / len(timers)
    med = lambda a, b: float(np.median([t[a].elapsed_time(t[b]) for t in timers]))
    ref_ms, rfwd_ms, fwd_ms, bwd_all_ms = med("ref0", "ref1"), med("rfwd0", "rfwd1"), med("fwd0", "fwd1"), med("bwd0", "bwd1")

    # ---- end to end through the public API with HOST inputs (e2e) ----------------------------
    # Every step uploads ITS G-buffer from pinned host memory and reads ITS loss + parameter gradients back, all inside the timed
    # region.  The upload of step i+1 runs on a copy stream while step i computes (two device buffer sets, event-ordered), the
    # way a training loop with a prefetching data loader behaves.  Eager launches (the graph is bound to one buffer set).
    copy_stream = torch.cuda.Stream(device=dev)
    sets = [w.gb, {k: torch.empty_like(t) for k, t in w.gb.items()}]
    up_done = [torch.cuda.Event() for _ in range(2)]
    use_done = [torch.cuda.Event() for _ in range(2)]
    host_out = torch.empty(w.flat_grad.numel() + 1, pin_memory=True)

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(use_done[slot])          # the step that last used this buffer set has finished
            for k, t in w.pinned.items():
                sets[slot][k].copy_(t, non_blocking=True)
            up_done[slot].record(copy_stream)

    def e2e_loop(n):
        for i in range(2):
            use_done[i].record()
        upload(0)
        for i in range(n):
            slot = i & 1
            if i + 1 < n:
                upload(slot ^ 1)                             # prefetch the next step's inputs
            torch.cuda.current_stream().wait_event(up_done[slot])
            w.gb = sets[slot]
            loss = w.step()
            use_done[slot].record()
            host_out[:1].copy_(loss.detach().reshape(1), non_blocking=True)      # device -> host: loss + parameter gradients
            host_out[1:].copy_(w.flat_grad, non_blocking=True)

    e2e_loop(2)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    e2e_loop(args.steps)
    e3.record()
    barrier()
    w.gb = sets[0]
    del sets
    e2e_ms_step = max_over_ranks(e2.elapsed_time(e3), world, dev, torch, dist) / args.steps
    e2e_value = total_rays_step / (e2e_ms_step * 1e-3) / 1e6

    # ---- sub-records: strong scaling (global batch fixed at 8 views) and the HDR-initialised probe ------------------------------
    strong = hdr = dp_check = None
    if not args.no_extras:
        if args.scaling == "strong" or (world == 1 and main_views == gbs):
            strong = {"global_batch": gbs, "views_per_gpu": main_views, "ms_per_step": round(ms_step, 3), "train_iters_per_s": round(1e3 / ms_step, 3),
                      "cuda_graph": graph_status, "same_run_as": "value"}
            ws = w
        elif strong_ok:
            ws = GpuWorkload(wl, rank, world, dev, views=gbs // world)
            s_ms, _, s_status = measure(ws, args.steps, args.warmup, not args.no_graph)
            s_ms /= args.steps
            strong = {"global_batch": gbs, "views_per_gpu": gbs // world, "ms_per_step": round(s_ms, 3), "train_iters_per_s": round(1e3 / s_ms, 3),
                      "cuda_graph": s_status,
                      "rays_per_pass_min_max_over_ranks": [int(-max_over_ranks(-float(ws.rays_per_pass), world, dev, torch, dist)),
                                                           int(max_over_ranks(float(ws.rays_per_pass), world, dev, torch, dist))],
                      "mrays_per_s": round(sum_over_ranks(ws.rays_per_pass, world, dev, torch, dist) * PASSES / (s_ms * 1e-3) / 1e6, 2)}
        else:
            ws = None
        if world > 1 and ws is not None and not args.no_verify:
            dp_check = dp_gradient_check(ws, wl, rank, world, dev, torch, dist)
        if ws is not None and ws is not w:
            del ws
        # trainable probe initialised from the box-filtered HDR environment: sun texel => light_grad atomics hot spot, peaked CDF
        wh = GpuWorkload(wl, rank, world, dev, views=main_views, light_init="hdr", global_views=w.global_views)
        h_steps = max(3, args.steps // 2)
        h_ms, _, h_status = measure(wh, h_steps, args.warmup, not args.no_graph)
        h_ms /= h_steps
        hdr = {"light_init": "256^2 box-filtered synth.hdr_light(1024, 2048) (sun at ~900x the sky)", "steps": h_steps, "ms_per_step": round(h_ms, 3),
               "train_iters_per_s": round(1e3 / h_ms, 3), "value": round(total_rays_step / (h_ms * 1e-3) / 1e6, 2), "cuda_graph": h_status}
        if rank == 0:
            hk_fwd, hk_bwd = time_env_kernels(wh)
            hdr["env_shade_fwd_kernel_ms"], hdr["env_shade_bwd_kernel_ms"] = round(hk_fwd, 3), round(hk_bwd, 3)
        del wh
        barrier()

    if rank != 0:
        return finish(world)

    # ---- rank 0: parity of this launch configuration, roofline of the dominant kernel, CPU baseline -----------------------------
    parity = None
    if not args.no_verify:
        try:
            parity = verify_launch(w)
        except Exception as e:      # noqa: BLE001 -- a failing checker must show up in the line, not kill the measurement
            parity = {"ok": False, "error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    k_fwd_ms, k_bwd_ms = time_env_kernels(w)
    hbm, hbm_src = peaks()
    tc = traversal_counts(wl)
    tfrac, vfrac = traced_fraction(w)
    sm_mhz = (clk.summary().get("sm_mhz") or 1965.0)
    issue_peak = SM_COUNT * SMSP_PER_SM * LANES * sm_mhz * 1e6 / 1e12           # T thread-instructions / s at the clock measured under load
    prof = dominant_kernel_profile(wl, main_views)
    # SURVEY 8d contract model:  A_ray = P/(2N^2) + 4 [perms] + 16 [light texel + pdf] + 44 [CDF probes] + 32*nodes + 36*tris
    a_fwd = 88.0 / (2 * N * N) + 4 + 16 + 44 + 32 * tc["nodes_per_ray"] + 36 * tc["tris_per_ray"]
    a_bwd = 136.0 / (2 * N * N) + vfrac * (20 + 12 + 12)
    contract_fwd = a_fwd * w.rays_per_pass / (k_fwd_ms * 1e-3) / 1e9
    roof = {"kernel": "env_shade_kernel<0> (fused env sampling + shadow rays + BSDF, forward; two launches per step)",
            "share_of_step_pct": round(100 * (rfwd_ms + fwd_ms) / eager_ms_step, 1),
            "kernel_ms": round(k_fwd_ms, 3), "rays_per_launch": w.rays_per_pass,
            "mrays_per_s_logical": round(w.rays_per_pass / k_fwd_ms / 1e3, 1), "mrays_per_s_traced": round(w.rays_per_pass * tfrac / k_fwd_ms / 1e3, 1),
            "traced_fraction": round(tfrac, 4), "visible_fraction": round(vfrac, 4)}
    if prof is not None:
        scale = w.rays_per_pass / float(prof["rays_per_launch"])                  # same config: ~1 (coverage of the captured launch)
        tinst = float(prof["thread_inst_per_launch"]) * scale
        ach = tinst / (k_fwd_ms * 1e-3) / 1e12
        dram = float(prof["dram_bytes_per_launch"]) * scale
        roof.update({"bound": "issue", "achieved": round(ach, 3), "peak": round(issue_peak, 2), "unit": "T thread-inst/s", "frac": round(ach / issue_peak, 4),
                     "peak_source": "148 SM x 4 SMSP x 32 lanes x %.0f MHz (SM clock sampled during the timed region)" % sm_mhz,
                     "traffic": int(dram), "frac_dram": round(dram / (k_fwd_ms * 1e-3) / 1e9 / hbm, 4), "dram_peak_gbs": hbm, "dram_peak_source": hbm_src,
                     "thread_inst_per_traced_ray": round(tinst / max(w.rays_per_pass * tfrac, 1), 1),
                     "active_lanes_per_instruction": prof.get("lanes_per_inst"), "issue_active_pct": prof.get("issue_active_pct"),
                     "profile": prof.get("source")})
    else:
        roof.update({"bound": "issue", "achieved": None, "peak": round(issue_peak, 2), "unit": "T thread-inst/s", "frac": None, "traffic": None,
                     "frac_dram": None, "note_profile": "no committed ncu capture of config %s (profiles/r02_dominant_kernel.json)" % config_key(wl, main_views)})
    roof["contract"] = {"bound": "hbm", "model": "SURVEY 8d LOGICAL bytes: every CDF probe, texel, canonical-LBVH node and triangle counted as a memory access",
                        "algorithmic_bytes_per_ray": round(a_fwd, 1), "achieved_gbs": round(contract_fwd, 1), "peak_gbs": hbm,
                        "frac_logical": round(contract_fwd / hbm, 4), "canonical_traversal": tc,
                        "note": "not a physical fraction: the tables of this scene (<1 MB nodes+triangles, 1.3 MB probe) are L1/L2 resident, the kernel walks a "
                                "4-wide quantised tree (~14 visits/ray instead of the canonical ~48 binary nodes) and skips rays with n.wi<=0; the physical "
                                "limiter is instruction issue (bound/achieved/peak above) and DRAM traffic is `traffic`"}
    roof["backward"] = {"kernel": "env_shade_replay_kernel (ray-record replay: adjoint BSDF + gradient scatter only)", "kernel_ms": round(k_bwd_ms, 3),
                        "algorithmic_bytes_per_ray": round(a_bwd, 1), "achieved_gbs": round(a_bwd * w.rays_per_pass / (k_bwd_ms * 1e-3) / 1e9, 1)}

    cpu = None
    if not args.no_cpu_baseline:
        ncores = host_cores()
        from common import oracle
        o = oracle()
        ncores = o.set_threads(ncores)
        es, kind = cpu_reference(o)
        res_s = 96
        case = cpu_case(o, wl, res_s)
        cov = int((case["mask"] > 0).sum())
        cpu_reference_step(o, case, N, wl["sigma"], 0, es)
        t0 = time.time(); reps = 2
        for i in range(reps):
            cpu_reference_step(o, case, N, wl["sigma"], 1 + i, es)
        dt = (time.time() - t0) / reps
        cpu = {"value": round(cov * 2 * N * N * PASSES / dt / 1e6, 4), "unit": "Mrays/s", "cores": ncores, "kind": kind,
               "sample": "same step on 1 view at %dx%d (%d rays/step), OpenMP; %s" % (res_s, res_s, cov * 2 * N * N * PASSES, REF_ARM_NOTE[kind])}

    traced_per_step = rays_pass_all * 2 * tfrac            # two traced passes: reference render + shade forward (backward replays the record)
    out = {
        "metric": "shadow_rays_per_second_train_step", "value": round(value, 2), "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": make_config(wl, main_views, world),
        "workload_measured": {"covered_pixels_rank0": w.covered, "coverage_rank0": round(w.covered / (main_views * wl["res"] ** 2), 4),
                              "rays_per_pass_min_max_over_ranks": [int(rays_min), int(rays_max)], "h2d_bytes_per_step": int(w.bytes_h2d)},
        "rays_counted": "covered px x 2N^2 per pass x %d passes, as the reference traces them (dataset reference render, shade forward, shade backward re-trace); "
                        "here the two forward passes trace (skipping rays with n.wi<=0, exactly-zero contribution) and the backward replays the forward's ray record: "
                        "see value_traced" % PASSES,
        "value_traced": round(traced_per_step / (ms_step * 1e-3) / 1e6, 2),
        "value_traced_note": "shadow rays actually traversed through the BVH per second over the whole step (Mrays/s)",
        "train_iters_per_s": round(1e3 / ms_step, 3),
        "cuda_graph": graph_status,
        "eager_ms_per_step": round(eager_ms_step, 3),
        "breakdown_ms": {"reference_render": round(ref_ms, 3), "reference_render_env_shade": round(rfwd_ms, 3), "env_shade_fwd": round(fwd_ms, 3), "backward_all": round(bwd_all_ms, 3),
                         "env_shade_fwd_kernel": round(k_fwd_ms, 3), "env_shade_bwd_kernel": round(k_bwd_ms, 3), "source": "eager steps with events between phases"},
        "strong": strong,
        "hdr_probe": hdr,
        "parity": parity,
        "dp_gradient_check": dp_check,
        "e2e": {"value": round(e2e_value, 2), "unit": "Mrays/s", "ms_per_step": round(e2e_ms_step, 3), "h2d_bytes_per_step": int(w.bytes_h2d),
                "d2h_bytes_per_step": int(host_out.numel() * 4), "train_iters_per_s": round(1e3 / e2e_ms_step, 3)},
        "gpu_launches": int(launches),
        "gpu_launches_per_step": int(launches_per_step),
        "ray_record_bytes": int(main_views * wl["res"] ** 2 * (2 * N * N * 20 + 4)),
        "clocks": clk.summary(),
        "roofline": roof,
        "cpu_baseline": cpu,
    }
    emit(out)
    finish(world)


if __name__ == "__main__":
    main()
