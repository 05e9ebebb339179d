"""Developer tool: CUDA-event timings of the secondary kernels against their rooflines (SURVEY 8d): the renderutils streaming ops
(HBM: algorithmic bytes / time vs MEASURED_PEAKS hbm_gbs), the bilateral denoiser (taps/s), the LBVH build (us, B/tri) and update_pdf.
usage: python tools/opbench.py [out.json]"""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import bench
import nvdiffrecmc_b200.renderutils as ru
import nvdiffrecmc_b200.optixutils as ou
from nvdiffrecmc_b200 import synth
from nvdiffrecmc_b200.light import EnvironmentLight

dev = torch.device("cuda:0")
peak, peak_src = bench.peaks()
flush = torch.empty(1 << 30, dtype=torch.uint8, device=dev)          # > 126 MB L2; long enough (~0.3 ms) to hide the host-side launch cost of the timed op


def timed(fn, reps=20):
    fn(); fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


out = {"hbm_peak_gbs": peak, "peak_source": peak_src, "l2_policy": "1 GB buffer rewritten between timed iterations", "ops": []}
g = torch.Generator().manual_seed(0)
for shape in [(1, 256, 256), (16, 512, 512), (1, 2048, 2048)]:          # test_bsdf.py RES-like + test_perf.py:54-56 sizes
    B, H, W = shape
    npx = B * H * W
    t = [torch.rand(B, H, W, 3, generator=g).to(dev) for _ in range(7)]
    kd, arm, pos, nrm, view, light, dout = t
    rough, dout1 = [torch.rand(B, H, W, 1, generator=g).to(dev) for _ in range(2)]
    ins = [x.clone().requires_grad_(True) for x in (kd, arm, pos, nrm, view, light, rough)]
    for name, fwd_bytes, bwd_bytes, used, f in [            # used: indices into ins of the op's differentiable inputs
        ("pbr_bsdf", 84, 156, range(6), lambda a: ru.pbr_bsdf(a[0], a[1], a[2], a[3], a[4], a[5])),
        ("prepare_shading_normal", 84, 156, range(6),
         lambda a: ru.prepare_shading_normal(a[2], a[4], a[0], a[3], a[1], a[5], two_sided_shading=True, opengl=True)),
        ("pbr_specular", 64, 116, (0, 3, 4, 5, 6), lambda a: ru.pbr_specular(a[0], a[1], a[2], a[3], a[4])),
        ("frostbite_diffuse", 44, 84, (3, 5, 4, 6), lambda a: ru.frostbite_diffuse(a[0], a[1], a[2], a[3])),
    ]:
        xs = [ins[i] for i in used]
        with torch.no_grad():
            ms_f = timed(lambda: f([x.detach() for x in xs]))
        y = f(xs)
        dy = dout if y.shape[-1] == 3 else dout1
        ms_b = timed(lambda: torch.autograd.grad(y, xs, dy, retain_graph=True))
        out["ops"].append({"op": name, "shape": list(shape), "fwd_ms": round(ms_f, 4), "fwd_gbs": round(npx * fwd_bytes / ms_f / 1e6, 1),
                           "fwd_frac_of_hbm_peak": round(npx * fwd_bytes / ms_f / 1e6 / peak, 3), "bwd_ms": round(ms_b, 4),
                           "bwd_gbs": round(npx * bwd_bytes / ms_b / 1e6, 1), "bwd_frac_of_hbm_peak": round(npx * bwd_bytes / ms_b / 1e6 / peak, 3),
                           "algorithmic_bytes_per_px": [fwd_bytes, bwd_bytes]})
        print(out["ops"][-1], flush=True)

# tail of shade(): denoiser normalisation + demodulated recombination (render.py:119-131), 8 x 512 x 512
B, H, W = 8, 512, 512
a4 = (torch.rand(B, H, W, 4, generator=g) + 0.5).to(dev).requires_grad_(True); b4 = (torch.rand(B, H, W, 4, generator=g) + 0.5).to(dev).requires_grad_(True)
kdc = torch.rand(B, H, W, 3, generator=g).to(dev).requires_grad_(True); ksc = torch.rand(B, H, W, 3, generator=g).to(dev).requires_grad_(True)
from nvdiffrecmc_b200.optixutils.ops import shade_combine
with torch.no_grad():
    ms_f = timed(lambda: shade_combine(a4.detach(), b4.detach(), kdc.detach(), ksc.detach()))
yc = shade_combine(a4, b4, kdc, ksc)
gyc = torch.rand_like(yc)
ms_b = timed(lambda: torch.autograd.grad(yc, [a4, b4, kdc, ksc], gyc, retain_graph=True))
npx = B * H * W
out["shade_combine"] = {"shape": [B, H, W], "fwd_ms": round(ms_f, 4), "fwd_gbs_at_68B_per_px": round(npx * 68 / ms_f / 1e6, 1), "fwd_frac_of_hbm_peak": round(npx * 68 / ms_f / 1e6 / peak, 3),
                        "bwd_ms": round(ms_b, 4), "bwd_gbs_at_124B_per_px": round(npx * 124 / ms_b / 1e6, 1), "bwd_frac_of_hbm_peak": round(npx * 124 / ms_b / 1e6 / peak, 3)}
print(out["shade_combine"], flush=True)

if os.environ.get("OPB_ONLY") == "ew":
    if len(sys.argv) > 1:
        json.dump(out, open(sys.argv[1], "w"), indent=1)
    sys.exit(0)

# bilateral denoiser, sigma = 2 (23 x 23 taps), 8 x 512 x 512
B, H, W = 8, 512, 512
col = torch.rand(B, H, W, 3, generator=g).to(dev).requires_grad_(True)
nrm = torch.nn.functional.normalize(torch.rand(B, H, W, 3, generator=g).to(dev) - 0.5, dim=-1)
zdz = torch.stack([torch.rand(B, H, W, generator=g).to(dev) + 1, torch.full((B, H, W), 0.01, device=dev)], -1)
with torch.no_grad():
    ms_f = timed(lambda: ou.bilateral_denoiser(col.detach(), nrm, zdz, 2.0))
y = ou.bilateral_denoiser(col, nrm, zdz, 2.0)
gy = torch.rand_like(y)
ms_b = timed(lambda: torch.autograd.grad(y, col, gy, retain_graph=True))
taps = B * H * W * 23 * 23
colB = torch.rand(B, H, W, 3, generator=g).to(dev)
with torch.no_grad():
    ms_f2 = timed(lambda: ou.bilateral_denoiser2(col.detach(), colB, nrm, zdz, 2.0))
out["bilateral_denoiser"] = {"shape": [B, H, W], "sigma": 2.0, "taps_per_px": 529, "fwd_ms": round(ms_f, 4), "fwd2_ms_two_signals": round(ms_f2, 4), "bwd_ms": round(ms_b, 4),
                             "fwd_gtaps_per_s": round(taps / ms_f / 1e6, 1), "fwd_gbs_compulsory_48B_per_px": round(B * H * W * 48 / ms_f / 1e6, 1)}
print(out["bilateral_denoiser"], flush=True)

# LBVH build
out["bvh_build"] = []
for kind, level in ([("blob+torus", 4), ("grid1m", 0)] if not os.environ.get("OPB_QUICK") else []):
    wl = dict(bench.WORKLOAD); wl["mesh"] = kind; wl["mesh_level"] = level
    v, f, _ = bench.build_scene_numpy(wl, 0)
    vt, ft = torch.tensor(v, device=dev), torch.tensor(f, device=dev)
    ctx = ou.OptiXContext()
    ms = timed(lambda: ou.optix_build_bvh(ctx, vt, ft, rebuild=1))
    ms_refit = timed(lambda: ou.optix_build_bvh(ctx, vt, ft, rebuild=0))
    T = int(ft.shape[0])
    out["bvh_build"].append({"mesh": kind, "triangles": T, "rebuild_ms": round(ms, 4), "refit_ms": round(ms_refit, 4),
                             "rebuild_gbs_at_248B_per_tri": round(T * 248 / ms / 1e6, 1), "mtris_per_s": round(T / ms / 1e3, 1)})
    print(out["bvh_build"][-1], flush=True)

# update_pdf
out["update_pdf"] = []
for hw in [(256, 256), (1024, 2048)]:
    lgt = EnvironmentLight(torch.rand(hw[0], hw[1], 3, generator=g).to(dev))
    ms = timed(lgt.update_pdf)
    ms_py = timed(lambda: lgt.update_pdf(use_python=True))
    out["update_pdf"].append({"probe": list(hw), "native_ms": round(ms, 4), "torch_ops_ms": round(ms_py, 4), "native_gbs_at_28B_per_texel": round(hw[0] * hw[1] * 28 / ms / 1e6, 1)})
    print(out["update_pdf"][-1], flush=True)

if len(sys.argv) > 1:
    json.dump(out, open(sys.argv[1], "w"), indent=1)
