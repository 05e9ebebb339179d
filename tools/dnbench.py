"""Developer tool: bilateral denoiser forward (one / two signals) and transposed two-signal filter at 8 x 512^2, sigma = 2, on both
staging paths: "tma" (contiguous operands, tensor-map halo tiles) and "plain" (the same values as strided channel views, which a
tensor map cannot describe -- the way the reference's sliced 8-channel tensor reaches the filter).  usage: python tools/dnbench.py"""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import ctypes as C
import numpy as np
import torch
import nvdiffrecmc_b200.optixutils as ou
from nvdiffrecmc_b200 import _lib as L
dev = torch.device("cuda:0")
flush = torch.empty(1 << 29, dtype=torch.uint8, device=dev)
def timed(fn, reps=20):
    fn(); fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))
g = torch.Generator().manual_seed(0)
B, H, W = 8, 512, 512
col = torch.rand(B, H, W, 3, generator=g).to(dev); colB = torch.rand(B, H, W, 3, generator=g).to(dev)
nrm = torch.nn.functional.normalize(torch.rand(B, H, W, 3, generator=g).to(dev) - 0.5, dim=-1)
zdz = torch.stack([torch.rand(B, H, W, generator=g).to(dev) + 1, torch.full((B, H, W), 0.01, device=dev)], -1)
ga, gb = torch.rand(B, H, W, 4, generator=g).to(dev), torch.rand(B, H, W, 4, generator=g).to(dev)
strided = lambda t: torch.cat([t, torch.zeros_like(t[..., :1])], -1)[..., :t.shape[-1]]      # same values, one extra float of pixel pitch
oa, ob = torch.empty(B, H, W, 3, device=dev), torch.empty(B, H, W, 3, device=dev)
out = {"shape": [B, H, W], "sigma": 2.0}
for path, lay in (("tma", lambda t: t), ("plain", strided)):
    c, cb, a4, b4 = lay(col), lay(colB), lay(ga), lay(gb)
    with torch.no_grad():
        f1 = timed(lambda: ou.bilateral_denoiser(c, nrm, zdz, 2.0))
        f2 = timed(lambda: ou.bilateral_denoiser2(c, cb, nrm, zdz, 2.0))
    b2 = timed(lambda: L.check(L.lib().mcs_bilateral_bwd2(C.byref(L.nhwc(nrm)), C.byref(L.nhwc(zdz)), 2.0, C.byref(L.nhwc(a4)), C.byref(L.nhwc(b4)),
                                                           oa.data_ptr(), ob.data_ptr(), L.stream_ptr()), "bilateral_denoiser2 (backward)"))
    out[path] = {"fwd1_ms": round(f1, 4), "fwd2_ms": round(f2, 4), "bwd2_ms": round(b2, 4), "gtaps_per_s_fwd2": round(B * H * W * 529 / f2 / 1e6, 1)}
print(json.dumps(out))
