"""Developer tool: tiny end-to-end pass of every kernel family, meant to run under compute-sanitizer
(memcheck / racecheck / initcheck) -- SURVEY.md section 5 "race detection"."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
from common import make_case
import nvdiffrecmc_b200.optixutils as ou
import nvdiffrecmc_b200.renderutils as ru

dev = torch.device("cuda:0")
for N in (4, 9):
    c = make_case(res=12, B=2, N=N, perm_rows=64)
    t = lambda k: torch.tensor(c[k], device=dev)
    ctx = ou.OptiXContext()
    ou.optix_build_bvh(ctx, t("verts"), t("tris"), 1)
    pos, kd, ks, light = [t(k).requires_grad_(True) for k in ("pos", "kd", "ks", "light")]
    nrm = ru.prepare_shading_normal(pos, t("view"), None, t("smooth_nrm"), t("tangent"), t("geom_nrm"))
    d, s = ou.optix_env_shade(ctx, t("mask"), t("ro"), pos, nrm, t("view"), kd, ks, light, t("pdf"), t("rows"), t("cols"), n_samples_x=N, rnd_seed=3,
                              perms=t("perms"))
    zdz = torch.stack([t("depth"), torch.full_like(t("depth"), 0.01)], -1)
    a, b = ou.bilateral_denoiser2(d, s, torch.nn.functional.normalize(nrm.detach() + 1e-6, dim=-1), zdz, 1.0)
    loss = ru.image_loss(a * kd + b, torch.rand_like(a), loss="l1", tonemapper="log_srgb")
    loss.backward()
    ou.optix_build_bvh(ctx, t("verts"), t("tris"), 0)
    v = ou.trace_visibility(ctx, t("ro").reshape(-1, 3), torch.nn.functional.normalize(torch.randn(c["ro"].size // 3, 3, device=dev), dim=-1))
    pts = ru.xfm_points(t("verts")[None], torch.rand(2, 4, 4, device=dev))
    # re-tracing backward (decorrelated seeds), update_pdf, rasterize / interpolate
    d2, s2 = ou.optix_env_shade(ctx, t("mask"), t("ro"), pos, nrm.detach().requires_grad_(True), t("view"), kd, ks, light, t("pdf"), t("rows"), t("cols"), n_samples_x=N, rnd_seed=None,
                                perms=t("perms"))
    (d2.sum() + s2.sum()).backward()
    from nvdiffrecmc_b200.light import EnvironmentLight
    from nvdiffrecmc_b200.raster import rasterize, interpolate
    lg = EnvironmentLight(light.detach())
    proj = torch.tensor([[2.4, 0, 0, 0], [0, -2.4, 0, 0], [0, 0, -1.02, -0.2], [0, 0, -1, 0]], device=dev)
    mv = torch.eye(4, device=dev); mv[2, 3] = -3.0
    rast = rasterize(ctx, (proj @ mv)[None], (24, 24))
    att = t("verts").clone().requires_grad_(True)
    interpolate(att, rast, t("tris"))[0].sum().backward()
# round 2: records entry point (MODE 2), fused shade tail, texel fetch, device-side seed
from nvdiffrecmc_b200.optixutils.ops import env_shade_records, shade_combine
from nvdiffrecmc_b200.raster import texel_fetch
env_shade_records(ctx, t("mask"), t("ro"), t("pos"), nrm.detach(), t("view"), t("kd"), t("ks"), t("light"), t("pdf"), t("rows"), t("cols"), t("perms"), n_samples_x=N, rnd_seed=1)
seed_t = torch.full((1,), 7, dtype=torch.int32, device=dev)
ou.optix_env_shade(ctx, t("mask"), t("ro"), t("pos"), nrm.detach(), t("view"), t("kd"), t("ks"), t("light"), t("pdf"), t("rows"), t("cols"), n_samples_x=N, rnd_seed=seed_t, perms=t("perms"))
a4 = (torch.rand(2, 12, 12, 4, device=dev) + 0.5).requires_grad_(True)
shade_combine(a4, a4 * 1.5, t("kd"), t("ks")).sum().backward()
tex = torch.rand(64, 3, device=dev, requires_grad=True)
texel_fetch(tex, torch.randint(0, 64, (2, 12, 12), device=dev)).sum().backward()
torch.cuda.synchronize()
print("sanitize workload ok", float(loss), int(v.sum()), tuple(pts.shape))
