"""Drop-in proof against the reference's own caller: `render.shade()` (render/render.py:30-164 of the reference, imported UNMODIFIED by
tests/golden/make_shade_golden.py with the oracle-backed optixutils stand-in and the reference's own PyTorch renderutils path) has its
output frozen in tests/golden/ref_shade_pbr.npz.

  * CPU: the oracle's restatement of shade()'s call chain reproduces the frozen output, and every call shade() and BilateralDenoiser
    make binds against this repository's signatures;
  * GPU: the product's ops, called in shade()'s order with shade()'s arguments, reproduce the frozen output.
"""
import inspect
import os

import numpy as np
import pytest
import torch

from common import rel_l2

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "ref_shade_pbr.npz")


def test_golden_fixture_is_sane():
    d = np.load(GOLDEN)
    assert d["out_shaded"].shape == d["rast"].shape and d["out_shaded"][..., 3].min() == 1.0
    covered = d["rast"][..., 3] > 0
    assert 0.2 < covered.mean() < 0.9
    assert np.abs(d["out_shaded"][covered][:, :3]).mean() > 0.05 and np.isfinite(d["out_shaded"]).all()
    # shade() composition (render.py:123-127): shaded = diffuse_light * kd * (1 - metalness) + specular_light
    comp = d["out_diffuse_light"][..., :3] * d["out_kd"][..., :3] + d["out_specular_light"][..., :3]
    assert rel_l2(comp, d["out_shaded"][..., :3]) < 1e-6


def test_oracle_shade_chain_reproduces_the_golden():
    """shade()'s call sequence (render.py:99-127) restated on the CPU oracle -- shading normal, env_shade, bilateral denoiser, recombination --
    reproduces the frozen output of the reference's own shade() within the bars the product is held to below."""
    from common import oracle
    d = np.load(GOLDEN)
    o = oracle()
    nrm = o.prepare_shading_normal(d["gb_pos"], d["view_pos"], None, d["gb_normal"], d["gb_tangent"], d["gb_geometric_normal"], True, True)
    ro = (d["gb_pos"] + nrm * np.float32(0.001)).astype(np.float32)
    pdf, rows, cols = o.update_pdf(d["light"])
    assert rel_l2(pdf, d["lgt_pdf"]) < 1e-6 and rel_l2(cols, d["lgt_cols"]) < 1e-6 and rel_l2(rows, d["lgt_rows"][:, 0]) < 1e-6
    mask = d["rast"][..., 3]
    diff, spec = o.env_shade(o.scene(d["verts"], d["tris"]), mask, ro, d["gb_pos"], nrm, d["view_pos"], d["kd"], d["ks"], d["light"], pdf, rows, cols,
                             d["perms"], BSDF="pbr", n_samples_x=int(d["n_samples_x"]), rnd_seed=int(d["rnd_seed"]), shadow_scale=float(d["shadow_scale"]))
    guide = nrm / np.sqrt(np.maximum((nrm * nrm).sum(-1, keepdims=True), 1e-20))     # denoiser.py:28 (safe-normalised guide)
    sigma = max(float(d["sigma_influence"]) * 2, 1e-4)                                  # denoiser.py:22-25
    dif, spc = o.bilateral_denoiser(diff, guide, d["gb_depth"], sigma), o.bilateral_denoiser(spec, guide, d["gb_depth"], sigma)
    shaded = dif * (d["kd"] * (1.0 - d["ks"][..., 2:3])) + spc
    cov = mask > 0
    assert rel_l2(nrm[cov], d["out_normal"][..., :3][cov]) < 1e-5
    assert rel_l2(dif, d["out_diffuse_light"][..., :3]) < 1e-4
    assert rel_l2(spc, d["out_specular_light"][..., :3]) < 1e-4
    assert rel_l2(shaded, d["out_shaded"][..., :3]) < 1e-4


def test_shade_call_sites_bind_against_this_package():
    """The calls render/render.py, render/light.py and denoiser/denoiser.py make (render.py:99,113-115; denoiser.py:31; dlmesh.py:50) bind
    against nvdiffrecmc_b200.{optixutils,renderutils}, and the light class computes the reference's pdf / CDFs (light.py:46-59, frozen in
    tests/golden/ref_update_pdf.npz)."""
    import nvdiffrecmc_b200.optixutils as ou
    import nvdiffrecmc_b200.renderutils as ru
    from nvdiffrecmc_b200.light import EnvironmentLight
    x = object()
    # render.py:113-115
    inspect.signature(ou.optix_env_shade).bind(x, x, x, x, x, x, x, x, x, x, x, x, BSDF='pbr', n_samples_x=8, rnd_seed=None, shadow_scale=1.0)
    # render.py:99
    inspect.signature(ru.prepare_shading_normal).bind(x, x, x, x, x, x, two_sided_shading=True, opengl=True)
    inspect.signature(ou.bilateral_denoiser).bind(x, x, x, 2.0)                 # denoiser.py:31
    inspect.signature(ou.optix_build_bvh).bind(x, x, x, rebuild=1)              # dlmesh.py:50, dataset_mesh.py:41
    assert callable(ou.OptiXContext)
    g = np.load(os.path.join(HERE, "golden", "ref_update_pdf.npz"))
    for k in ("a", "b"):
        lgt = EnvironmentLight(torch.tensor(g[k + "_base"]))
        assert torch.allclose(lgt._pdf, torch.tensor(g[k + "_pdf"])) and torch.allclose(lgt.cols, torch.tensor(g[k + "_cols"]))
        assert torch.allclose(lgt.rows, torch.tensor(g[k + "_rows"]))


def _product_shade(d, dev):
    """shade()'s call sequence (render.py:99-127) on the product: same arguments, same order."""
    import nvdiffrecmc_b200.optixutils as ou
    import nvdiffrecmc_b200.renderutils as ru
    from nvdiffrecmc_b200.denoiser import BilateralDenoiser
    from nvdiffrecmc_b200.light import EnvironmentLight
    t = lambda k: torch.tensor(d[k], device=dev)
    ctx = ou.OptiXContext()
    ou.optix_build_bvh(ctx, t("verts"), t("tris"), rebuild=1)
    lgt = EnvironmentLight(t("light"))
    rast, gb_depth, gb_pos, view_pos, kd, ks = t("rast"), t("gb_depth"), t("gb_pos"), t("view_pos"), t("kd"), t("ks")
    gb_normal = ru.prepare_shading_normal(gb_pos, view_pos, None, t("gb_normal"), t("gb_tangent"), t("gb_geometric_normal"), two_sided_shading=True, opengl=True)
    ro = gb_pos + gb_normal * 0.001
    diffuse_accum, specular_accum = ou.optix_env_shade(ctx, rast[..., -1], ro, gb_pos, gb_normal, view_pos, kd, ks, lgt.base, lgt._pdf, lgt.rows[:, 0], lgt.cols,
                                                       BSDF='pbr', n_samples_x=int(d["n_samples_x"]), rnd_seed=int(d["rnd_seed"]),
                                                       shadow_scale=float(d["shadow_scale"]), perms=t("perms"))
    den = BilateralDenoiser(influence=float(d["sigma_influence"]))
    diffuse_d = den.forward(torch.cat((diffuse_accum, gb_normal, gb_depth), dim=-1))
    specular_d = den.forward(torch.cat((specular_accum, gb_normal, gb_depth), dim=-1))
    shaded = diffuse_d * (kd * (1.0 - ks[..., 2:3])) + specular_d
    # the fused tail used by bench.py (one denoiser launch for both signals + one recombination launch)
    from nvdiffrecmc_b200.denoiser import _safe_normalize
    fused = ou.denoise_and_combine(diffuse_accum, specular_accum, _safe_normalize(gb_normal), gb_depth, den.sigma, kd, ks)
    return gb_normal, diffuse_d, specular_d, shaded, fused


@pytest.mark.gpu
def test_product_reproduces_the_reference_shade_output(dev):
    d = np.load(GOLDEN)
    nrm, dif, spc, shaded, fused = _product_shade(d, dev)
    cov = d["rast"][..., 3] > 0
    n = lambda x: x.detach().cpu().numpy()
    assert rel_l2(n(nrm)[cov], d["out_normal"][..., :3][cov]) < 1e-5
    assert rel_l2(n(dif), d["out_diffuse_light"][..., :3]) < 1e-4
    assert rel_l2(n(spc), d["out_specular_light"][..., :3]) < 1e-4
    assert rel_l2(n(shaded), d["out_shaded"][..., :3]) < 1e-4
    assert rel_l2(n(fused), d["out_shaded"][..., :3]) < 1e-4
