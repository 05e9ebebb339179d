"""GPU parity: fused env-light shading kernel (mcs_env_shade_*) vs the CPU oracle
(oracle/mcoracle.c: orc_env_shade, a restatement of optixutils/c_src/envsampling/kernel.cu).

Bars (BASELINE.json north_star): integer records (env texel per ray, shadow-ray visibility bit)
BIT-EXACT; radiance and gradients <= 1e-4 relative L2 for the same seed / perms.
"""
import numpy as np
import pytest
import torch

from common import make_case, oracle, pick, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _t(c, k, dev, **kw):
    return torch.tensor(c[k], device=dev, **kw)


def _ctx(c, dev):
    import nvdiffrecmc_b200.optixutils as ou
    ctx = ou.OptiXContext()
    ou.optix_build_bvh(ctx, _t(c, "verts", dev), _t(c, "tris", dev), rebuild=1)
    return ctx


def _args(c, dev):
    return [_t(c, k, dev) for k in ("mask", "ro", "pos", "nrm", "view", "kd", "ks", "light", "pdf", "rows", "cols")]


@pytest.mark.parametrize("bsdf", ["pbr", "diffuse", "white"])
@pytest.mark.parametrize("N,light,lhw", [(4, "random", (32, 64)), (3, "hdr", (64, 128)), (8, "random", (16, 16))])
def test_forward_and_records(dev, bsdf, N, light, lhw):
    from nvdiffrecmc_b200.optixutils.ops import env_shade_records
    c = make_case(res=24, B=2, N=N, light=light, light_hw=lhw, seed=N)
    if bsdf == "white":
        c["kd"] = np.ones_like(c["kd"])        # render.py:107
    ctx = _ctx(c, dev)
    a = _args(c, dev)
    perms = _t(c, "perms", dev)
    diff, spec, rec_t, rec_v = env_shade_records(ctx, *a, perms, BSDF=bsdf, n_samples_x=N, rnd_seed=11, shadow_scale=1.0)
    o = oracle()
    d_ref, s_ref, (rt, rv) = o.env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"],
                                         c["rows"], c["cols"], c["perms"], BSDF=bsdf, n_samples_x=N, rnd_seed=11, records=True)
    rec_t, rec_v = rec_t.cpu().numpy(), rec_v.cpu().numpy()
    assert np.array_equal(rec_t, rt), "env texel selection differs from the oracle (%d of %d rays)" % ((rec_t != rt).sum(), rt.size)
    traced = rec_v != 2
    assert np.array_equal(rec_v[traced], rv[traced]), "visibility bits differ from the oracle"
    assert traced[c["mask"] > 0].mean() > 0.2
    assert rel_l2(diff.cpu().numpy(), d_ref) < TOL
    assert rel_l2(spec.cpu().numpy(), s_ref) < TOL
    # masked pixels are exactly zero
    m = c["mask"] <= 0
    assert (diff.cpu().numpy()[m] == 0).all() and (spec.cpu().numpy()[m] == 0).all()


@pytest.mark.parametrize("bsdf", ["pbr", "diffuse"])
@pytest.mark.parametrize("shadow_scale", [1.0, 0.5])
def test_backward(dev, bsdf, shadow_scale):
    import nvdiffrecmc_b200.optixutils as ou
    N = 4
    c = make_case(res=24, B=2, N=N, seed=2)
    ctx = _ctx(c, dev)
    mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
    for x in (pos, nrm, kd, ks, light):
        x.requires_grad_(True)
    perms = _t(c, "perms", dev)
    diff, spec = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, BSDF=bsdf, n_samples_x=N, rnd_seed=5,
                                    shadow_scale=shadow_scale, perms=perms)
    rng = np.random.default_rng(0)
    dg = rng.uniform(0, 1, size=diff.shape).astype(np.float32); sg = rng.uniform(0, 1, size=spec.shape).astype(np.float32)
    torch.autograd.backward([diff, spec], [torch.tensor(dg, device=dev), torch.tensor(sg, device=dev)])
    o = oracle()
    ref = o.env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"], c["cols"],
                      c["perms"], BSDF=bsdf, n_samples_x=N, rnd_seed=5, shadow_scale=shadow_scale, grads=(dg, sg))
    names = ["gb_pos", "gb_normal", "gb_kd", "gb_ks", "light"]
    got = [pos.grad, nrm.grad, kd.grad, ks.grad, light.grad]
    for n, g, r in zip(names, got, ref):
        if np.linalg.norm(r) == 0:
            assert float(g.abs().max()) == 0, n
        else:
            assert rel_l2(g.cpu().numpy(), r) < TOL, "%s gradient: rel-L2 %.3e" % (n, rel_l2(g.cpu().numpy(), r))
    d_ref, s_ref = o.env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"],
                               c["cols"], c["perms"], BSDF=bsdf, n_samples_x=N, rnd_seed=5, shadow_scale=shadow_scale)
    assert rel_l2(diff.detach().cpu().numpy(), d_ref) < TOL and rel_l2(spec.detach().cpu().numpy(), s_ref) < TOL


def test_strided_and_broadcast_inputs(dev):
    """The reference's call site passes non-contiguous views: rast[...,-1] (stride 4), all_tex[...,0:3] / [...,3:6]
    (stride 6), lgt.rows[:,0] (stride W) and a broadcast view_pos [B,1,1,3] (render.py:66,113-114)."""
    import nvdiffrecmc_b200.optixutils as ou
    N = 4
    c = make_case(res=16, B=2, N=N, seed=4)
    ctx = _ctx(c, dev)
    mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
    perms = _t(c, "perms", dev)
    ref = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=3, perms=perms)
    rast = torch.zeros(*mask.shape, 4, device=dev); rast[..., -1] = mask
    alltex = torch.cat([kd, ks], -1)
    rows2d = rows[:, None].repeat(1, cols.shape[1])
    got = ou.optix_env_shade(ctx, rast[..., -1], ro, pos, nrm, view, alltex[..., 0:3], alltex[..., 3:6], light, pdf, rows2d[:, 0], cols,
                             n_samples_x=N, rnd_seed=3, perms=perms)
    assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])


def test_batch_offset_matches_single_gpu_stream(dev):
    """Data-parallel parity (SURVEY 8e): views [1,2) rendered with batch_offset=1 equal slice 1 of the full batch."""
    import nvdiffrecmc_b200.optixutils as ou
    N = 4
    c = make_case(res=16, B=2, N=N, seed=6)
    ctx = _ctx(c, dev)
    mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
    perms = _t(c, "perms", dev)
    full = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=9, perms=perms)
    s = slice(1, 2)
    part = ou.optix_env_shade(ctx, mask[s], ro[s], pos[s], nrm[s], view[s], kd[s], ks[s], light, pdf, rows, cols, n_samples_x=N, rnd_seed=9,
                              perms=perms, batch_offset=1)
    assert torch.equal(full[0][s], part[0]) and torch.equal(full[1][s], part[1])


def test_errors_are_loud(dev):
    import nvdiffrecmc_b200.optixutils as ou
    c = make_case(res=8, B=1, N=2, seed=1)
    ctx = ou.OptiXContext()
    a = _args(c, dev)
    with pytest.raises(RuntimeError, match="acceleration structure"):
        ou.optix_env_shade(ctx, *a, n_samples_x=2, rnd_seed=0, perms=_t(c, "perms", dev))
    with pytest.raises(AssertionError, match="empty training triangle mesh"):
        ou.optix_build_bvh(ctx, torch.zeros(3, 3, device=dev), torch.zeros(0, 3, dtype=torch.int32, device=dev), 1)
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        ou.optix_build_bvh(ctx, torch.zeros(3, 3), torch.zeros(1, 3, dtype=torch.int32), 1)


def test_backward_replays_the_visibility_record(dev):
    """With a shared seed the backward pass replays what the forward pass recorded -- the evaluated rays ("rays", default) or one
    visibility bit per sample ("bits") -- instead of re-tracing like the reference (None); all three must agree."""
    import nvdiffrecmc_b200.optixutils as ou
    from nvdiffrecmc_b200.optixutils import ops
    N = 4
    c = make_case(res=20, B=2, N=N, seed=7)
    ctx = _ctx(c, dev)
    perms = _t(c, "perms", dev)
    grads = {}
    default_mode = ops.HIT_RECORD_REPLAY
    assert default_mode == "rays"
    for replay in ("rays", "bits", None):
        ops.HIT_RECORD_REPLAY = replay
        try:
            mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
            for x in (pos, nrm, kd, ks, light):
                x.requires_grad_(True)
            d, s = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=21, perms=perms)
            (d.sum() * 0.7 + (s * s).sum()).backward()
            grads[replay] = [x.grad.clone() for x in (pos, nrm, kd, ks, light)]
        finally:
            ops.HIT_RECORD_REPLAY = default_mode
    for mode in ("rays", "bits"):
        for a, b in zip(grads[mode][:4], grads[None][:4]):
            assert torch.equal(a, b), mode                    # per-pixel gradients: same rays, same order, same arithmetic
        assert rel_l2(grads[mode][4].cpu().numpy(), grads[None][4].cpu().numpy()) < 1e-6      # env-map gradient: atomics reorder
    # a context rebuilt between forward and backward invalidates the record: the op falls back to re-tracing (no stale replay)
    mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
    light.requires_grad_(True)
    d, s = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=21, perms=perms)
    ou.optix_build_bvh(ctx, _t(c, "verts", dev), _t(c, "tris", dev), rebuild=1)
    (d.sum() + s.sum()).backward()
    assert torch.isfinite(light.grad).all()


def test_decorrelated_mode_and_multi_fill_pixels(dev):
    """rnd_seed=None draws independent seeds for forward and backward (ops.py:83,100: no replay possible); n_samples_x=9 needs two
    queue fills per pixel (162 sample slots > 128)."""
    import nvdiffrecmc_b200.optixutils as ou
    N = 9
    c = make_case(res=12, B=1, N=N, seed=8, perm_rows=64)
    ctx = _ctx(c, dev)
    mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
    for x in (kd, light):
        x.requires_grad_(True)
    perms = _t(c, "perms", dev)
    d, s = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=4, perms=perms)
    o = oracle()
    d_ref, s_ref = o.env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"],
                               c["cols"], c["perms"], n_samples_x=N, rnd_seed=4)
    assert rel_l2(d.detach().cpu().numpy(), d_ref) < TOL and rel_l2(s.detach().cpu().numpy(), s_ref) < TOL
    dg = np.random.default_rng(1).uniform(0, 1, size=d.shape).astype(np.float32)
    torch.autograd.backward([d, s], [torch.tensor(dg, device=dev), torch.tensor(dg, device=dev)])
    ref = o.env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"], c["cols"],
                      c["perms"], n_samples_x=N, rnd_seed=4, grads=(dg, dg))
    assert rel_l2(kd.grad.cpu().numpy(), ref[2]) < TOL and rel_l2(light.grad.cpu().numpy(), ref[4]) < TOL
    np.random.seed(0)
    d2, s2 = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=None, perms=perms)
    (d2.sum() + s2.sum()).backward()
    assert torch.isfinite(d2).all() and torch.isfinite(light.grad).all()


def test_records_on_a_large_mesh(dev):
    """344 k triangles: leaf boxes are ~100x smaller relative to the scene than in the other cases, which is where the 16-bit
    quantised nodes lose the most precision.  Visibility must stay bit-exact (conservative culling), radiance within tolerance."""
    from nvdiffrecmc_b200.optixutils.ops import env_shade_records
    N = 4
    c = make_case(res=20, B=1, N=N, level=7, seed=1)
    assert c["tris"].shape[0] > 300000
    ctx = _ctx(c, dev)
    a = _args(c, dev)
    diff, spec, rec_t, rec_v = env_shade_records(ctx, *a, _t(c, "perms", dev), BSDF="pbr", n_samples_x=N, rnd_seed=5, shadow_scale=1.0)
    d_ref, s_ref, (rt, rv) = oracle().env_shade(c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"],
                                                c["rows"], c["cols"], c["perms"], BSDF="pbr", n_samples_x=N, rnd_seed=5, records=True, vis_mode="bvh")
    rec_t, rec_v = rec_t.cpu().numpy(), rec_v.cpu().numpy()
    assert np.array_equal(rec_t, rt)
    traced = rec_v != 2
    assert np.array_equal(rec_v[traced], rv[traced]) and (rv[traced] == 0).sum() > 100
    assert rel_l2(diff.cpu().numpy(), d_ref) < TOL and rel_l2(spec.cpu().numpy(), s_ref) < TOL


@pytest.mark.parametrize("n_occ", [0, 1, 3, 6])
def test_tiny_and_flat_meshes(dev, n_occ):
    """1-4 triangles take the 'root is one leaf run' path of the node emitters; an axis-aligned plane has zero extent in one axis
    (degenerate quantisation grid); with occluders hovering above the plane some shadow rays are blocked.  Bit-exact vs brute force."""
    from nvdiffrecmc_b200.optixutils.ops import env_shade_records
    import nvdiffrecmc_b200.optixutils as ou
    rng = np.random.default_rng(n_occ)
    v = [[-2, 0, -2], [2, 0, -2], [2, 0, 2], [-2, 0, 2]]
    f = [[0, 1, 2], [0, 2, 3]] if n_occ != 0 else [[0, 1, 2]]
    for k in range(n_occ):
        c = rng.uniform(-1, 1, 3) * [1.0, 0.0, 1.0] + [0, 0.4 + 0.2 * k, 0]
        b = len(v)
        v += [list(c + [-0.6, 0, -0.5]), list(c + [0.6, 0.05, -0.4]), list(c + [0.0, 0.0, 0.7])]
        f.append([b, b + 1, b + 2])
    v = np.asarray(v, np.float32); f = np.asarray(f, np.int32)
    if n_occ == 0:
        assert f.shape[0] == 1
    H = W = 12
    N = 4
    xs = np.linspace(-0.9, 0.9, W, dtype=np.float32)
    gx, gz = np.meshgrid(xs, xs, indexing="xy")
    pos = np.stack([gx, np.zeros((H, W), np.float32), gz], -1)[None].astype(np.float32)                   # points on the plane y = 0
    if n_occ == 0:
        pos = pos * np.float32(0.4) + np.float32([0.6, 0, -0.6])       # stay inside the single triangle
    nrm = np.zeros_like(pos); nrm[..., 1] = 1
    view = np.float32([0.3, 2.0, 0.4]).reshape(1, 1, 1, 3)
    kd = rng.uniform(0.1, 1, pos.shape).astype(np.float32); ks = rng.uniform(0.1, 1, pos.shape).astype(np.float32); ks[..., 0] = 0
    mask = np.ones((1, H, W), np.float32)
    ro = (pos + nrm * np.float32(0.001)).astype(np.float32)
    o = oracle()
    from nvdiffrecmc_b200 import synth
    light = synth.random_light(32, seed=3)
    pdf, rows, cols = o.update_pdf(light)
    perms = synth.make_perms(N, seed=4, rows=128)
    ctx = ou.OptiXContext()
    ou.optix_build_bvh(ctx, torch.tensor(v, device=dev), torch.tensor(f, device=dev), rebuild=1)
    t = lambda a: torch.tensor(a, device=dev)
    diff, spec, rec_t, rec_v = env_shade_records(ctx, t(mask), t(ro), t(pos), t(nrm), t(view), t(kd), t(ks), t(light), t(pdf), t(rows), t(cols), t(perms),
                                                 BSDF="pbr", n_samples_x=N, rnd_seed=2, shadow_scale=1.0)
    d_ref, s_ref, (rt, rv) = o.env_shade(o.scene(v, f), mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, perms, BSDF="pbr", n_samples_x=N,
                                         rnd_seed=2, records=True)
    rec_t, rec_v = rec_t.cpu().numpy(), rec_v.cpu().numpy()
    assert np.array_equal(rec_t, rt)
    traced = rec_v != 2
    assert np.array_equal(rec_v[traced], rv[traced])
    if n_occ >= 3:
        assert (rv[traced] == 0).sum() > 20                      # some rays really are occluded
    assert rel_l2(diff.cpu().numpy(), d_ref) < TOL and rel_l2(spec.cpu().numpy(), s_ref) < TOL


def _compiled_reference_case():
    c = make_case(res=24, B=2, N=4, seed=3)
    ra = (c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"], c["cols"], c["perms"])
    g = np.random.default_rng(1)
    gd = g.uniform(size=c["pos"].shape).astype(np.float32); gs = g.uniform(size=c["pos"].shape).astype(np.float32)
    return c, ra, gd, gs


GRAD_NAMES = ("pos", "nrm", "kd", "ks", "light")


def ref_product_case(ref, bsdf):
    """What the reference's raygen program returns for test_product_against_the_compiled_reference (frozen in tests/golden)."""
    c, ra, gd, gs = _compiled_reference_case()
    d_r, s_r = ref.env_shade(*ra, BSDF=bsdf, n_samples_x=4, rnd_seed=9)
    g_r = ref.env_shade(*ra, BSDF=bsdf, n_samples_x=4, rnd_seed=9, grads=(gd, gs))
    out = dict(diff=pick(d_r), spec=pick(s_r), **{n: pick(g) for n, g in zip(GRAD_NAMES, g_r)})
    out.update({n + "_absmax": np.abs(g).max() for n, g in zip(GRAD_NAMES, g_r)})
    return out


@pytest.mark.parametrize("bsdf", ["pbr", "diffuse"])
def test_product_against_the_compiled_reference(dev, bsdf):
    """The CUDA path against the REFERENCE's own raygen program (kernel.cu compiled unmodified for the host, shadow rays answered by the
    oracle's predicate), whose outputs are frozen in tests/golden/ref_compiled_kernels.npz at a fixed sample of pixels / texels.
    Radiance within 1e-4; gradients within the fp32 noise floor that separates the reference itself from the fp64 evaluation of the
    same samples."""
    import nvdiffrecmc_b200.optixutils as ou
    from common import frozen_reference
    N = 4
    c, ra, gd, gs = _compiled_reference_case()
    r_ref = frozen_reference("product-" + bsdf)
    ctx = _ctx(c, dev)
    a = _args(c, dev)
    for i in (2, 3, 5, 6, 7):
        a[i].requires_grad_(True)                                       # pos, nrm, kd, ks, light
    diff, spec = ou.optix_env_shade(ctx, *a, BSDF=bsdf, n_samples_x=N, rnd_seed=9, perms=_t(c, "perms", dev))
    assert rel_l2(pick(diff.detach().cpu().numpy()), r_ref["diff"]) < TOL
    if bsdf == "pbr":
        assert rel_l2(pick(spec.detach().cpu().numpy()), r_ref["spec"]) < TOL
    torch.autograd.backward([diff, spec], [torch.tensor(gd, device=dev), torch.tensor(gs, device=dev)])
    o64 = oracle(f64=True)
    g64 = o64.env_shade(o64.scene(c["verts"], c["tris"]), *ra[1:], BSDF=bsdf, n_samples_x=N, rnd_seed=9, grads=(gd, gs),
                        sampling_gbuffer=(c["pos"], c["nrm"], c["kd"], c["ks"]))
    for name, t, r64 in zip(GRAD_NAMES, (a[2], a[3], a[5], a[6], a[7]), g64):
        got = t.grad.cpu().numpy() if t.grad is not None else np.zeros_like(r64)
        if r_ref[name + "_absmax"] == 0:
            assert np.abs(got).max() == 0, name
            continue
        got, r, r64 = pick(got), r_ref[name], pick(r64)
        floor = rel_l2(r, r64)                                          # how far the fp32 reference is from exact arithmetic here
        assert rel_l2(got, r) < max(TOL, 2.0 * floor), (name, rel_l2(got, r), floor)


@pytest.mark.parametrize("tag,bsdf", [("pbr", "pbr"), ("diffuse", "diffuse")])
def test_product_against_frozen_reference_outputs(dev, tag, bsdf):
    """tests/golden/ref_env_shade_*.npz (reference raygen program, compiled for the host, outputs frozen with their inputs): the CUDA
    path reproduces them without needing oracle/_ref on this machine."""
    import os
    import nvdiffrecmc_b200.optixutils as ou
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_env_shade_%s.npz" % tag))
    t = lambda k, **kw: torch.tensor(d[k], device=dev, **kw)
    ctx = ou.OptiXContext()
    ou.optix_build_bvh(ctx, t("verts"), t("tris"), rebuild=1)
    pos, nrm, kd, ks, light = [t(k).requires_grad_(True) for k in ("pos", "nrm", "kd", "ks", "light")]
    diff, spec = ou.optix_env_shade(ctx, t("mask"), t("ro"), pos, nrm, t("view"), kd, ks, light, t("pdf"), t("rows"), t("cols"), BSDF=bsdf,
                                    n_samples_x=int(d["n_samples_x"]), rnd_seed=int(d["rnd_seed"]), shadow_scale=float(d["shadow_scale"]), perms=t("perms"))
    assert rel_l2(diff.detach().cpu().numpy(), d["diff"]) < TOL
    if bsdf == "pbr":
        assert rel_l2(spec.detach().cpu().numpy(), d["spec"]) < TOL
    torch.autograd.backward([diff, spec], [t("diff_grad"), t("spec_grad")])
    for name, x in zip(("pos", "nrm", "kd", "ks", "light"), (pos, nrm, kd, ks, light)):
        r = d[name + "_grad"]
        got = x.grad.cpu().numpy() if x.grad is not None else np.zeros_like(r)
        if np.abs(r).max() == 0:
            assert np.abs(got).max() == 0, name
        else:
            assert rel_l2(got, r) < 1e-3, (name, rel_l2(got, r))                # the frozen side is fp32: noise floor 2-5e-4 on the GGX adjoints


def test_device_resident_seed(dev):
    """rnd_seed may be a 1-element CUDA int32 tensor (C ABI: seed_offset_dev): the kernel reads it when it RUNS, so a CUDA-graph-captured
    step can advance the seed in-graph (render.py:116 bumps a host counter).  Same rays as the host seed of equal value, forward and in
    all three backward modes; a graph captured once follows the tensor."""
    import nvdiffrecmc_b200.optixutils as ou
    from nvdiffrecmc_b200.optixutils import ops
    N = 4
    c = make_case(res=16, B=2, N=N, seed=9)
    ctx = _ctx(c, dev)
    perms = _t(c, "perms", dev)
    seed_t = torch.full((1,), 7, dtype=torch.int32, device=dev)

    def run(seed, replay):
        default = ops.HIT_RECORD_REPLAY
        ops.HIT_RECORD_REPLAY = replay
        try:
            mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols = _args(c, dev)
            for x in (pos, nrm, kd, ks, light):
                x.requires_grad_(True)
            d, s = ou.optix_env_shade(ctx, mask, ro, pos, nrm, view, kd, ks, light, pdf, rows, cols, n_samples_x=N, rnd_seed=seed, perms=perms)
            (d.sum() + (s * s).sum()).backward()
            return d.detach(), s.detach(), kd.grad.clone(), light.grad.clone()
        finally:
            ops.HIT_RECORD_REPLAY = default
    for replay in ("rays", "bits", None):
        a, b = run(7, replay), run(seed_t, replay)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        assert rel_l2(b[3].cpu().numpy(), a[3].cpu().numpy()) < 1e-6              # env-map gradient: atomics reorder
    seed_t += 1
    a, b = run(8, "rays"), run(seed_t, "rays")
    assert torch.equal(a[0], b[0]) and not torch.equal(a[0], run(7, "rays")[0])
    with pytest.raises(RuntimeError, match="1-element CUDA int32"):
        ou.optix_env_shade(ctx, *_args(c, dev), n_samples_x=N, rnd_seed=torch.zeros(1, dtype=torch.int64, device=dev), perms=perms)
    # one captured forward launch, replayed with an advancing device seed
    args = _args(c, dev)
    seed_g = torch.full((1,), 20, dtype=torch.int32, device=dev)
    ou.optix_env_shade(ctx, *args, n_samples_x=N, rnd_seed=seed_g, perms=perms)      # warm up outside capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        seed_g += 1
        dg, sg = ou.optix_env_shade(ctx, *args, n_samples_x=N, rnd_seed=seed_g, perms=perms)
    for k in (1, 2):
        g.replay()
        ref = ou.optix_env_shade(ctx, *args, n_samples_x=N, rnd_seed=20 + k, perms=perms)      # capture records, it does not execute
        assert torch.equal(dg, ref[0]) and torch.equal(sg, ref[1]), k
