"""CPU: the oracle against the REFERENCE ITSELF -- the unmodified raygen program of render/optixutils/c_src/envsampling/kernel.cu
(with bsdf.h, math_utils.h, common.h, accessor.h, params.h), denoising.cu and the renderutils kernels (bsdf.cu, normal.cu, loss.cu,
mesh.cu), compiled for the host by oracle/ref_shim (oracle/_ref).  The shadow-ray hit/miss decision is the one thing that source
delegates to the closed OptiX runtime; it is supplied by the oracle's visibility predicate, everything else (RNG, strata, CDF sampling,
lat-long mapping, MIS, BSDF forward and hand-derived adjoints, gradient scatter) is the reference's own code.

The reference's outputs are frozen in tests/golden/ref_compiled_kernels.npz: tests/golden/make_ref_kernels_golden.py runs the
`ref_*` function of every case below through oracle.Reference where the reference sources exist.  Each case rebuilds its inputs from
the same seeds and compares the oracle with the frozen outputs; large outputs are stored at a fixed sample of their rows (common.pick)."""
import numpy as np
import pytest

from common import frozen_reference, make_case, oracle, pick, rel_l2


def _args(c, kd=None):
    return (c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"] if kd is None else kd, c["ks"], c["light"], c["pdf"], c["rows"],
            c["cols"], c["perms"])


BSDFS = ["pbr", "diffuse", "white"]
FWD_CASES = [(4, "random", (32, 64), 1.0), (3, "hdr", (64, 128), 0.5), (8, "random", (16, 16), 1.0)]


def _fwd_case(bsdf, N, light, lhw, shadow):
    c = make_case(res=20, B=2, N=N, light=light, light_hw=lhw, seed=N)
    kd = np.ones_like(c["kd"]) if bsdf == "white" else None
    return c, _args(c, kd), dict(BSDF=bsdf, n_samples_x=N, rnd_seed=11, shadow_scale=shadow)


def ref_forward(ref, bsdf, N, light, lhw, shadow):
    c, args, kw = _fwd_case(bsdf, N, light, lhw, shadow)
    d, s = ref.env_shade(*args, **kw)
    return dict(diff=pick(d), spec=pick(s), diff_absmax=np.abs(d).max(), spec_absmax=np.abs(s).max(), masked_nonzero=(d[c["mask"] <= 0] != 0).sum())


@pytest.mark.parametrize("bsdf", BSDFS)
@pytest.mark.parametrize("N,light,lhw,shadow", FWD_CASES)
def test_forward_matches_the_compiled_reference(bsdf, N, light, lhw, shadow):
    c, args, kw = _fwd_case(bsdf, N, light, lhw, shadow)
    r = frozen_reference("fwd-%s-%d" % (bsdf, N))
    d_o, s_o = oracle().env_shade(*args, **kw)
    # host libm vs the oracle's fixed transcendental kernels may move a few rays per million to a neighbouring texel: 1e-4 bar, typically 1e-7
    assert rel_l2(pick(d_o), r["diff"]) < 1e-4 and np.abs(pick(d_o) - r["diff"]).max() < 1e-3 * max(float(r["diff_absmax"]), 1e-6)
    if bsdf == "pbr":
        assert rel_l2(pick(s_o), r["spec"]) < 1e-4
    else:
        assert r["spec_absmax"] == 0 and np.abs(s_o).max() == 0
    m = c["mask"] <= 0
    assert r["masked_nonzero"] == 0 and (d_o[m] == 0).all()


GRAD_NAMES = ("pos", "nrm", "kd", "ks", "light")


def _bwd_case():
    c = make_case(res=20, B=2, N=4, seed=2)
    g = np.random.default_rng(0)
    gd = g.uniform(size=c["pos"].shape).astype(np.float32); gs = g.uniform(size=c["pos"].shape).astype(np.float32)
    return c, gd, gs


def ref_backward(ref, bsdf):
    c, gd, gs = _bwd_case()
    g_r = ref.env_shade(*_args(c), grads=(gd, gs), BSDF=bsdf, n_samples_x=4, rnd_seed=11)
    out = {n: pick(g) for n, g in zip(GRAD_NAMES, g_r)}
    out.update({n + "_absmax": np.abs(g).max() for n, g in zip(GRAD_NAMES, g_r)})
    return out


@pytest.mark.parametrize("bsdf", ["pbr", "diffuse"])
def test_backward_matches_the_compiled_reference_within_fp32_noise(bsdf):
    """The hand-derived GGX adjoints are ill-conditioned in fp32 (DESIGN.md section 2): reference and oracle are both ~2-4e-4 away from the
    fp64 evaluation of the same samples, so they are compared with each other relative to that noise floor."""
    c, gd, gs = _bwd_case()
    kw = dict(BSDF=bsdf, n_samples_x=4, rnd_seed=11)
    r_ref = frozen_reference("bwd-" + bsdf)
    g_o = oracle().env_shade(*_args(c), grads=(gd, gs), **kw)
    o64 = oracle(f64=True)
    g64 = o64.env_shade(o64.scene(c["verts"], c["tris"]), *_args(c)[1:], grads=(gd, gs), sampling_gbuffer=(c["pos"], c["nrm"], c["kd"], c["ks"]), **kw)
    for name, a, r in zip(GRAD_NAMES, g_o, g64):
        if r_ref[name + "_absmax"] == 0:
            assert np.abs(a).max() == 0, name                    # 'diffuse': no kd / ks / pos gradient in either
            continue
        a, b, r = pick(a), r_ref[name], pick(r)
        floor = max(rel_l2(b, r), rel_l2(a, r))                  # fp32 noise of this quantity on this input
        assert rel_l2(a, b) < 2.0 * floor + 1e-5, (name, rel_l2(a, b), floor)
        assert rel_l2(a, r) < 1e-3 and rel_l2(b, r) < 1e-3, name


def ref_visibility(ref):
    c = make_case(res=16, B=1, N=4, seed=1)
    a = ref.env_shade(*_args(c), n_samples_x=4, rnd_seed=3, vis_mode="brute")
    b = ref.env_shade(*_args(c), n_samples_x=4, rnd_seed=3, vis_mode="bvh")
    d = ref.env_shade(*_args(c), n_samples_x=4, rnd_seed=4)
    return dict(diff=a[0], spec=a[1], brute_equals_bvh=np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]),
                seed_changes_output=not np.array_equal(a[0], d[0]))


def test_visibility_modes_and_determinism():
    r = frozen_reference("vis")
    assert r["brute_equals_bvh"] and r["seed_changes_output"]             # canonical LBVH == brute force, also through the reference
    c = make_case(res=16, B=1, N=4, seed=1)
    o = oracle()
    a = o.env_shade(*_args(c), n_samples_x=4, rnd_seed=3, vis_mode="brute")
    b = o.env_shade(*_args(c), n_samples_x=4, rnd_seed=3, vis_mode="bvh")
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert rel_l2(a[0], r["diff"]) < 1e-4 and rel_l2(a[1], r["spec"]) < 1e-4
    assert not np.array_equal(a[0], o.env_shade(*_args(c), n_samples_x=4, rnd_seed=4)[0])


SIGMAS = [1e-4, 0.7, 2.0]


def _denoise_case():
    g = np.random.default_rng(1)
    B, H, W = 2, 21, 17
    col = g.uniform(size=(B, H, W, 3)).astype(np.float32)
    nrm = g.normal(size=(B, H, W, 3)).astype(np.float32); nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    nrm[0, 3, 4] = 0                                                   # degenerate guide normal
    zdz = np.stack([g.uniform(1, 2, size=(B, H, W)), g.uniform(0.0, 0.02, size=(B, H, W))], -1).astype(np.float32)
    zdz[1, 5, 5, 1] = 0                                                # zero depth gradient: the FLT_EPS guard (denoising.cu:59,118)
    og = g.uniform(size=(B, H, W, 4)).astype(np.float32)
    return col, nrm, zdz, og


def ref_denoiser(ref, sigma):
    col, nrm, zdz, og = _denoise_case()
    return dict(fwd=ref.bilateral_fwd(col, nrm, zdz, sigma), bwd=ref.bilateral_bwd(nrm, zdz, sigma, og))


@pytest.mark.parametrize("sigma", SIGMAS)
def test_denoiser_matches_the_compiled_reference_kernels(sigma):
    """bilateral_denoiser_fwd_kernel / _bwd_kernel of denoising.cu, unmodified, on the host: the oracle restatement is bit-identical."""
    col, nrm, zdz, og = _denoise_case()
    r = frozen_reference("den-%g" % sigma)
    o = oracle()
    assert np.array_equal(o.bilateral_fwd(col, nrm, zdz, sigma), r["fwd"])
    assert np.array_equal(o.bilateral_bwd(nrm, zdz, sigma, og), r["bwd"])


_RU_OPS = [
    # name, oracle forward, oracle backward, input channels, output channels, extras (f0, i0, i1), oracle kwargs
    ("lambert", "lambert", "lambert_bwd", [3, 3], 1, (0.0, 0, 0), {}),
    ("frostbite", "frostbite_diffuse", "frostbite_diffuse_bwd", [3, 3, 3, 1], 1, (0.0, 0, 0), {}),
    ("fresnel", "fresnel_shlick", "fresnel_shlick_bwd", [3, 3, 1], 3, (0.0, 0, 0), {}),
    ("ndf", "ndf_ggx", "ndf_ggx_bwd", [1, 1], 1, (0.0, 0, 0), {}),
    ("lambda", "lambda_ggx", "lambda_ggx_bwd", [1, 1], 1, (0.0, 0, 0), {}),
    ("masking", "masking_smith", "masking_smith_bwd", [1, 1, 1], 1, (0.0, 0, 0), {}),
    ("specular", "pbr_specular", "pbr_specular_bwd", [3, 3, 3, 3, 1], 3, (0.08, 0, 0), {"min_roughness": 0.08}),
    ("bsdf", "pbr_bsdf", "pbr_bsdf_bwd", [3] * 6, 3, (0.08, 0, 0), {"min_roughness": 0.08, "bsdf": "lambert"}),
    ("bsdf", "pbr_bsdf", "pbr_bsdf_bwd", [3] * 6, 3, (0.08, 1, 0), {"min_roughness": 0.08, "bsdf": "frostbite"}),
    ("psn", "prepare_shading_normal", "prepare_shading_normal_bwd", [3] * 6, 3, (0.0, 1, 1), {"two_sided_shading": True, "opengl": True}),
    ("psn", "prepare_shading_normal", "prepare_shading_normal_bwd", [3] * 6, 3, (0.0, 0, 0), {"two_sided_shading": False, "opengl": False}),
]


def _ru_case(chans, out_c):
    g = np.random.default_rng(len(chans) * 7 + out_c)
    ins = [g.uniform(size=(2, 9, 11, c)).astype(np.float32) for c in chans]
    dout = g.uniform(size=(2, 9, 11, out_c)).astype(np.float32)
    return ins, dout


def ref_renderutils(ref, i):
    kernel, _, _, chans, out_c, extras, _ = _RU_OPS[i]
    ins, dout = _ru_case(chans, out_c)
    out = ref.renderutils(kernel + "_fwd", ins, out_c, f0=extras[0], i0=extras[1], i1=extras[2])
    grads = ref.renderutils(kernel + "_bwd", ins, dout=dout, f0=extras[0], i0=extras[1], i1=extras[2])
    return dict(out=out, n_grads=len(grads), **{"grad%d" % k: g for k, g in enumerate(grads)})


@pytest.mark.parametrize("kernel,fwd,bwd,chans,out_c,extras,kw", _RU_OPS)
def test_renderutils_kernels_match_the_compiled_reference(kernel, fwd, bwd, chans, out_c, extras, kw):
    """The CUDA kernels of render/renderutils/c_src/bsdf.cu and normal.cu themselves (unmodified, host build) on the reference tests'
    input distribution (torch.rand, tests/test_bsdf.py): where the CUDA code and the PyTorch twin differ (safe-normalize, division by
    the raw cosine), this is the flavour the oracle -- and the product -- must follow."""
    ins, dout = _ru_case(chans, out_c)
    r = frozen_reference("ru-%d" % _RU_OPS.index((kernel, fwd, bwd, chans, out_c, extras, kw)))
    o = oracle()
    a = getattr(o, fwd)(*ins, **kw)
    assert rel_l2(a, r["out"]) < 2e-6, (kernel, rel_l2(a, r["out"]))
    ga = getattr(o, bwd)(*ins, dout, **kw)
    ga = ga if isinstance(ga, (list, tuple)) else [ga]
    assert len(ga) == r["n_grads"]
    # the GGX adjoints (arm / alpha gradients of pbr_specular, pbr_bsdf) carry fp32 noise of a few 1e-4 on this input distribution
    # (tests/test_gpu_elementwise.py measures it against the fp64 oracle); everything else agrees to ~1e-6
    tol = 2e-4 if kernel in ("bsdf", "specular") else 2e-5
    for i, x in enumerate(ga):
        assert rel_l2(x, r["grad%d" % i]) < tol, (kernel, i, rel_l2(x, r["grad%d" % i]))


def _broadcast_case():
    g = np.random.default_rng(3)
    full = lambda: g.uniform(size=(2, 5, 6, 3)).astype(np.float32)
    kd, arm, pos, nrm = full(), full(), full(), full()
    view = g.uniform(size=(1, 1, 1, 3)).astype(np.float32); light = g.uniform(size=(2, 1, 1, 3)).astype(np.float32)
    return kd, arm, pos, nrm, view, light


def ref_broadcast(ref):
    return dict(out=ref.renderutils("bsdf_fwd", list(_broadcast_case()), 3, f0=0.08, i0=0))


def test_renderutils_broadcast_view_position():
    """view_pos / light_pos arrive as [1,1,1,3] (render.py passes the camera position broadcast): tensor.h:32 nhwcIndex semantics."""
    a = oracle().pbr_bsdf(*_broadcast_case())
    assert rel_l2(a, frozen_reference("bcast")["out"]) < 2e-6


LOSSES = ["l1", "mse", "relmse", "smape", "n2n"]
TONEMAPPERS = ["none", "log_srgb"]


def _loss_case():
    g = np.random.default_rng(5)
    img = (g.uniform(size=(2, 9, 7, 3)) * 4).astype(np.float32); tgt = (g.uniform(size=(2, 9, 7, 3)) * 4).astype(np.float32)
    img[0, 0, 0] = -0.5; img[0, 0, 1] = 70000.0; tgt[0, 1, 0] = 0.0
    return img, tgt


def ref_image_loss(ref, loss, tm):
    img, tgt = _loss_case()
    gi, gt = ref.image_loss(img, tgt, loss, tm, dout=1.0)
    return dict(loss=np.float64(ref.image_loss(img, tgt, loss, tm)), img_grad=gi, target_grad=gt)


@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("tm", TONEMAPPERS)
def test_image_loss_matches_the_compiled_reference(loss, tm):
    """imgLossFwdKernel / imgLossBwdKernel of loss.cu, unmodified ('n2n' selected by its enum: the reference's string mapping never
    reaches it, torch_bindings.cpp:727-737).  Bit-identical per-pixel losses and gradients, clamp / zero-gradient edges included."""
    img, tgt = _loss_case()
    r = frozen_reference("loss-%s-%s" % (loss, tm))
    o = oracle()
    assert abs(o.image_loss(img, tgt, loss, tm) / float(r["loss"]) - 1) < 1e-7
    ga = o.image_loss_bwd(img, tgt, loss, tm)
    assert np.array_equal(ga[0], r["img_grad"]) and np.array_equal(ga[1], r["target_grad"])


def _xfm_case(bp):
    g = np.random.default_rng(6)
    pts = g.uniform(size=(bp, 37, 3)).astype(np.float32); mtx = g.uniform(size=(3, 4, 4)).astype(np.float32)
    return pts, mtx, g


def ref_xfm(ref, is_points, bp):
    pts, mtx, g = _xfm_case(bp)
    out = ref.xfm(pts, mtx, is_points)
    d = g.uniform(size=out.shape).astype(np.float32)
    return dict(out=out, grad=ref.xfm(pts, mtx, is_points, dout=d))


@pytest.mark.parametrize("is_points", [True, False])
@pytest.mark.parametrize("bp", [1, 3])
def test_xfm_matches_the_compiled_reference(is_points, bp):
    pts, mtx, g = _xfm_case(bp)
    r = frozen_reference("xfm-%d-%d" % (is_points, bp))
    o = oracle()
    a = o.xfm(pts, mtx, is_points)
    assert np.array_equal(a, r["out"])
    d = g.uniform(size=a.shape).astype(np.float32)
    assert np.array_equal(o.xfm_bwd(mtx, d, is_points), r["grad"])


def _edge_case(chans, out_c):
    g = np.random.default_rng(11)
    shape = (1, 6, 8)
    ins = [g.normal(size=shape + (c,)).astype(np.float32) * (3.0 if c == 3 else 1.0) for c in chans]
    for a in ins:
        a[0, 0, 0] = 0.0                      # all-zero vectors / scalars
        a[0, 0, 1] = 1.0
        a[0, 0, 2] = -1.0
        a[0, 1, 0] = 1e-6
        a[0, 1, 1] = 1e4
    dout = g.uniform(size=shape + (out_c,)).astype(np.float32)
    return ins, dout


def ref_renderutils_edge(ref, i):
    kernel, _, _, chans, out_c, extras, _ = _RU_OPS[i]
    ins, dout = _edge_case(chans, out_c)
    out = ref.renderutils(kernel + "_fwd", ins, out_c, f0=extras[0], i0=extras[1], i1=extras[2])
    grads = ref.renderutils(kernel + "_bwd", ins, dout=dout, f0=extras[0], i0=extras[1], i1=extras[2])
    return dict(out=out, n_grads=len(grads), **{"grad%d" % k: g for k, g in enumerate(grads)})


@pytest.mark.parametrize("kernel,fwd,bwd,chans,out_c,extras,kw", _RU_OPS)
def test_renderutils_edge_inputs_match_the_compiled_reference(kernel, fwd, bwd, chans, out_c, extras, kw):
    """Inputs the reference tests never draw: zero vectors (safe-normalise guard), back-facing / grazing configurations (the cosine
    gates of bsdf.cu:146-160, 236), roughness at both ends of its clamp range, negative and > 1 values.  Forward values and gradients of
    the oracle must follow the compiled CUDA source through every branch; NaNs must appear in the same places."""
    ins, dout = _edge_case(chans, out_c)
    r = frozen_reference("edge-%d" % _RU_OPS.index((kernel, fwd, bwd, chans, out_c, extras, kw)))
    o = oracle()
    a, b = getattr(o, fwd)(*ins, **kw), r["out"]
    assert np.array_equal(np.isnan(a), np.isnan(b)), kernel
    ok = ~np.isnan(b)
    scale = max(float(np.abs(b[ok]).max()), 1e-30) if ok.any() else 1.0
    assert np.abs(a[ok] - b[ok]).max() <= 2e-5 * scale, (kernel, np.abs(a[ok] - b[ok]).max(), scale)
    ga = getattr(o, bwd)(*ins, dout, **kw)
    ga = ga if isinstance(ga, (list, tuple)) else [ga]
    assert len(ga) == r["n_grads"]
    for i, x in enumerate(ga):
        y = r["grad%d" % i]
        assert np.array_equal(np.isnan(x), np.isnan(y)), (kernel, i)
        ok = ~np.isnan(y) & np.isfinite(y)
        if ok.any():
            scale = max(float(np.abs(y[ok]).max()), 1e-30)
            assert np.abs(x[ok] - y[ok]).max() <= 1e-3 * scale, (kernel, i, np.abs(x[ok] - y[ok]).max(), scale)


def _edge_shade_case():
    N = 4
    c = make_case(res=16, B=1, N=N, seed=4)
    m = c["mask"][0] > 0
    ys, xs = np.nonzero(m)
    assert len(ys) > 40
    nrm, kd, ks, pos = c["nrm"].copy(), c["kd"].copy(), c["ks"].copy(), c["pos"].copy()
    px = lambda k: (0, ys[k], xs[k])
    nrm[px(0)] = 0.0
    nrm[px(1)] = -nrm[px(1)]                                  # back-facing shading normal
    ks[px(2)] = [0.0, 0.0, 0.0]; ks[px(3)] = [0.0, 1.0, 1.0]; ks[px(4)] = [0.0, 0.08, 0.5]
    kd[px(5)] = 0.0; kd[px(6)] = 1.0
    light = c["light"].copy(); light[3] = 0.0; light[10, ::2] = 0.0
    pdf, rows, cols = oracle().update_pdf(light)
    args = (c["scene"], c["mask"], c["ro"], pos, nrm, c["view"], kd, ks, light, pdf, rows, cols, c["perms"])
    g = np.random.default_rng(0)
    gd = g.uniform(size=c["pos"].shape).astype(np.float32); gs = g.uniform(size=c["pos"].shape).astype(np.float32)
    black = np.flatnonzero(light.max(-1) == 0)               # the planted black texels: always in the stored sample of the light gradient
    return args, dict(BSDF="pbr", n_samples_x=N, rnd_seed=21), gd, gs, black


def ref_edge_shade(ref):
    args, kw, gd, gs, black = _edge_shade_case()
    d, s = ref.env_shade(*args, **kw)
    g = ref.env_shade(*args, grads=(gd, gs), **kw)
    out = dict(diff=d, spec=s, light_nan=np.isnan(g[4]).sum())
    out.update({n: (pick(x, keep=black) if n == "light" else x) for n, x in zip(GRAD_NAMES, g)})
    return out


def test_env_shade_edge_materials_and_geometry_match_the_compiled_reference():
    """Pixels the synthetic scenes never contain: zero shading normal, camera behind the surface (NdotV < 0: bsdf_pdf's early-out,
    kernel.cu:376-378), roughness 0 and 1 (min-roughness clamp), pure metal, black albedo, and a probe with black rows / texels."""
    args, kw, gd, gs, black = _edge_shade_case()
    r = frozen_reference("edgeshade")
    d_r, s_r = r["diff"], r["spec"]
    d_o, s_o = oracle().env_shade(*args, **kw)
    assert np.array_equal(np.isnan(d_r), np.isnan(d_o)) and np.array_equal(np.isnan(s_r), np.isnan(s_o))
    f = lambda a: np.nan_to_num(a)
    assert rel_l2(f(d_o), f(d_r)) < 1e-4 and rel_l2(f(s_o), f(s_r)) < 1e-4
    g_o = oracle().env_shade(*args, grads=(gd, gs), **kw)
    assert np.isnan(g_o[4]).sum() == r["light_nan"]
    for name, a in zip(GRAD_NAMES, g_o):
        a, b = (pick(a, keep=black) if name == "light" else a), r[name]
        assert np.array_equal(np.isnan(a), np.isnan(b)), name
        assert rel_l2(f(a), f(b)) < 2e-3, (name, rel_l2(f(a), f(b)))        # fp32 noise of the GGX adjoints, larger at the roughness clamp


RAY_CASES = [(2, 4, "random", (32, 64)), (3, 8, "hdr", (64, 128)), (5, 3, "random", (256, 256))]


def _rays_case(seed, N, light, lhw):
    c = make_case(res=28, B=2, N=N, seed=seed, light=light, light_hw=lhw)
    return c, (c["scene"], c["mask"], c["ro"], c["pos"], c["nrm"], c["view"], c["kd"], c["ks"], c["light"], c["pdf"], c["rows"], c["cols"], c["perms"])


def ref_traced_rays(ref, seed, N, light, lhw):
    c, args = _rays_case(seed, N, light, lhw)
    _, _, dirs = ref.env_shade(*args, n_samples_x=N, rnd_seed=11, ray_log=True)
    m = c["mask"] > 0
    return dict(dirs=pick(dirs[m].reshape(-1, 3), 256), layout_ok=np.isfinite(dirs[m]).all() and np.isnan(dirs[~m]).all(),
                max_norm_error=np.abs(np.linalg.norm(dirs[m], axis=-1) - 1).max())


@pytest.mark.parametrize("seed,N,light,lhw", RAY_CASES)
def test_traced_rays_of_the_reference_hit_the_texels_the_oracle_records(seed, N, light, lhw):
    """Per-RAY agreement, not only per-pixel sums: the OptiX stand-in logs the direction of every shadow ray the reference's raygen
    program traces (sample-slot order: light i, BSDF i, ...); mapped to env texels they must equal the oracle's per-ray texel record --
    the record the CUDA product reproduces bit-exactly (tests/test_gpu_envshade.py).  Host libm vs the oracle's fixed transcendental
    kernels could move a ray across a texel border in the last ulp: tolerated at 1e-4 of the rays, observed 0 of 208 512."""
    c, args = _rays_case(seed, N, light, lhw)
    r = frozen_reference("rays-%d" % seed)
    assert r["layout_ok"] and r["max_norm_error"] < 1e-3          # exactly 2 n^2 unit rays per covered pixel, none elsewhere
    o = oracle()
    _, _, (rt, rv) = o.env_shade(*args, n_samples_x=N, rnd_seed=11, records=True)
    m = c["mask"] > 0
    want = pick(rt.reshape(m.shape + (-1,))[m].reshape(-1, 1), 256)[:, 0]
    tex = o.dirs_to_texels(r["dirs"], lhw[0], lhw[1])
    assert (tex != want).mean() <= 1e-4, int((tex != want).sum())


def reference_cases():
    """(case name, function of an oracle.Reference, arguments) of every frozen reference output this module compares with."""
    cases = [("fwd-%s-%d" % (b, N), ref_forward, (b, N, light, lhw, shadow)) for b in BSDFS for N, light, lhw, shadow in FWD_CASES]
    cases += [("bwd-" + b, ref_backward, (b,)) for b in ("pbr", "diffuse")]
    cases += [("vis", ref_visibility, ()), ("bcast", ref_broadcast, ()), ("edgeshade", ref_edge_shade, ())]
    cases += [("den-%g" % s, ref_denoiser, (s,)) for s in SIGMAS]
    cases += [("ru-%d" % i, ref_renderutils, (i,)) for i in range(len(_RU_OPS))]
    cases += [("edge-%d" % i, ref_renderutils_edge, (i,)) for i in range(len(_RU_OPS))]
    cases += [("loss-%s-%s" % (l, t), ref_image_loss, (l, t)) for l in LOSSES for t in TONEMAPPERS]
    cases += [("xfm-%d-%d" % (p, bp), ref_xfm, (p, bp)) for p in (True, False) for bp in (1, 3)]
    cases += [("rays-%d" % seed, ref_traced_rays, (seed, N, light, lhw)) for seed, N, light, lhw in RAY_CASES]
    return cases
