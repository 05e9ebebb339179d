"""Shared builders for the parity tests: seeded synthetic scenes (numpy) consumable by both the CPU
oracle and the CUDA product."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from nvdiffrecmc_b200 import synth  # noqa: E402

_ORACLE = {}


def oracle(f64=False):
    from oracle import Oracle
    if f64 not in _ORACLE:
        _ORACLE[f64] = Oracle(f64=f64)
    return _ORACLE[f64]


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def pick(a, k=128, keep=()):
    """A fixed sample of the rows (pixels, texels, rays) of `a` over all but its last dimension: at most k evenly spaced rows plus
    every row listed in `keep` (flat row indices of the inputs a test plants on purpose).  Only the frozen reference outputs too large
    to store whole are stored at these rows; all of `a` when it has no more than k rows."""
    a = np.asarray(a)
    rows = a.reshape(-1, a.shape[-1])
    even = np.linspace(0, rows.shape[0] - 1, min(k, rows.shape[0])).round().astype(np.int64)
    return rows[np.unique(np.concatenate([even, np.asarray(keep, np.int64)]))]


FROZEN_REFERENCE = os.path.join(ROOT, "tests", "golden", "ref_compiled_kernels.npz")
_FROZEN = {}


def frozen_reference(case):
    """The frozen outputs of the reference's own kernels for one test case (tests/golden/make_ref_kernels_golden.py): {field: array}."""
    if not _FROZEN:
        with np.load(FROZEN_REFERENCE) as z:
            for key in z.files:
                c, field = key.split("|", 1)
                _FROZEN.setdefault(c, {})[field] = z[key]
    return _FROZEN[case]


def make_case(res=32, B=1, N=4, mesh="blob+torus", level=2, light="random", light_hw=(32, 64), seed=0, ks_mode="random",
              perm_rows=512, closest=None):
    """Returns a dict of numpy arrays describing one env_shade problem.
    closest(verts, tris, ro[n,3], rd[n,3]) -> (tri_id[n], tuv[n,3]) overrides the oracle's brute-force primary visibility."""
    o = oracle()
    v, f = synth.scene_mesh(mesh, level=level, seed=5 + seed)
    vn = synth.vertex_normals(v, f)
    scene = o.scene(v, f)
    gbs = []
    for b in range(B):
        mv = synth.orbit_view(0.7 * b + 0.3 * seed)
        campos, ro, rd = synth.primary_rays(mv, res)
        if closest is None:
            tid, tuv = scene.closest_hit(ro.reshape(-1, 3), rd.reshape(-1, 3))
        else:
            tid, tuv = closest(v, f, ro.reshape(-1, 3), rd.reshape(-1, 3))
        gbs.append(synth.assemble_gbuffer(v, f, vn, np.asarray(tid).reshape(res, res), np.asarray(tuv).reshape(res, res, 3), campos,
                                          seed=1 + b + 10 * seed, ks_mode=ks_mode))
    st = lambda k: np.stack([g[k] for g in gbs])
    view = st("view_pos").reshape(B, 1, 1, 3)
    pos, sn, tg, gn = st("pos"), st("smooth_nrm"), st("tangent"), st("geom_nrm")
    nrm = o.prepare_shading_normal(pos, view, None, sn, tg, gn)       # render.py:99
    mask = st("mask")
    nrm = nrm * (mask[..., None] > 0)
    ro = (pos + nrm * np.float32(0.001)).astype(np.float32)             # render.py:110
    if light == "random":
        base = synth.random_light(light_hw[0], seed=2 + seed)
        if light_hw[0] != light_hw[1]:
            base = np.ascontiguousarray(np.random.default_rng(2 + seed).uniform(0.25, 0.75, size=(light_hw[0], light_hw[1], 3)), np.float32)
    else:
        base = synth.hdr_light(light_hw[0], light_hw[1], seed=7 + seed)
    pdf, rows, cols = o.update_pdf(base)
    perms = synth.make_perms(N, seed=3 + seed, rows=perm_rows)
    return dict(verts=v, tris=f, scene=scene, mask=mask, ro=ro, pos=pos, nrm=nrm.astype(np.float32), view=view.astype(np.float32),
                kd=st("kd"), ks=st("ks"), depth=st("depth"), smooth_nrm=sn, tangent=tg, geom_nrm=gn,
                light=base, pdf=pdf, rows=rows, cols=cols, perms=perms, N=N, B=B, res=res)
