"""CPU: on-disk formats (row f4): Radiance HDR (flat + run-length encoded) and Wavefront OBJ, round trips and hand-made files."""
import os

import numpy as np
import pytest

from nvdiffrecmc_b200 import assetio, synth


def test_hdr_roundtrip_and_precision(tmp_path):
    img = synth.hdr_light(24, 40)
    p = str(tmp_path / "a.hdr")
    assetio.save_hdr(p, img)
    back = assetio.load_hdr(p)
    assert back.shape == img.shape
    # RGBE: 8-bit mantissa shared exponent => relative error < 2^-7 of the pixel's max channel
    tol = img.max(-1, keepdims=True) / 128.0
    assert (np.abs(back - img) <= tol + 1e-30).all()
    assert assetio.load_hdr(p).dtype == np.float32


def test_hdr_reads_run_length_encoded_scanlines(tmp_path):
    """Hand-encode a 2 x 16 image with new-style RLE (what HDR tools and the reference's probes use)."""
    H, W = 2, 16
    rgbe = np.zeros((H, W, 4), np.uint8)
    rgbe[0, :, :] = [128, 64, 32, 129]                        # constant row -> pure run
    rgbe[1, :, 0] = np.arange(W) * 3; rgbe[1, :, 1] = 7; rgbe[1, :, 2] = np.arange(W)[::-1]; rgbe[1, :, 3] = 130
    body = bytearray()
    for y in range(H):
        body += bytes([2, 2, W >> 8, W & 255])
        for c in range(4):
            row = rgbe[y, :, c]
            if (row == row[0]).all():
                body += bytes([128 + W, int(row[0])])
            else:
                body += bytes([8]) + row[:8].tobytes() + bytes([8]) + row[8:].tobytes()      # two literal dumps
    p = str(tmp_path / "rle.hdr")
    with open(p, "wb") as f:
        f.write(b"#?RADIANCE\n# hand made\nFORMAT=32-bit_rle_rgbe\nEXPOSURE=1\n\n-Y 2 +X 16\n" + bytes(body))
    img = assetio.load_hdr(p)
    assert np.allclose(img[0, 3], np.array([128, 64, 32]) * 2.0 ** (129 - 136))
    assert np.allclose(img[1, 5], np.array([15, 7, 10]) * 2.0 ** (130 - 136))
    with open(p, "wb") as f:
        f.write(b"P6\n")
    with pytest.raises(ValueError):
        assetio.load_hdr(p)


def test_obj_roundtrip_and_polygons(tmp_path):
    v, f = synth.scene_mesh("blob", level=1)
    vn = synth.vertex_normals(v, f)
    p = str(tmp_path / "m.obj")
    assetio.save_obj(p, v, f, v_nrm=vn, t_nrm_idx=f, mtllib="m.mtl", usemtl="mat0")
    m = assetio.load_obj(p)
    assert np.array_equal(m["v_pos"], v) and np.array_equal(m["t_pos_idx"], f) and np.array_equal(m["t_nrm_idx"], f)
    assert np.allclose(m["v_nrm"], vn) and m["mtllib"] == "m.mtl" and m["usemtl"][0][0] == "mat0" and m["v_tex"] is None
    # quads, negative indices, texcoords with the OpenGL v flip (obj.py:77)
    q = str(tmp_path / "q.obj")
    with open(q, "w") as fh:
        fh.write("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 0.25\nf 1/1 2/2 3/3 4/4\nf -4/-4 -3/-3 -2/-2\n")
    m = assetio.load_obj(q)
    assert m["t_pos_idx"].tolist() == [[0, 1, 2], [0, 2, 3], [0, 1, 2]]
    assert m["t_tex_idx"].tolist() == [[0, 1, 2], [0, 2, 3], [0, 1, 2]] and np.allclose(m["v_tex"][3], [0, 0.75])


def test_reads_the_reference_assets_when_present():
    """Real files of the reference's data set, cut down to fixtures by tests/golden/make_asset_fixtures.py: the probe header with two of
    its run-length encoded scanlines (aerodynamics_workshop_2k.hdr, rows 0-1) and the first 64 faces of spot.obj with the lines they use."""
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    img = assetio.load_hdr(os.path.join(golden, "probe_rows2.hdr"))
    assert img.shape == (2, 2048, 3) and img.dtype == np.float32 and np.isfinite(img).all() and img.min() >= 0
    # rows 0-1 of the full 1024 x 2048 probe decode to these values (sum in float64, max)
    assert abs(img.astype(np.float64).sum() / 588.616943359375 - 1) < 1e-9 and img.max() == np.float32(0.07666015625)
    m = assetio.load_obj(os.path.join(golden, "spot_head.obj"))
    assert m["v_pos"].shape == (74, 3) and m["v_tex"].shape == (74, 2) and m["v_nrm"].shape == (74, 3)
    for k in ("t_pos_idx", "t_tex_idx", "t_nrm_idx"):
        assert m[k].shape == (64, 3) and m[k].min() == 0 and m[k].max() == 73, k
    assert m["mtllib"] == "spot.mtl" and m["usemtl"] == [("initialShadingGroup", 0)]
    assert np.abs(np.linalg.norm(m["v_nrm"], axis=-1) - 1).max() < 1e-3 and (m["v_tex"] >= 0).all() and (m["v_tex"] <= 1).all()


def test_mtl_roundtrip_and_reference_asset(tmp_path):
    from nvdiffrecmc_b200 import assetio
    mats = [{"name": "metal", "bsdf": "pbr", "kd": np.array([0.5, 0.25, 1.0], np.float32), "ks": np.array([0, 0.2, 1], np.float32), "map_kd": "tex/kd.png",
             "bump": "nrm.png"}, {"name": "second", "kd": np.array([1, 1, 1], np.float32)}]
    p = tmp_path / "m.mtl"
    assetio.save_mtl(str(p), mats)
    got = assetio.load_mtl(str(p))
    assert [m["name"] for m in got] == ["metal", "second"] and got[0]["map_kd"] == "tex/kd.png" and got[0]["bump"] == "nrm.png"
    assert np.array_equal(got[0]["ks"], mats[0]["ks"]) and np.allclose(got[0]["kd"], mats[0]["kd"]) and got[1]["bsdf"] == "pbr"
    (tmp_path / "c.mtl").write_text("# comment\nnewmtl a\nKd 0.1 0.2 0.3 # trailing\nbump -bm 1.0 n.png\nillum 2\n")
    c = assetio.load_mtl(str(tmp_path / "c.mtl"))[0]
    assert np.allclose(c["kd"], [0.1, 0.2, 0.3]) and c["bump"] == "n.png" and c["illum"][0] == 2
    m = assetio.load_mtl(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "spot_metal.mtl"))   # the reference's data/spot/metal.mtl
    assert len(m) == 1 and m[0]["name"] == "initialShadingGroup" and m[0]["bsdf"] == "pbr" and m[0]["map_kd"] == "spot_texture.png"
    assert np.array_equal(m[0]["ks"], np.float32([0.0, 0.2, 1.0]))


@pytest.mark.parametrize("shape,dtype", [((17, 23), np.uint8), ((9, 31, 3), np.uint8), ((8, 8, 4), np.uint8), ((5, 7, 2), np.uint8), ((6, 10, 3), np.uint16), ((4, 4), np.uint16)])
def test_png_roundtrip(tmp_path, shape, dtype):
    from nvdiffrecmc_b200 import assetio
    rng = np.random.default_rng(3)
    img = rng.integers(0, np.iinfo(dtype).max + 1, size=shape).astype(dtype)
    p = str(tmp_path / "a.png")
    assetio.save_png(p, img)
    got = assetio.load_png(p)
    assert got.dtype == dtype and got.shape == shape and np.array_equal(got, img)


def test_png_filters_and_float_write(tmp_path):
    """Decode all five scanline filter types (our writer only emits type 0, so build a file by hand)."""
    import struct, zlib
    from nvdiffrecmc_b200 import assetio
    rng = np.random.default_rng(4)
    H, W, C = 5, 6, 3
    img = rng.integers(0, 256, size=(H, W, C)).astype(np.uint8)
    flat = img.reshape(H, W * C).astype(np.int32)
    rows = []
    for y in range(H):
        ft = y % 5
        cur = flat[y]; up = flat[y - 1] if y else np.zeros_like(cur)
        left = np.concatenate([np.zeros(C, np.int32), cur[:-C]]); ul = np.concatenate([np.zeros(C, np.int32), up[:-C]])
        if ft == 0: enc = cur
        elif ft == 1: enc = cur - left
        elif ft == 2: enc = cur - up
        elif ft == 3: enc = cur - ((left + up) >> 1)
        else:
            p_ = left + up - ul
            pa, pb, pc = abs(p_ - left), abs(p_ - up), abs(p_ - ul)
            pred = np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, up, ul))
            enc = cur - pred
        rows.append(bytes([ft]) + (enc & 255).astype(np.uint8).tobytes())
    def chunk(t, b): return struct.pack(">I", len(b)) + t + b + struct.pack(">I", zlib.crc32(t + b) & 0xFFFFFFFF)
    p = tmp_path / "f.png"
    p.write_bytes(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0)) + chunk(b"IDAT", zlib.compress(b"".join(rows))) + chunk(b"IEND", b""))
    assert np.array_equal(assetio.load_png(str(p)), img)
    assetio.save_png(str(tmp_path / "g.png"), np.linspace(0, 1, 12, dtype=np.float32).reshape(3, 4))
    g = assetio.load_png(str(tmp_path / "g.png"))
    assert g.dtype == np.uint8 and g[0, 0] == 0 and g[-1, -1] == 255
    (tmp_path / "bad.png").write_bytes(b"not a png")
    with pytest.raises(ValueError):
        assetio.load_png(str(tmp_path / "bad.png"))
