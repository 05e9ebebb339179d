"""Cut small real-world asset fixtures for tests/test_assetio.py out of the reference's data files (run where the reference tree exists):

  * probe_rows2.hdr: the header of data/irrmaps/aerodynamics_workshop_2k.hdr with its resolution line set to two rows, followed by the
    file's first two run-length encoded scanlines, byte for byte;
  * spot_head.obj: the first 64 faces of data/spot/spot.obj with the `v` / `vt` / `vn` lines they use (verbatim, in file order) and the
    file's other statements; face indices are renumbered to the kept lines.

usage: python tests/golden/make_asset_fixtures.py <reference root>"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
N_ROWS, N_FACES = 2, 64


def scanline_end(data, pos, width):
    """Byte offset after one new-style RLE scanline starting at `pos`."""
    assert data[pos] == 2 and data[pos + 1] == 2 and (data[pos + 2] << 8 | data[pos + 3]) == width
    pos += 4
    for _ in range(4):
        n = 0
        while n < width:
            c = data[pos]
            pos, n = (pos + 2, n + c - 128) if c > 128 else (pos + 1 + c, n + c)
        assert n == width
    return pos


def cut_hdr(src, dst):
    data = open(src, "rb").read()
    head_end = data.index(b"\n\n") + 2
    res_end = data.index(b"\n", head_end) + 1
    ys, h, xs, w = data[head_end:res_end].split()
    assert ys == b"-Y" and xs == b"+X"
    pos = res_end
    for _ in range(N_ROWS):
        pos = scanline_end(data, pos, int(w))
    with open(dst, "wb") as f:
        f.write(data[:head_end] + b"-Y %d +X %d\n" % (N_ROWS, int(w)) + data[res_end:pos])


def cut_obj(src, dst):
    lines = open(src).read().splitlines()
    kinds = {"v": [], "vt": [], "vn": []}
    for i, l in enumerate(lines):
        k = l.split(" ", 1)[0]
        if k in kinds:
            kinds[k].append(i)
    faces = [i for i, l in enumerate(lines) if l.startswith("f ")][:N_FACES]
    used = {k: set() for k in kinds}
    for i in faces:
        for corner in lines[i].split()[1:]:
            for k, idx in zip(("v", "vt", "vn"), corner.split("/")):
                used[k].add(int(idx) - 1)
    keep_line = {kinds[k][j] for k in kinds for j in used[k]}
    renum = {k: {j: n + 1 for n, j in enumerate(sorted(used[k]))} for k in kinds}
    out = []
    for i, l in enumerate(lines):
        k = l.split(" ", 1)[0]
        if k in kinds:
            if i in keep_line:
                out.append(l)
        elif k == "f":
            if i in faces:
                out.append("f " + " ".join("/".join(str(renum[kk][int(x) - 1]) for kk, x in zip(("v", "vt", "vn"), c.split("/")))
                                           for c in l.split()[1:]))
        else:
            out.append(l)
    with open(dst, "w") as f:
        f.write("\n".join(out) + "\n")
    return {k: len(used[k]) for k in kinds}


if __name__ == "__main__":
    ref = sys.argv[1]
    cut_hdr(os.path.join(ref, "data", "irrmaps", "aerodynamics_workshop_2k.hdr"), os.path.join(HERE, "probe_rows2.hdr"))
    print("spot_head.obj:", cut_obj(os.path.join(ref, "data", "spot", "spot.obj"), os.path.join(HERE, "spot_head.obj")))
