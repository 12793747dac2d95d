"""Host-side ingest of the C ABI (b200rt_obj_load, b200rt_hdr_load): CPU tests, no GPU needed.

The OBJ reader is checked against the reference's own parse of its three bundled scenes (tests/golden/scenes.npz, frozen from
Utils::parse_obj by make_golden.py); the HDR reader against files in the layout the reference's stb writer produces (run-length
encoded scanlines) and against a flat file, both written here from the format description."""
import os

import numpy as np
import pytest

from conftest import load_golden

OBJS = {"cornell": "cornell_pbr.obj", "mis": "MIS.obj", "area": "test_triangle_area_sampling.obj"}


def write_obj_from_parse(path, tri9, mat_idx, mats10):
    """OBJ + MTL whose parse is (tri9, mat_idx, mats10): shared vertices written once with round-trip precision, one MTL
    record per material slot after the built-in slot 0, `usemtl` wherever the slot changes. Every slot of mat_idx must be >= 1."""
    assert (mat_idx >= 1).all()
    g = lambda v: format(float(v), ".9g")
    with open(path + ".mtl", "w") as f:
        for i, m in enumerate(mats10[1:], start=1):
            f.write(f"newmtl m{i}\nKe {g(m[0])} {g(m[1])} {g(m[2])}\nKd {g(m[4])} {g(m[5])} {g(m[6])}\nPm {g(m[8])}\nPr {g(m[9])}\nillum 2\n\n")
    corners = np.ascontiguousarray(tri9, np.float32).reshape(-1, 3)
    _, first, index = np.unique(corners.view(np.uint32), axis=0, return_index=True, return_inverse=True)
    order = np.argsort(first)                                # vertices in order of first use
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    faces = rank[index.reshape(-1)].reshape(-1, 3) + 1
    with open(path + ".obj", "w") as f:
        f.write(f"mtllib {os.path.basename(path)}.mtl\n")
        f.writelines(f"v {g(x)} {g(y)} {g(z)}\n" for x, y, z in corners[first[order]])
        cur = None
        for (a, b, c), m in zip(faces, mat_idx):
            if m != cur:
                cur = m
                f.write(f"usemtl m{m}\n")
            f.write(f"f {a} {b} {c}\n")


@pytest.mark.parametrize("key", list(OBJS))
def test_parse_obj_equals_the_reference_parse(rt, key, tmp_path):
    """The reference's bundled OBJ files are not part of this repository: the scene is written back from the reference's frozen
    parse of OBJS[key] (same triangles, materials and material runs) and the library's reader must reproduce that parse bit for bit."""
    g = load_golden("scenes.npz")
    base = str(tmp_path / os.path.splitext(OBJS[key])[0])
    write_obj_from_parse(base, g[f"{key}_tri9"], g[f"{key}_mat_idx"], g[f"{key}_mats10"])
    o = rt.parse_obj(base + ".obj")
    assert np.array_equal(o["tri9"].view(np.uint32), g[f"{key}_tri9"].view(np.uint32)), "triangle list (order, quad diagonals) must match"
    assert np.array_equal(o["mat_idx"], g[f"{key}_mat_idx"]) and np.array_equal(o["emissive"], g[f"{key}_emissive"])
    assert np.array_equal(o["mats10"].view(np.uint32), g[f"{key}_mats10"].view(np.uint32))


def test_parse_obj_rules(rt, tmp_path):
    """A hand-written OBJ: negative indices, v/vt/vn references, a quad cut along its shorter diagonal (both cases), a pentagon
    fanned, faces before any usemtl -> default material 0, roughness clamp, illum 0 rule, emissive list, errors."""
    (tmp_path / "m.mtl").write_text("newmtl light\nKe 2 2 2\nKd 0 0 0\nPr 0.5\nPm 0.25\nillum 2\n\nnewmtl glossy\nKd 0.1 0.2 0.3\nPr 0\nPm 1\nillum 2\n"
                                   "newmtl legacy\nKd 0.5 0.5 0.5\nPr 0.3\nPm 0.7\n")
    (tmp_path / "s.obj").write_text(
        "mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nv 3 0 0\nv 0 0.5 0\nv 2 2 1\n"
        "f 1 2 3\n"                       # default material
        "usemtl light\nf 1/1/1 2/2/2 3/3/3 4/4/4\n"          # square: d02 == d13 -> 1-3 diagonal
        "usemtl glossy\nf 1 5 3 6\n"      # |p0-p2|^2 = 2 < |p1-p3|^2 = 9.25 -> 0-2 diagonal
        "usemtl legacy\nf -7 -6 -5 -4 -1\n")
    o = rt.parse_obj(str(tmp_path / "s.obj"))
    V = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [3, 0, 0], [0, 0.5, 0], [2, 2, 1]], np.float32)
    T = lambda a, b, c: np.concatenate([V[a], V[b], V[c]])
    want = np.stack([T(0, 1, 2), T(0, 1, 3), T(1, 2, 3), T(0, 4, 2), T(0, 2, 5), T(0, 1, 2), T(0, 2, 3), T(0, 3, 6)])
    assert np.array_equal(o["tri9"], want)
    assert o["mat_idx"].tolist() == [0, 1, 1, 2, 2, 3, 3, 3] and o["emissive"].tolist() == [1, 2]
    m = o["mats10"]
    assert m.shape == (4, 10) and m[0].tolist() == [1, 0, 1, 1, 0, 0, 0, 1, 0, 1]
    assert m[1].tolist() == [2, 2, 2, 1, 0, 0, 0, 1, 0.25, 0.5]
    assert np.allclose(m[2], [0, 0, 0, 1, 0.1, 0.2, 0.3, 1, 1.0, 0.01])            # roughness 0 clamped to 1e-2 (utils.cpp:82)
    assert np.allclose(m[3], [0, 0, 0, 1, 0.5, 0.5, 0.5, 1, 0.0, 1.0])             # no illum line = illum 0: default roughness / metalness
    with pytest.raises(rt.B200RTError):
        rt.parse_obj(str(tmp_path / "missing.obj"))
    (tmp_path / "bad.obj").write_text("v 0 0 0\nv 1 0 0\nf 1 2 9\n")
    with pytest.raises(rt.B200RTError):
        rt.parse_obj(str(tmp_path / "bad.obj"))
    (tmp_path / "nomtl.obj").write_text("mtllib nothere.mtl\nv 0 0 0\n")
    with pytest.raises(rt.B200RTError):
        rt.parse_obj(str(tmp_path / "nomtl.obj"))


def write_flat_hdr(path, rgb):
    h, w, _ = rgb.shape
    m = rgb.max(axis=-1)
    mant, ex = np.frexp(m.astype(np.float64))
    scale = np.where(m > 1e-32, mant * 256.0 / np.maximum(m, 1e-38), 0.0)
    rgbe = np.zeros((h, w, 4), np.uint8)
    rgbe[..., :3] = np.clip(rgb * scale[..., None], 0, 255).astype(np.uint8)
    rgbe[..., 3] = np.where(m > 1e-32, ex + 128, 0).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n" + f"-Y {h} +X {w}\n".encode())
        f.write(rgbe.tobytes())
    dec = np.where(rgbe[..., 3:4] != 0, rgbe[..., :3].astype(np.float32) * np.ldexp(np.float32(1.0), rgbe[..., 3:4].astype(np.int32) - 136), 0.0)
    return dec.astype(np.float32)


def test_hdr_reader_flat_scanlines(rt, tmp_path):
    rng = np.random.default_rng(0)
    rgb = (rng.random((9, 13, 3)) * np.array([1.0, 100.0, 1e4])).astype(np.float32)
    rgb[2, 3] = 0.0
    dec = write_flat_hdr(str(tmp_path / "a.hdr"), rgb)
    got = rt.read_image_float(str(tmp_path / "a.hdr"), flip_y=True)
    assert got.shape == (9, 13, 3) and np.array_equal(got, dec[::-1])               # row 0 = bottom row, as the reference loads it
    assert np.array_equal(rt.read_image_float(str(tmp_path / "a.hdr"), flip_y=False), dec)
    assert np.abs(got - rgb[::-1]).max() <= rgb.max() / 128.0
    (tmp_path / "bad.hdr").write_bytes(b"P6\n1 1\n255\nxxx")
    with pytest.raises(rt.B200RTError):
        rt.read_image_float(str(tmp_path / "bad.hdr"))


def stb_rle_channel(comp):
    """One channel of a scanline as stb_image_write's stbi_write_hdr encodes it: literal dumps of at most 128 bytes (count byte
    1..128), runs of three or more equal bytes as (128 + length, value) with length at most 127."""
    out, w, x = bytearray(), len(comp), 0
    while x < w:
        r = x
        while r + 2 < w and not (comp[r] == comp[r + 1] == comp[r + 2]):
            r += 1
        if r + 2 >= w:
            r = w
        while x < r:
            n = min(r - x, 128)
            out += bytes([n]) + bytes(comp[x:x + n])
            x += n
        if r < w:
            while r < w and comp[r] == comp[x]:
                r += 1
            while x < r:
                n = min(r - x, 127)
                out += bytes([128 + n, comp[x]])
                x += n
    return bytes(out)


def write_stb_hdr(path, rgb):
    """The reference's write_image_hdr (stbi_write_hdr with the vertical flip on): stb's header, scanlines of width 8..32767
    run-length encoded channel by channel, other widths flat. Returns the float image read_image_float makes of the file
    (flip on load; channel = byte * 2^(e - 136), e == 0 -> 0)."""
    h, w, _ = rgb.shape
    rgb = np.ascontiguousarray(rgb, np.float32)
    m = rgb.max(axis=-1)
    mant, ex = np.frexp(m.astype(np.float64))
    scale = np.where(m >= np.float32(1e-32), mant.astype(np.float32) * np.float32(256.0) / np.maximum(m, np.float32(1e-32)), np.float32(0))
    rgbe = np.zeros((h, w, 4), np.uint8)
    rgbe[..., :3] = (rgb * scale[..., None]).astype(np.uint8)
    rgbe[..., 3] = np.where(m >= np.float32(1e-32), ex + 128, 0).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\n# Written by stb_image_write\nFORMAT=32-bit_rle_rgbe\n")
        f.write(f"EXPOSURE=          1.0000000000000\n\n-Y {h} +X {w}\n".encode())
        for row in rgbe[::-1]:                                  # file row 0 = the image's last row
            if 8 <= w < 32768:
                f.write(bytes([2, 2, w >> 8, w & 0xFF]) + b"".join(stb_rle_channel(row[:, c].tobytes()) for c in range(4)))
            else:
                f.write(row.tobytes())
    f1 = np.ldexp(np.float32(1.0), rgbe[..., 3].astype(np.int32) - 136).astype(np.float32)
    return np.where(rgbe[..., 3:4] != 0, rgbe[..., :3].astype(np.float32) * f1[..., None], np.float32(0)).astype(np.float32)


def test_hdr_reader_equals_the_reference_loader(rt, tmp_path):
    """The reference's write_image_hdr -> Utils::read_image_float round trip (stb: run-length encoded scanlines, flat below
    8 pixels of width) against b200rt_hdr_load on the same file: bit for bit."""
    from sycl_ray_tracing_b200 import scenes
    for w, h in ((256, 128), (6, 5), (40, 3)):
        env = np.ascontiguousarray(scenes.procedural_sky(256, 128)[:h, :w, :3])
        path = str(tmp_path / f"sky_{w}.hdr")
        ref = write_stb_hdr(path, env)
        mine = rt.read_image_float(path)
        assert np.array_equal(mine.view(np.uint32), ref.view(np.uint32)), (w, h)
        assert np.abs(mine - env).max() <= env.max() / 128.0
