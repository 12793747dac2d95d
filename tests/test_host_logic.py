"""not gpu: the C-ABI library loads and exports what include/b200rt.h declares; host-side logic (BVH builder, tile
bookkeeping, Camera/Image/CDF mirrors, scene generators). No CUDA compute is invoked."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_golden, scene_arrays


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_library_exports_every_declared_symbol(rt):
    header = open(os.path.join(ROOT, "include", "b200rt.h")).read()
    declared = sorted(set(re.findall(r"\b(b200rt_[a-z_0-9]+)\s*\(", header)))
    assert set(declared) == set(rt.binding.EXPORTS), set(declared) ^ set(rt.binding.EXPORTS)
    lib = rt.load_library()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert b"sm_100a" in lib.b200rt_version()


def test_header_cites_reference_interfaces():
    header = open(os.path.join(ROOT, "include", "b200rt.h")).read()
    for cite in ("render_kernel.h:24-46", "render_kernel.cpp:189-211", "flattened_bvh.h:25-39", "bvh.cpp:62-65", "utils.cpp:126-142",
                 "image_io.cpp:165-182", "bvh.cpp:19-60", "render_kernel.cpp:532-567"):
        assert cite in header


NO_GPU_CHECK = """
import numpy as np
import pytest
import sycl_ray_tracing_b200 as rt
g = np.load("tests/golden/scenes.npz")
a = {k: g["cornell_" + k] for k in ("tri9", "mat_idx", "mats10", "emissive")}
with pytest.raises(rt.B200RTError, match="no CUDA device"):
    rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"])
# the stages either side of the path have no CPU fallback either
with pytest.raises(rt.B200RTError, match="no CUDA device"):
    rt.BVH(a["tri9"], on_device=True)
with pytest.raises(rt.B200RTError, match="no CUDA device"):
    rt.quantise_rgba8(np.zeros((4, 4, 4), np.float32))
"""


def test_compute_fails_loudly_without_a_gpu():
    """In a process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so that GPU machines check it too."""
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join(p for p in (ROOT, os.environ.get("PYTHONPATH")) if p))
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", NO_GPU_CHECK], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("key", ["cornell", "mis", "area"])
def test_bvh_builder_invariants_bundled(rt, golden_scenes, key):
    a = scene_arrays(golden_scenes, key)
    for leaf, diag in ((4, True), (1, True), (15, False)):
        b = rt.BVH(a["tri9"], max_leaf_size=leaf, use_diag_slabs=diag)
        b.check()
        info = b.info()
        assert info["n_triangles"] == len(a["tri9"]) and info["max_leaf_size"] <= leaf and info["max_depth"] <= 60
        assert info["n_leaves"] == info["n_inner_nodes"] + 1 or info["n_inner_nodes"] == 1
        f = b.flatten()
        assert f.axis.shape == (info["n_inner_nodes"], 16) and f.tris.shape == (len(a["tri9"]), 12)
        assert sorted(f.tris[:, 3].view(np.int32).tolist()) == list(range(len(a["tri9"])))


def test_bvh_builder_degenerate_inputs(rt):
    rng = np.random.default_rng(3)
    cases = {
        "empty": np.zeros((0, 9), np.float32),
        "one": rng.random((1, 9)).astype(np.float32),
        "two": rng.random((2, 9)).astype(np.float32),
        "duplicates": np.repeat(rng.random((1, 9)).astype(np.float32), 300, axis=0),
        "collinear_centroids": np.concatenate([np.stack([np.full(9, i, np.float32) + np.array([0, 0, 0, 1, 0, 0, 0, 1, 0], np.float32) * 0 for i in range(100)])]),
        "huge_and_tiny": np.concatenate([rng.random((50, 9)).astype(np.float32) * 1e6, rng.random((50, 9)).astype(np.float32) * 1e-6]),
        "random_soup": (rng.random((5000, 9)).astype(np.float32) * 10 - 5),
    }
    for name, tri in cases.items():
        b = rt.BVH(tri)
        b.check()
        assert b.info()["max_depth"] <= 60, name


def test_bvh_builder_c2_mesh(rt):
    from sycl_ray_tracing_b200 import scenes
    c2 = scenes.c2_scene(nu=200, nv=100)
    assert c2["tri9"].shape == (40000, 9)
    b = rt.BVH(c2["tri9"])
    b.check()
    info = b.info()
    assert info["max_depth"] <= 40 and info["sah_cost"] < 200


def test_leaf_reference_packing(rt, golden_scenes):
    a = scene_arrays(golden_scenes, "mis")
    f = rt.BVH(a["tri9"]).flatten()
    refs = f.axis[:, 12:14].view(np.int32)
    counts = f.axis[:, 14:16].view(np.int32)
    leaf = refs < 0
    packed = ~refs[leaf]
    assert np.array_equal(packed & 15, counts[leaf]), "count lives in the low 4 bits of ~ref"
    first = packed >> 4
    assert (first >= 0).all() and (first + counts[leaf] <= len(a["tri9"])).all()
    assert counts[leaf].sum() == len(a["tri9"]) and (counts[~leaf] == 0).all()
    assert (refs[~leaf] > 0).all() and (refs[~leaf] < len(f.axis)).all()


def test_tiles_for_rank_partition(rt):
    from sycl_ray_tracing_b200 import distributed as D
    for (w, h) in [(1920, 1080), (512, 512), (100, 70), (16, 16), (17, 1), (3840, 2160)]:
        n = ((w + 15) // 16) * ((h + 15) // 16)
        for world in (1, 2, 3, 4, 8):
            per = [rt.tiles_for_rank(w, h, r, world) for r in range(world)]
            assert per == [D.tiles_for_rank(w, h, r, world) for r in range(world)]
            assert sum(per) == n and max(per) == per[0] and max(per) - min(per) <= 1
            seen = np.zeros((h, w), np.int32)
            for r in range(world):
                xy = D.tile_slot_coords(w, h, r, world, per[0])
                ok = xy[:, 0] >= 0
                np.add.at(seen, (xy[ok, 1], xy[ok, 0]), 1)
            assert (seen == 1).all(), "every pixel belongs to exactly one rank's tile buffer"
    assert rt.tiles_for_rank(0, 10, 0, 1) == 0 and rt.tiles_for_rank(10, 10, 2, 2) == 0


def test_tile_numbering_is_a_bijection_for_any_skew(monkeypatch):
    """device_types.h tile_xy / tile_number (mirrored in distributed.py): tile number <-> (tx, ty) is one-to-one whatever the
    skew (B200RT_TILE_SKEW), and skew 0 is plain row-major numbering."""
    from sycl_ray_tracing_b200 import distributed as D
    for skew in (0, 1, 5, 13, 120, 1000):
        monkeypatch.setattr(D, "TILE_SKEW", skew)
        for tiles_x, tiles_y in ((120, 68), (7, 5), (1, 9), (240, 135)):
            L = np.arange(tiles_x * tiles_y)
            tx, ty = D.tile_xy(L, tiles_x)
            assert ((0 <= tx) & (tx < tiles_x) & (0 <= ty) & (ty < tiles_y)).all()
            assert np.array_equal(D.tile_number(tx, ty, tiles_x), L)
            assert len(set(zip(tx.tolist(), ty.tolist()))) == len(L)
            if skew == 0:
                assert np.array_equal(tx, L % tiles_x) and np.array_equal(ty, L // tiles_x)


def test_camera_presets_and_image_mirror(rt, golden_cameras):
    for name, key in [("CORNELL_BOX_CAMERA", "cornell"), ("GANESHA_CAMERA", "ganesha"), ("ITE_ORB_CAMERA", "ite_orb"),
                      ("PBRT_DRAGON_CAMERA", "dragon"), ("MIS_CAMERA", "mis")]:
        assert np.array_equal(bits(getattr(rt.Camera, name).as_array17()), bits(golden_cameras[key])), name
    c = rt.Camera(45.0, rt.Translation(0.0, 0.0, 10.5))
    assert np.array_equal(bits(c.as_array17()), bits(golden_cameras["c2"]))
    # a rotated camera agrees with the reference's sinf/cosf to an ulp
    c = rt.Camera(45.0, rt.api.compose_transform(rt.RotationX(-45.0), rt.Translation(0.0, -1.0, 10.5)))
    assert np.allclose(c.as_array17(), golden_cameras["dragon"], rtol=3e-7, atol=1e-7)
    img = rt.Image(5, 3)
    assert img.width() == 5 and img.height() == 3 and np.array_equal(img.pixels[0, 0], [0, 0, 0, 1])
    m = rt.SimpleMaterial()
    assert np.array_equal(m.as_array10(), np.array([0, 0, 0, 1, 1, 0.2, 0.7, 1, 0, 1], np.float32))


def test_env_cdf_mirror_matches_reference(rt):
    from sycl_ray_tracing_b200 import scenes
    g = load_golden("env_cdf.npz")
    sky = scenes.procedural_sky(int(g["sky_w"]), int(g["sky_h"]))
    assert np.array_equal(bits(rt.compute_env_map_cdf(sky)), bits(g["cdf"]))
    r = load_golden("render_cornell_env.npz")
    assert np.array_equal(bits(rt.compute_env_map_cdf(r["env"])), bits(r["cdf"]))


def test_scene_generators_are_deterministic_and_sized(rt):
    from sycl_ray_tracing_b200 import scenes
    a, b = scenes.displaced_sphere(64, 32), scenes.displaced_sphere(64, 32)
    assert a.shape == (2 * 64 * 32, 9) and np.array_equal(bits(a), bits(b))
    c3 = scenes.c3_scene(nu=64, nv=32, sky_w=32, sky_h=16)
    assert len(c3["tri9"]) == 2 * 64 * 32 + 2 and c3["mat_idx"][-1] == 2 and c3["env"].shape == (16, 32, 4)
    assert c3["env"][..., :3].max() > 100 and (c3["env"][..., 3] == 0).all()
    out, inn = scenes.displaced_sphere(16, 8, outward=True), scenes.displaced_sphere(16, 8, outward=False)
    n_out = np.cross(out[:, 3:6] - out[:, :3], out[:, 6:9] - out[:, :3])
    assert (np.einsum("ij,ij->i", n_out, out[:, :3]) > 0).mean() > 0.95, "outward winding faces away from the centre"
    assert not np.array_equal(out, inn)
    assert [scenes.algorithmic_bytes_per_ray(n) for n in (32, 10 ** 6, 870000, 2 * 10 ** 7)] == [768, 3008, 3008, 3904]


def test_c2_known_answer_through_the_oracle():
    """SURVEY Appendix A: 502 161 of the 2 073 600 un-jittered primary rays hit the 1M-triangle C2 mesh."""
    from oracle.oracle import PortOracle
    from sycl_ray_tracing_b200 import scenes
    c2 = scenes.c2_scene()
    ps = PortOracle().scene_from_arrays(c2["tri9"], c2["mat_idx"], c2["mats10"], c2["emissive"])
    prim, t, _ = ps.primary(c2["camera"].as_array17(), 1920, 1080, mode=0)
    assert int((prim >= 0).sum()) == 502161


# ---- the 8-ary quantised layout, decoded and traversed on the CPU (numpy) -----------------------------------------------------------
def _wide_grid(q):
    """plane byte -> grid value: the float whose bits are 0x43000000 | q << 16 (csrc/pt_device.cuh B200RT_Q)."""
    return (np.uint32(0x43000000) | (np.asarray(q, np.uint32) << np.uint32(16))).view(np.float32)


def _wide_closest(flat, ray):
    """Independent restatement of trav8_node / trav8_tris for ONE ray on the host arrays: boxes decoded in float64
    (plane = p + 2^(e-127) * v(q)), children visited in slot ^ (7 - octant) order through an explicit stack of node groups,
    exact triangle tests on the leaf-ordered stream (a, e1, e2 as stored), ties to the lower original index."""
    wide, tris = flat.wide, flat.tris
    o = ray[:3].astype(np.float64); d = ray[3:].astype(np.float64)
    inv = 1.0 / np.where(np.abs(d) < 1e-20, np.copysign(1e-20, d), d)
    octant = 7 - (int(inv[0] < 0) | (int(inv[1] < 0) << 1) | (int(inv[2] < 0) << 2))
    best_t, best_p, visited = np.inf, -1, 0
    stack = [0]
    f32 = np.float32
    o32, d32 = ray[:3].astype(f32), ray[3:].astype(f32)
    while stack:
        n = wide[stack.pop()]
        visited += 1
        cell = np.ldexp(1.0, n["e"].astype(np.int64) - 127)
        lo = np.stack([n["p"][a] + cell[a] * _wide_grid(n[k]).astype(np.float64) for a, k in enumerate(("lox", "loy", "loz"))], 1)   # [slot, axis]
        hi = np.stack([n["p"][a] + cell[a] * _wide_grid(n[k]).astype(np.float64) for a, k in enumerate(("hix", "hiy", "hiz"))], 1)
        t0 = (lo - o) * inv; t1 = (hi - o) * inv
        tn = np.maximum(np.minimum(t0, t1).max(1), 0.0); tf = np.minimum(np.maximum(t0, t1).min(1), best_t)
        hit = tn <= tf * (1 + 1e-6)
        imask, valid = int(n["imask"]), int(n["valid24"])
        inner = [s for s in range(8) if hit[s] and (imask >> s) & 1]
        # triangles first (as the device does), then the inner children front to back: push in reverse priority
        for s in range(8):
            if not hit[s] or (imask >> s) & 1:
                continue
            for i in range(3):
                b = 3 * s + i
                if not (valid >> b) & 1:
                    continue
                slot = int(n["tri_base"]) + bin(valid & ((1 << b) - 1)).count("1")
                a_, prim = tris[slot, 0:3], int(tris[slot, 3:4].view(np.int32)[0])
                e1, e2 = tris[slot, 4:7], tris[slot, 8:11]
                # triangle.h:16-60 with vec.h's left-to-right dot and cross, every operation rounded to float32
                dot = lambda p_, q_: f32(f32(f32(p_[0] * q_[0]) + f32(p_[1] * q_[1])) + f32(p_[2] * q_[2]))
                cross = lambda p_, q_: np.array([f32(f32(p_[1] * q_[2]) - f32(p_[2] * q_[1])), f32(f32(p_[2] * q_[0]) - f32(p_[0] * q_[2])),
                                                 f32(f32(p_[0] * q_[1]) - f32(p_[1] * q_[0]))], f32)
                h = cross(d32, e2); det = dot(e1, h)
                if -1e-7 < det < 1e-7:
                    continue
                f = f32(f32(1.0) / det); s_ = (o32 - a_).astype(f32); u = f32(f * dot(s_, h))
                if u < 0 or u > 1:
                    continue
                q = cross(s_, e1); v = f32(f * dot(d32, q))
                if v < 0 or f32(u + v) > 1:
                    continue
                t = f32(f * dot(e2, q))
                if t > 1e-7 and (t < best_t or (t == best_t and prim < best_p)):
                    best_t, best_p = float(t), prim
        for s in sorted(inner, key=lambda s: s ^ octant):           # lowest priority first onto the stack
            rank = bin(imask & ((1 << s) - 1)).count("1")
            stack.append(int(n["child_base"]) + rank)
    return best_p, (np.float32(best_t) if best_p >= 0 else np.float32(-1.0)), visited


@pytest.mark.parametrize("key", ["cornell", "area", "soup"])
def test_wide_layout_decodes_and_traverses_on_the_cpu(rt, golden_scenes, key):
    """The 80-byte node format is a contract between the builders and the kernels: decode it independently (numpy) and find
    the same closest hits as a brute force over all triangles. Also pins that traversal prunes (visits far fewer nodes than exist)."""
    from conftest import brute_force_closest
    rng = np.random.default_rng(23)
    tri = (rng.random((400, 9)).astype(np.float32) * 4 - 2) if key == "soup" else scene_arrays(golden_scenes, key)["tri9"]
    flat = rt.BVH(tri).flatten()
    assert flat.wide.dtype.itemsize == 80 and len(flat.wide) == flat.bvh.info()["n_wide_nodes"] >= 1
    lo, hi = tri.reshape(-1, 3).min(0), tri.reshape(-1, 3).max(0)
    n = 60
    o = (lo + (hi - lo) * rng.random((n, 3))).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    rays = np.concatenate([o, d], 1).astype(np.float32)
    rays = np.concatenate([rays, np.array([[0, 1, 3.5, 0, 0, -1], [0, 1, 3.5, 1, 0, 0], [5, 5, 5, 0, 1, 0]], np.float32)])     # axis-parallel, and one that misses
    bp, bt = brute_force_closest(tri, rays)
    visited = 0
    for r in range(len(rays)):
        p, t, v = _wide_closest(flat, rays[r])
        visited += v
        assert p == bp[r], (key, r, p, bp[r])
        assert np.float32(t).view(np.uint32) == np.float32(bt[r]).view(np.uint32), (key, r)
    if len(flat.wide) > 40:
        assert visited / len(rays) < 0.5 * len(flat.wide)


def test_c_abi_compiles_and_links_as_plain_c(rt, tmp_path):
    """include/b200rt.h is a C header: a C99 translation unit (-pedantic -Werror) includes it, links libb200rt.so, builds and
    checks a BVH on the host through the C ABI and reads the 8-ary nodes back; the compute call fails loudly without a GPU."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text(r"""
#include <stdio.h>
#include <string.h>
#include "b200rt.h"
int main(void)
{
    float tri[4 * 9] = { 0,0,0, 1,0,0, 0,1,0,   0,0,1, 1,0,1, 0,1,1,   2,0,0, 3,0,0, 2,1,0,   0,2,0, 1,2,0, 0,3,0 };
    b200rt_bvh* bvh = NULL;
    b200rt_bvh_options o;
    b200rt_bvh_info info;
    const void* nodes = NULL;
    int n_nodes = -1;
    b200rt_bvh_default_options(&o);
    if (b200rt_bvh_build(tri, 4, &o, &bvh) != B200RT_OK) { printf("build: %s\n", b200rt_last_error()); return 1; }
    if (b200rt_bvh_check(bvh, tri, 4) != B200RT_OK) { printf("check: %s\n", b200rt_last_error()); return 2; }
    if (b200rt_bvh_get_info(bvh, &info) != B200RT_OK || info.n_triangles != 4) return 3;
    if (b200rt_bvh_get_wide_nodes(bvh, &nodes, &n_nodes) != B200RT_OK || n_nodes < 1 || !nodes) return 4;
    printf("%s nodes=%d depth=%d\n", b200rt_version(), n_nodes, info.wide_max_depth);
    b200rt_bvh_destroy(bvh);
    return 0;
}
""")
    exe = tmp_path / "abi"
    libdir = os.path.join(ROOT, "sycl-ray-tracing_b200")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-lb200rt", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out and "nodes=1" in out


def test_env_alias_table_encodes_luminance_over_total(rt):
    """The alias table B200RT_FLAG_ENV_ALIAS samples from: the distribution it implies (accept texel i with prob[i], else take
    alias[i], i uniform) must be each texel's luminance over the exact total — to 1e-6 relative (prob is stored as float)."""
    from sycl_ray_tracing_b200 import scenes
    rng = np.random.default_rng(9)
    for env in (rng.random((16, 32, 4)).astype(np.float32) * np.array([1, 1, 1, 0], np.float32),
                scenes.procedural_sky(128, 64),                                                   # sun 5e4 next to sky 0.3: the float running-sum CDF stagnates here
                np.concatenate([np.zeros((4, 8, 4), np.float32), np.ones((4, 8, 4), np.float32)])):      # zero-luminance texels are never picked
        prob, alias, total = rt.env_alias_table(env)
        n = prob.size
        e64 = env.astype(np.float64)
        lum = (0.3086 * e64[..., 0] + 0.6094 * e64[..., 1] + 0.0820 * e64[..., 2]).astype(np.float32).astype(np.float64).ravel()    # image.h:80-85
        assert abs(total - lum.sum()) <= 1e-9 * lum.sum()
        assert ((prob >= 0) & (prob <= 1)).all() and ((alias >= 0) & (alias < n)).all()
        implied = prob.astype(np.float64) / n
        np.add.at(implied, alias, (1.0 - prob.astype(np.float64)) / n)
        want = lum / lum.sum()
        assert np.abs(implied - want).max() <= 1e-6 * want.max() + 1e-12
        assert (implied[lum == 0] == 0).all()
