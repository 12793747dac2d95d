"""-m gpu: in-place BVH rebuilds of a resident scene (b200rt_scene_rebuild_bvh[_device]).

A rebuild must leave the scene holding exactly the tree b200rt_bvh_build_device builds for the new vertices (two device builds of
the same vertices are identical, so that tree is an oracle), and, since closest hits do not depend on the tree, every output must
equal a freshly created scene's bit for bit, as after a refit. The deformations, the output set and its comparison are the refit
tests'."""
import ctypes as C
import gc

import numpy as np
import pytest

from conftest import scene_arrays
from test_gpu_refit import (BOUNCES, DEFORMATIONS, H, SPP, W, assert_arrays_equal, assert_same_outputs, build_scene, c3_small,
                            camera_for, outputs, rigid, sah_numpy, smooth, twist)

pytestmark = pytest.mark.gpu

INFO_KEYS = ("n_triangles", "n_inner_nodes", "n_leaves", "max_leaf_size", "max_depth", "has_diag_slabs", "n_wide_nodes", "wide_max_depth")


def builder_arrays(rt, tri):
    f = rt.BVH(tri, on_device=True).flatten()
    return dict(wide=f.wide.copy(), axis=f.axis.copy(), diag=f.diag.copy(), tris=f.tris.copy()), f.bvh.info()


def assert_is_device_build(rt, sc, tri, what):
    """The scene's arrays and info are b200rt_bvh_build_device's for tri (build_seconds apart; sah_cost to 1e-12). A scene's sah_cost
    is sah_cost_of over the binary records, which is what b200rt_bvh_get_info reports for a device-built tree; the host builder
    reports its own figure, over its unpadded build nodes."""
    want, winfo = builder_arrays(rt, tri)
    assert_arrays_equal(sc.bvh_arrays(), want, what)
    info = sc.bvh_info()
    for k in INFO_KEYS:
        assert info[k] == winfo[k], f"{what}: {k} {info[k]} != {winfo[k]}"
    sah = sah_numpy(want["axis"]) if winfo["has_diag_slabs"] else winfo["sah_cost"]
    assert abs(info["sah_cost"] - sah) <= 1e-12 * sah, (what, info["sah_cost"], sah)
    assert info["build_seconds"] > 0.0
    return info


def scene_for(rt, golden_scenes, key):
    a = c3_small() if key == "c3small" else scene_arrays(golden_scenes, key)
    return a, np.ascontiguousarray(a["tri9"], np.float32)


# ---- 1: the builder's bytes -----------------------------------------------------------------------------------------------------------
IDENTITY = [("cornell", "host"), ("mis", "host"), ("area", "host"), ("cornell", "device"), ("mis", "device"), ("area", "device"),
            ("c3small", "host"), ("c3small", "device")]


@pytest.mark.parametrize("key,kind", IDENTITY)
def test_rebuild_holds_the_device_builders_tree(rt, golden_scenes, key, kind):
    """C3-small's ground quad is outsized: the device builder hangs it under a top-level node in front of the tree's root."""
    a, tri0 = scene_for(rt, golden_scenes, key)
    sc = build_scene(rt, a, tri0, kind)
    new = smooth(tri0, a["emissive"], None)
    st = sc.rebuild_bvh(new)
    assert st["gpu_launches"] > 4 and st["kernel_ms"] > 0.0 and st["total_ms"] > 0.0, st
    assert st["h2d_bytes"] >= new.nbytes and st["d2h_bytes"] > 0, st
    info = assert_is_device_build(rt, sc, new, f"{key}/{kind}")
    assert info["has_diag_slabs"] == 0
    if key == "c3small":
        assert sc.bvh_arrays()["wide"][0]["imask"] == 1              # record 0 is a top-level node: its one inner child is the tree
    # the oracle itself: two device builds of the same vertices are identical
    b1, i1 = builder_arrays(rt, new)
    b2, i2 = builder_arrays(rt, new)
    assert_arrays_equal(b1, b2, f"{key}: two device builds")
    assert all(i1[k] == i2[k] for k in INFO_KEYS) and i1["sah_cost"] == i2["sah_cost"]


def test_rebuild_of_three_triangles_uses_the_host_builder(rt, golden_scenes, golden_cameras):
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"][:3], np.float32)
    a = dict(tri9=tri0, mat_idx=a["mat_idx"][:3], mats10=a["mats10"], emissive=np.zeros(0, np.int32))
    sc = build_scene(rt, a, tri0)
    new = rigid(tri0, a["emissive"], None)
    sc.rebuild_bvh(new)
    info = assert_is_device_build(rt, sc, new, "three triangles")
    assert info["has_diag_slabs"] == 1                              # b200rt_bvh_build_device hands <= 3 triangles to the host builder
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, build_scene(rt, a, new), cam, new), "three triangles")


def test_rebuild_deep_chain(rt):
    """test_deep_chain's nested triangles (8-ary depth 14 from the host builder)."""
    n = 2000
    s = 1.005 ** np.arange(n)
    tri = np.zeros((n, 9))
    tri[:, 0] = 3 * s; tri[:, 1] = -s; tri[:, 2] = -s
    tri[:, 3] = 3 * s; tri[:, 4] = -s; tri[:, 5] = 2 * s
    tri[:, 6] = 3 * s; tri[:, 7] = 2 * s; tri[:, 8] = -s
    tri = tri.astype(np.float32)
    mats = np.array([[1, 0, 1, 1, 0, 0, 0, 1, 0, 1], [0, 0, 0, 1, .9, .8, .7, 1, 1.0, 0.3]], np.float32)
    a = dict(tri9=tri, mat_idx=np.ones(n, np.int32), mats10=mats, emissive=np.zeros(0, np.int32))
    sc = build_scene(rt, a, tri)
    v = tri.reshape(-1, 3).astype(np.float64)
    v[:, 1] += 0.3 * np.sin(v[:, 0] * 0.01) * np.sqrt(np.abs(v[:, 0]))
    new = v.reshape(-1, 9).astype(np.float32)
    sc.rebuild_bvh(new)
    info = assert_is_device_build(rt, sc, new, "deep chain")
    builder = "host SAH" if info["has_diag_slabs"] else "device"
    print(f"deep chain: served by the {builder} builder, 8-ary depth {info['wide_max_depth']}, binary depth {info['max_depth']}")
    cam = rt.Camera.from_array17(np.array([0, 0, 1, -1.0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 2.41421342], np.float32))
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, build_scene(rt, a, new), cam, new), "deep chain")


# ---- 2: outputs against fresh scenes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", ["cornell", "mis", "area"])
@pytest.mark.parametrize("deform", list(DEFORMATIONS))
def test_rebuild_equals_fresh_scene(rt, golden_scenes, golden_cameras, key, deform):
    """The fresh scene is host-built (diagonal slabs and all); the rebuilt one is device-built, and B200RT_FLAG_DIAG_SLABS traverses
    its axis slabs: every output still agrees."""
    a = scene_arrays(golden_scenes, key)
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    new = DEFORMATIONS[deform](tri0, a["emissive"], np.random.default_rng(3))
    sc.rebuild_bvh(new)
    fresh = build_scene(rt, a, new)
    cam = camera_for(rt, golden_cameras, key, new, tri0)
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, fresh, cam, new), f"{key}/{deform}")


def test_c2_half_turn_primary_maps(rt):
    """C2 (1 M triangles) rotated half a turn about y: the rebuilt scene's primary maps are a fresh scene's, and no tree-sized array
    crossed PCIe."""
    from sycl_ray_tracing_b200 import scenes
    c2 = scenes.c2_scene()
    sc = rt.Scene(c2["tri9"], c2["mat_idx"], c2["mats10"], c2["emissive"])
    v = c2["tri9"].reshape(-1, 3).astype(np.float64)
    new = np.stack([-v[:, 0], v[:, 1], -v[:, 2]], 1).reshape(-1, 9).astype(np.float32)
    st = sc.rebuild_bvh(new)
    info = sc.bvh_info()
    tree_bytes = 80 * info["n_wide_nodes"] + 64 * info["n_inner_nodes"] + 48 * info["n_triangles"]
    assert st["h2d_bytes"] - new.nbytes < 0.01 * tree_bytes and st["d2h_bytes"] < 0.01 * tree_bytes, (st, tree_bytes)
    fresh = rt.Scene(new, c2["mat_idx"], c2["mats10"], c2["emissive"])
    for flags in (0, rt.FLAG_BVH8, rt.FLAG_DIAG_SLABS):
        p, t, _ = sc.trace_primary(c2["camera"], 1920, 1080, flags=flags)
        pf, tf, _ = fresh.trace_primary(c2["camera"], 1920, 1080, flags=flags)
        assert np.array_equal(p, pf) and np.array_equal(t.view(np.uint32), tf.view(np.uint32)), flags
        assert (p >= 0).sum() > 400_000
    print(f"C2 half turn rebuild: {st['kernel_ms']:.2f} ms kernel, {st['total_ms']:.1f} ms total, {st['gpu_launches']} launches, "
          f"h2d {st['h2d_bytes']} B (vertices {new.nbytes}), d2h {st['d2h_bytes']} B, tree {tree_bytes} B")


# ---- 3: refits of a rebuilt tree ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("start", ["host", "leaf8"])
def test_refit_after_rebuild(rt, golden_scenes, start):
    """Rebuild to B, then refit to C: byte for byte a scene created with BVH(B, on_device=True) and refitted to C. From the leaf8
    tree (no 8-ary layout) the 8-ary node count grows from 0 across the rebuild, and the refit state must follow it."""
    a = scene_arrays(golden_scenes, "mis")
    tri_a = np.ascontiguousarray(a["tri9"], np.float32)
    tri_b = smooth(tri_a, a["emissive"], None)
    tri_c = rigid(tri_b, a["emissive"], None)
    sc = build_scene(rt, a, tri_a, start)
    sc.update_triangles(tri_a)                                   # refit state made for the old tree
    before = sc.bvh_info()
    sc.rebuild_bvh(tri_b)
    after = sc.bvh_info()
    if start == "leaf8":
        assert before["n_wide_nodes"] == 0 and after["n_wide_nodes"] > 0
    sc.update_triangles(tri_c)
    want = rt.Scene(tri_b, a["mat_idx"], a["mats10"], a["emissive"], skysphere=sc.env, bvh=rt.BVH(tri_b, on_device=True))
    want.update_triangles(tri_c)
    assert_arrays_equal(sc.bvh_arrays(), want.bvh_arrays(), f"{start}: rebuild B, refit C")
    assert sc.bvh_info()["sah_cost"] == want.bvh_info()["sah_cost"]


def test_rebuild_there_and_back(rt, golden_scenes):
    a = scene_arrays(golden_scenes, "area")
    tri_a = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri_a)
    sc.rebuild_bvh(tri_a)
    first = sc.bvh_arrays()
    sc.rebuild_bvh(rigid(tri_a, a["emissive"], None))
    sc.rebuild_bvh(tri_a)
    assert_arrays_equal(sc.bvh_arrays(), first, "A -> B -> A")
    assert_is_device_build(rt, sc, tri_a, "A -> B -> A")


# ---- 4: multi-device -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_ranks", [2, 3])
def test_multi_device_rebuild(rt, golden_scenes, golden_cameras, n_ranks):
    import torch
    have = torch.cuda.device_count()
    devs = [i % have for i in range(n_ranks)]
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    multi = build_scene(rt, a, tri0, devices=devs)
    new = rigid(tri0, a["emissive"], None)
    multi.rebuild_bvh(new)
    want, _ = builder_arrays(rt, new)
    for r in range(n_ranks):
        assert_arrays_equal(multi.bvh_arrays(r), want, f"replica {r}")
    single = build_scene(rt, a, tri0)
    single.rebuild_bvh(new)
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    fb0 = (np.random.default_rng(9).random((H, W, 4)) * 0.3).astype(np.float32)
    got, exp = fb0.copy(), fb0.copy()
    _, sg = multi.render(cam, W, H, SPP, BOUNCES, framebuffer=got)
    _, sw = single.render(cam, W, H, SPP, BOUNCES, framebuffer=exp)
    assert np.array_equal(got.view(np.uint32), exp.view(np.uint32)) and sg["rays"] == sw["rays"]
    # the device variant on a multi-device scene, then a refit of every replica's new tree
    t = torch.from_numpy(smooth(tri0, a["emissive"], None)).cuda(devs[0])
    multi.rebuild_bvh_device(t.data_ptr(), len(tri0))
    multi.update_triangles(new)
    host = build_scene(rt, a, tri0)
    host.rebuild_bvh(t.cpu().numpy())
    host.update_triangles(new)
    for r in range(n_ranks):
        assert_arrays_equal(multi.bvh_arrays(r), host.bvh_arrays(0), f"device variant and refit, replica {r}")


# ---- 5: ordering and survival --------------------------------------------------------------------------------------------------------------
def test_device_variant_orders_after_the_callers_stream(rt, golden_scenes, golden_cameras):
    import torch
    a = scene_arrays(golden_scenes, "mis")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    new = smooth(tri0, a["emissive"], None)
    sc = build_scene(rt, a, tri0)
    torch.cuda.set_device(0)
    base = torch.from_numpy(new).cuda()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(20_000_000)                   # the stream is busy; the copy below lands well after the call is issued
        dev = torch.empty_like(base)
        dev.copy_(base)
        st = sc.rebuild_bvh_device(dev.data_ptr(), len(new), side.cuda_stream)
    assert torch.cuda.current_device() == 0
    assert st["kernel_ms"] > 0.0, st
    assert_is_device_build(rt, sc, new, "device variant")
    cam = rt.Camera.from_array17(golden_cameras["mis"])
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, build_scene(rt, a, new), cam, new), "device variant")


def test_accumulator_survives_a_rebuild_and_materials_still_set(rt, golden_scenes, golden_cameras):
    """4 samples on the host-built tree, a rebuild with the same vertices (now the device-built tree), 12 more: the render of 16."""
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    acc = rt.Accumulator(sc, cam, W, H, 16, BOUNCES)
    acc.add(4)
    sc.rebuild_bvh(tri0)
    assert sc.bvh_info()["has_diag_slabs"] == 0
    acc.add(12)
    want, _ = build_scene(rt, a, tri0).render(cam, W, H, 16, BOUNCES)
    assert np.array_equal(acc.resolve().view(np.uint32), want.view(np.uint32))
    del acc
    gc.collect()
    mats = a["mats10"].copy()
    mats[:, 4:7] *= 0.5
    sc.set_materials(mats)
    fresh = build_scene(rt, a, tri0)
    fresh.set_materials(mats)
    assert np.array_equal(sc.render(cam, W, H, SPP, BOUNCES)[0].view(np.uint32), fresh.render(cam, W, H, SPP, BOUNCES)[0].view(np.uint32))


# ---- 6: refusals and leaks -------------------------------------------------------------------------------------------------------------------
def test_refusals_change_nothing(rt, golden_scenes, golden_cameras):
    import torch
    L = rt.load_library()
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    sc.update_triangles(rigid(tri0, a["emissive"], None))         # refit state in place too
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    before, nbytes, info = sc.bvh_arrays(), sc.device_bytes(), sc.bvh_info()
    img = sc.render(cam, W, H, SPP, BOUNCES)[0]
    n = len(tri0)
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    assert L.b200rt_scene_rebuild_bvh(sc._h, fp(tri0), n - 1, None) == 1
    assert L.b200rt_scene_rebuild_bvh(sc._h, fp(tri0), n + 1, None) == 1
    assert L.b200rt_scene_rebuild_bvh(sc._h, fp(tri0), 1 << 27, None) == 1
    assert L.b200rt_scene_rebuild_bvh(sc._h, None, n, None) == 1
    assert L.b200rt_scene_rebuild_bvh(None, fp(tri0), n, None) == 1
    assert L.b200rt_scene_rebuild_bvh_device(sc._h, None, n, None, None) == 1
    assert L.b200rt_scene_rebuild_bvh_device(sc._h, C.c_void_p(tri0.ctypes.data), n, None, None) == 1     # host memory
    assert b"device memory" in L.b200rt_last_error()
    for bad in (np.nan, np.inf, -np.inf):
        t = tri0.copy()
        t[-1, 7] = bad
        assert L.b200rt_scene_rebuild_bvh(sc._h, fp(t), n, None) == 1
        assert b"NaN or infinite" in L.b200rt_last_error()
        d = torch.from_numpy(t).cuda()
        assert L.b200rt_scene_rebuild_bvh_device(sc._h, C.c_void_p(d.data_ptr()), n, None, None) == 1
    with pytest.raises(ValueError):
        sc.rebuild_bvh(tri0[:-1])
    assert_arrays_equal(sc.bvh_arrays(), before, "after refusals")
    assert sc.device_bytes() == nbytes and sc.bvh_info() == info
    assert np.array_equal(sc.render(cam, W, H, SPP, BOUNCES)[0].view(np.uint32), img.view(np.uint32))


def test_alternating_rebuilds_do_not_leak(rt):
    import torch
    from sycl_ray_tracing_b200 import scenes
    c2 = scenes.c2_scene(nu=256, nv=128)
    tri_a = np.ascontiguousarray(c2["tri9"], np.float32)
    tri_b = twist(tri_a, 0.5)
    sc = rt.Scene(tri_a, c2["mat_idx"], c2["mats10"], c2["emissive"])
    torch.cuda.synchronize()
    sc.rebuild_bvh(tri_b)
    sc.update_triangles(tri_b)
    torch.cuda.synchronize()
    first = (sc.device_bytes(), torch.cuda.mem_get_info()[0])
    for i in range(20):
        sc.rebuild_bvh(tri_a if i % 2 == 0 else tri_b)
        sc.update_triangles(tri_a if i % 2 == 0 else tri_b)
    torch.cuda.synchronize()
    last = (sc.device_bytes(), torch.cuda.mem_get_info()[0])
    assert last[0] == first[0], (first, last)
    assert abs(last[1] - first[1]) <= 4 << 20, (first, last)          # one tree here is ~10 MB
