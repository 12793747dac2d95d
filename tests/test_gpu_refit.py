"""-m gpu: geometry updates of a resident scene (b200rt_scene_update_triangles[_device]) and the BVH refit behind them.

Closest hits do not depend on the tree's shape (exact Moller-Trumbore, ties to the lowest original index), so a scene refitted to new
vertices has an exact oracle: a scene freshly created from the same vertices. Every output is compared with it bit for bit, ray counts
included. The refitted arrays are also checked on their own in float64 numpy: every decoded 8-ary child box, axis box and diagonal
slab contains every vertex beneath it, and the triangle stream is {a, b - a, c - a} of the new vertices."""
import ctypes as C
import gc

import numpy as np
import pytest

from conftest import load_golden, scene_arrays

pytestmark = pytest.mark.gpu

W, H, SPP, BOUNCES = 64, 48, 4, 4
CAM_OF = {"cornell": "cornell", "mis": "mis", "area": "cornell"}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def env():
    return load_golden("render_cornell_env.npz")["env"]


def build_scene(rt, a, tri, bvh_kind="host", devices=None):
    bvh = None
    if bvh_kind == "device":
        bvh = rt.BVH(tri, on_device=True)
    elif bvh_kind == "leaf8":
        bvh = rt.BVH(tri, max_leaf_size=8)
    return rt.Scene(tri, a["mat_idx"], a["mats10"], a["emissive"], skysphere=env(), bvh=bvh, devices=devices)


# ---- deformations: (n, 9) float32 -> (n, 9) float32, all computed in float64 and rounded once ---------------------------------
def _bbox(tri):
    v = tri.reshape(-1, 3).astype(np.float64)
    return v.min(0), v.max(0)


def rigid(tri, emissive, rng):
    lo, hi = _bbox(tri)
    c = 0.5 * (lo + hi)
    ax = np.array([0.3, 1.0, 0.2]); ax /= np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    a = 0.4
    R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    v = (tri.reshape(-1, 3).astype(np.float64) - c) @ R.T + c + 0.05 * (hi - lo)
    return v.reshape(-1, 9).astype(np.float32)


def smooth(tri, emissive, rng):
    lo, hi = _bbox(tri)
    s = float((hi - lo).max())
    v = tri.reshape(-1, 3).astype(np.float64)
    u = (v - lo) / s
    d = 0.04 * s * np.stack([np.sin(5 * u[:, 1] + 1), np.sin(4 * u[:, 2] + 2 * u[:, 0]), np.cos(6 * u[:, 0] - u[:, 1])], 1)
    return (v + d).reshape(-1, 9).astype(np.float32)


def emissive_only(tri, emissive, rng):
    out = tri.copy()
    if len(emissive):
        lo, hi = _bbox(tri)
        v = tri[emissive].reshape(-1, 3).astype(np.float64)
        c = v.mean(0)
        out[emissive] = ((v - c) * 0.7 + c + np.array([0.1, -0.15, 0.05]) * (hi - lo)).reshape(-1, 9).astype(np.float32)
    return out


def far_and_large(tri, emissive, rng):
    return (tri.astype(np.float64) * 1000.0 + np.tile([1.2e4, -0.8e4, 1.0e4], 3)).astype(np.float32)


def collapse(tri, emissive, rng):
    out = tri.copy()
    idx = np.arange(0, len(tri), 3)
    out[idx, 3:6] = out[idx, 0:3]
    out[idx, 6:9] = out[idx, 0:3]
    return out


def permute(tri, emissive, rng):
    return np.ascontiguousarray(tri[rng.permutation(len(tri))])


DEFORMATIONS = {"rigid": rigid, "smooth": smooth, "emissive_only": emissive_only, "far_and_large": far_and_large,
                "collapse": collapse, "permute": permute}


def camera_for(rt, golden_cameras, key, tri, original):
    """The scene's golden camera; for a scaled/translated scene the same view of the moved geometry."""
    c = golden_cameras[CAM_OF[key]].copy()
    lo0, hi0 = _bbox(original)
    lo1, hi1 = _bbox(tri)
    k = float((hi1 - lo1).max() / max((hi0 - lo0).max(), 1e-30))
    if k > 10.0:                                    # the far_and_large deformation: scale about the origin, then translate
        m = c[:16].reshape(4, 4).astype(np.float64)
        m[:3, 3] = m[:3, 3] * 1000.0 + np.array([1.2e4, -0.8e4, 1.0e4])
        c[:16] = m.reshape(16).astype(np.float32)
    return rt.Camera.from_array17(c)


def random_rays(tri, n=3000, seed=11):
    rng = np.random.default_rng(seed)
    lo, hi = _bbox(tri)
    c, ext = 0.5 * (lo + hi), (hi - lo).max()
    o = c + (rng.random((n, 3)) - 0.5) * 1.6 * ext
    tgt = c + (rng.random((n, 3)) - 0.5) * 0.8 * ext
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d], 1).astype(np.float32)


def outputs(rt, sc, cam, tri, wide=True):
    """Every entry point the refit must leave exact: integrators on a non-black framebuffer, RGBA8, a region, feature buffers,
    primary maps under every layout flag, ray batches (closest hits, any-hit flags)."""
    out = {}
    fb0 = (np.random.default_rng(5).random((H, W, 4)) * 0.3).astype(np.float32)
    integrators = [("wavefront", rt.INTEGRATOR_WAVEFRONT), ("megakernel", rt.INTEGRATOR_MEGAKERNEL)]
    if wide:
        integrators.append(("persistent", rt.INTEGRATOR_PERSISTENT))
    for name, integ in integrators:
        fb = fb0.copy()
        _, st = sc.render(cam, W, H, SPP, BOUNCES, framebuffer=fb, integrator=integ)
        out[f"render_{name}"] = fb
        out[f"rays_{name}"] = st["rays"]
    out["rgba8"] = sc.render_rgba8(cam, W, H, SPP, BOUNCES, framebuffer=fb0)[0]
    out["region"] = sc.render_region(cam, W, H, SPP, BOUNCES, 10, 7, 37, 29)[0]
    alb, nrm, _ = sc.render_aovs(cam, W, H, 2)
    out["albedo"], out["normal"] = alb, nrm
    for fname, flags in (("default", 0), ("bvh8", rt.FLAG_BVH8), ("bvh2", rt.FLAG_BVH2), ("diag", rt.FLAG_DIAG_SLABS)):
        prim, t, _ = sc.trace_primary(cam, W, H, flags=flags)
        out[f"primary_{fname}"] = (prim, t)
    rays = random_rays(tri)
    out["closest"] = sc.trace_rays(rays)
    # any hit: the flag only; its t is whichever hit the traversal meets first, which depends on the tree's shape
    out["any"] = (sc.trace_rays(rays, any_hit=True)[0],)
    return out


def assert_same_outputs(got, want, what):
    assert got.keys() == want.keys()
    for k in want:
        g, w = got[k], want[k]
        if isinstance(w, tuple):
            for i, (x, y) in enumerate(zip(g, w)):
                assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), f"{what}: {k}[{i}] differs"
        elif isinstance(w, np.ndarray):
            assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), f"{what}: {k} differs ({(g != w).sum()} values)"
        else:
            assert g == w, f"{what}: {k} {g} != {w}"


# ---- structural checks in float64 -------------------------------------------------------------------------------------------------
def wide_order(wide):
    order, i = [0], 0
    while i < len(order):
        w = wide[order[i]]
        order += [int(w["child_base"]) + k for k in range(bin(int(w["imask"])).count("1"))]
        i += 1
    assert sorted(order) == list(range(len(wide))), "the 8-ary nodes are not one tree rooted at node 0"
    return order


def axis_order(axis):
    refs = axis[:, 12:14].view(np.int32)
    order, i = [0], 0
    while i < len(order):
        order += [int(r) for r in refs[order[i]] if r >= 0]
        i += 1
    assert sorted(order) == list(range(len(axis))), "the binary records are not one tree rooted at record 0"
    return order


def grid(q):
    q = q.astype(np.int64)
    return np.where(q < 128, 128 + q, 2 * q).astype(np.float64)


def diag_d(v):
    x, y, z = v[:, 0], v[:, 1], v[:, 2]
    return np.stack([x + y + z, -x + y + z, -x - y + z, x - y + z], 1)


def check_structure(arrs, tri):
    """Every decoded child box / slab contains every vertex of every triangle beneath it; the stream is {a, b - a, c - a}."""
    V = tri.astype(np.float64).reshape(-1, 3, 3)
    tris = arrs["tris"]
    prim = tris[:, 3].view(np.int32)
    assert sorted(prim.tolist()) == list(range(len(tri)))
    a = tri[prim, 0:3]
    assert same_bits(tris[:, 0:3], a)
    assert same_bits(tris[:, 4:7], (tri[prim, 3:6] - a).astype(np.float32))
    assert same_bits(tris[:, 8:11], (tri[prim, 6:9] - a).astype(np.float32))
    assert not bits(tris[:, [7, 11]]).any()
    wide = arrs["wide"]
    if len(wide):
        lo = np.full((len(wide), 3), np.inf); hi = np.full((len(wide), 3), -np.inf)
        for ni in reversed(wide_order(wide)):
            w = wide[ni]
            rank, at = 0, int(w["tri_base"])
            cell = 2.0 ** (w["e"].astype(np.int64) - 127)
            p = w["p"].astype(np.float64)
            for s in range(8):
                m = (int(w["valid24"]) >> (3 * s)) & 7
                if (int(w["imask"]) >> s) & 1:
                    c = int(w["child_base"]) + rank; rank += 1
                    clo, chi = lo[c], hi[c]
                elif m:
                    cnt = bin(m).count("1")
                    v = V[prim[at:at + cnt]].reshape(-1, 3)
                    clo, chi = v.min(0), v.max(0)
                    at += cnt
                else:
                    continue
                dlo = p + cell * grid(np.array([w["lox"][s], w["loy"][s], w["loz"][s]]))
                dhi = p + cell * grid(np.array([w["hix"][s], w["hiy"][s], w["hiz"][s]]))
                assert (clo >= dlo).all() and (chi <= dhi).all(), f"8-ary node {ni} slot {s} does not contain its vertices"
                lo[ni] = np.minimum(lo[ni], clo); hi[ni] = np.maximum(hi[ni], chi)
    axis, diag = arrs["axis"], arrs["diag"]
    refs = axis[:, 12:14].view(np.int32)
    lo = np.full((len(axis), 3), np.inf); hi = np.full((len(axis), 3), -np.inf)
    dn = np.full((len(axis), 4), np.inf); df = np.full((len(axis), 4), -np.inf)
    for ri in reversed(axis_order(axis)):
        for side in range(2):
            r = int(refs[ri, side])
            if r >= 0:
                clo, chi, cdn, cdf = lo[r], hi[r], dn[r], df[r]
            else:
                first, cnt = (~r) >> 4, (~r) & 15
                if cnt == 0:
                    continue
                v = V[prim[first:first + cnt]].reshape(-1, 3)
                clo, chi, d = v.min(0), v.max(0), diag_d(v)
                cdn, cdf = d.min(0), d.max(0)
            blo, bhi = axis[ri, 6 * side:6 * side + 3].astype(np.float64), axis[ri, 6 * side + 3:6 * side + 6].astype(np.float64)
            assert (clo >= blo).all() and (chi <= bhi).all(), f"axis record {ri} side {side} does not contain its vertices"
            if len(diag):
                near, far = diag[ri, 8 * side:8 * side + 4].astype(np.float64), diag[ri, 8 * side + 4:8 * side + 8].astype(np.float64)
                assert (cdn >= near).all() and (cdf <= far).all(), f"diag record {ri} side {side} does not contain its vertices"
            lo[ri] = np.minimum(lo[ri], clo); hi[ri] = np.maximum(hi[ri], chi)
            dn[ri] = np.minimum(dn[ri], cdn); df[ri] = np.maximum(df[ri], cdf)


def sah_numpy(axis):
    """sah_cost_of (csrc/bvh_build.cpp) restated: 1 + sum over records of child area / root area, leaves times their count."""
    def half_area(lo, hi):
        d = hi.astype(np.float64) - lo.astype(np.float64)
        a = d[:, 0] * d[:, 1] + d[:, 1] * d[:, 2] + d[:, 2] * d[:, 0]
        return np.where((d < 0).any(1), 0.0, a)
    r = axis[0]
    root = max(1e-30, float(half_area(np.minimum(r[0:3], r[6:9])[None], np.maximum(r[3:6], r[9:12])[None])[0]))
    refs = axis[:, 12:14].view(np.int32); cnt = axis[:, 14:16].view(np.int32)
    s = 1.0
    for side in range(2):
        a = half_area(axis[:, 6 * side:6 * side + 3], axis[:, 6 * side + 3:6 * side + 6]) / root
        s += float(np.where(refs[:, side] >= 0, a, a * cnt[:, side]).sum())
    return s


def assert_arrays_equal(got, want, what, skip_wide=(), skip_axis=()):
    for k in ("tris", "diag"):
        assert np.array_equal(got[k].view(np.uint8), want[k].view(np.uint8)), f"{what}: {k} differs"
    gw, ww = got["wide"].copy(), want["wide"].copy()
    ga, wa = got["axis"].copy(), want["axis"].copy()
    for i in skip_wide:
        gw[i] = ww[i]
    for i in skip_axis:
        ga[i] = wa[i]
    assert np.array_equal(gw.view(np.uint8), ww.view(np.uint8)), f"{what}: 8-ary nodes differ at {np.nonzero((gw.view(np.uint8).reshape(len(gw), -1) != ww.view(np.uint8).reshape(len(ww), -1)).any(1))[0][:8]}"
    assert np.array_equal(ga.view(np.uint8), wa.view(np.uint8)), f"{what}: axis records differ"


# ---- 1, 2: fresh-scene identity and structure after every deformation ---------------------------------------------------------------
SCENES = [("cornell", "host"), ("mis", "host"), ("area", "host"), ("mis", "device")]


@pytest.mark.parametrize("key,kind", SCENES)
@pytest.mark.parametrize("deform", list(DEFORMATIONS))
def test_refit_equals_fresh_scene(rt, golden_scenes, golden_cameras, key, kind, deform):
    a = scene_arrays(golden_scenes, key)
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0, kind)
    new = DEFORMATIONS[deform](tri0, a["emissive"], np.random.default_rng(3))
    st = sc.update_triangles(new)
    assert st["gpu_launches"] >= 4 and st["kernel_ms"] > 0.0 and st["h2d_bytes"] == new.nbytes, st
    fresh = build_scene(rt, a, new, kind)
    cam = camera_for(rt, golden_cameras, key, new, tri0)
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, fresh, cam, new), f"{key}/{kind}/{deform}")
    check_structure(sc.bvh_arrays(), new)
    info = sc.bvh_info()
    assert abs(info["sah_cost"] - sah_numpy(sc.bvh_arrays()["axis"])) <= 1e-9 * info["sah_cost"]


# ---- 3: identity and history ---------------------------------------------------------------------------------------------------------
def c3_small():
    from sycl_ray_tracing_b200 import scenes
    c3 = scenes.c3_scene(nu=64, nv=32, sky_w=64, sky_h=32)
    return dict(tri9=c3["tri9"], mat_idx=c3["mat_idx"], mats10=c3["mats10"], emissive=c3["emissive"])


IDENTITY = [("cornell", "host"), ("mis", "host"), ("area", "host"), ("c2small", "device"), ("c3small", "device"), ("mis", "leaf8")]


def identity_scene(rt, golden_scenes, key, kind):
    if key == "c3small":
        a = c3_small()
    elif key == "c2small":
        from sycl_ray_tracing_b200 import scenes
        c2 = scenes.c2_scene(nu=64, nv=32)
        a = dict(tri9=c2["tri9"], mat_idx=c2["mat_idx"], mats10=c2["mats10"], emissive=c2["emissive"])
    else:
        a = scene_arrays(golden_scenes, key)
    return a, np.ascontiguousarray(a["tri9"], np.float32)


@pytest.mark.parametrize("key,kind", IDENTITY)
def test_update_with_creation_vertices_and_history(rt, golden_scenes, key, kind):
    """An update with the creation vertices changes no byte, except the top-level nodes the device builder hangs outsized triangles
    under (C3-small's ground quad: 8-ary node 0 and binary record 0), whose boxes become padded-once exact boxes. A -> B -> A gives
    the arrays of A again, and the SAH cost stays the build's."""
    a, tri0 = identity_scene(rt, golden_scenes, key, kind)
    sc = build_scene(rt, a, tri0, kind)
    built = sc.bvh_arrays()
    sah_built = sah_numpy(built["axis"])
    sc.update_triangles(tri0)
    after = sc.bvh_arrays()
    top = (0,) if key == "c3small" else ()
    assert_arrays_equal(after, built, f"{key}/{kind} identity", skip_wide=top, skip_axis=top)
    if top:
        assert not np.array_equal(after["axis"][0].view(np.uint8), built["axis"][0].view(np.uint8))
    check_structure(after, tri0)
    assert abs(sc.bvh_info()["sah_cost"] - sah_built) <= 1e-9 * sah_built
    if kind == "device" and not top:
        assert abs(sc.bvh_info()["sah_cost"] - rt.BVH(tri0, on_device=True).info()["sah_cost"]) <= 1e-9 * sah_built
    sc.update_triangles(smooth(tri0, a["emissive"], None))
    sc.update_triangles(tri0)
    assert_arrays_equal(sc.bvh_arrays(), after, f"{key}/{kind} A -> B -> A")
    if kind == "leaf8":
        assert sc.bvh_info()["n_wide_nodes"] == 0 and len(after["wide"]) == 0


# ---- 4: large and deep trees ------------------------------------------------------------------------------------------------------------
def twist(tri, turns=0.6):
    """Rotation about y by an angle that grows with height (the refit benchmark's animation)."""
    v = tri.reshape(-1, 3).astype(np.float64)
    lo, hi = v[:, 1].min(), v[:, 1].max()
    ang = 2 * np.pi * turns * (v[:, 1] - lo) / max(hi - lo, 1e-30)
    c, s = np.cos(ang), np.sin(ang)
    out = np.stack([c * v[:, 0] + s * v[:, 2], v[:, 1], -s * v[:, 0] + c * v[:, 2]], 1)
    return out.reshape(-1, 9).astype(np.float32)


def test_c2_twisted_primary_maps(rt):
    from sycl_ray_tracing_b200 import scenes
    c2 = scenes.c2_scene()
    sc = rt.Scene(c2["tri9"], c2["mat_idx"], c2["mats10"], c2["emissive"])
    sah0 = sc.bvh_info()["sah_cost"]
    new = twist(c2["tri9"])
    st = sc.update_triangles(new)
    fresh = rt.Scene(new, c2["mat_idx"], c2["mats10"], c2["emissive"])
    for flags in (0, rt.FLAG_BVH8, rt.FLAG_DIAG_SLABS):
        p, t, _ = sc.trace_primary(c2["camera"], 1920, 1080, flags=flags)
        pf, tf, _ = fresh.trace_primary(c2["camera"], 1920, 1080, flags=flags)
        assert np.array_equal(p, pf) and same_bits(t, tf), flags
        assert (p >= 0).sum() > 400_000
    print(f"C2 twist refit: {st['kernel_ms']:.3f} ms kernel, {st['total_ms']:.1f} ms total, sah {sah0:.2f} -> {sc.bvh_info()['sah_cost']:.2f}")


def test_deep_chain(rt):
    """The geometric chain of nested triangles (8-ary depth 14: deeper than the shared-memory stack of the cooperative trace)."""
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
    assert sc.bvh_info()["wide_max_depth"] > 10
    v = tri.reshape(-1, 3).astype(np.float64)
    v[:, 1] += 0.3 * np.sin(v[:, 0] * 0.01) * np.sqrt(np.abs(v[:, 0]))
    new = v.reshape(-1, 9).astype(np.float32)
    sc.update_triangles(new)
    fresh = build_scene(rt, a, new)
    cam = rt.Camera.from_array17(np.array([0, 0, 1, -1.0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 2.41421342], np.float32))
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, fresh, cam, new), "deep chain")
    check_structure(sc.bvh_arrays(), new)


def test_leaf8_tree_without_wide_layout(rt, golden_scenes, golden_cameras):
    a = scene_arrays(golden_scenes, "mis")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0, "leaf8")
    assert sc.bvh_info()["n_wide_nodes"] == 0
    new = smooth(tri0, a["emissive"], None)
    sc.update_triangles(new)
    fresh = build_scene(rt, a, new, "leaf8")
    cam = camera_for(rt, golden_cameras, "mis", new, tri0)
    assert_same_outputs(outputs(rt, sc, cam, new, wide=False), outputs(rt, fresh, cam, new, wide=False), "leaf8")
    check_structure(sc.bvh_arrays(), new)


# ---- 5: multi-device ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_ranks", [2, 3])
def test_multi_device_update(rt, golden_scenes, golden_cameras, n_ranks):
    import torch
    have = torch.cuda.device_count()
    devs = [i % have for i in range(n_ranks)]
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    multi = build_scene(rt, a, tri0, devices=devs)
    new = rigid(tri0, a["emissive"], None)
    st = multi.update_triangles(new)
    assert st["h2d_bytes"] == n_ranks * new.nbytes, st
    fresh = build_scene(rt, a, new)
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    fb0 = (np.random.default_rng(9).random((H, W, 4)) * 0.3).astype(np.float32)
    got, want = fb0.copy(), fb0.copy()
    _, sg = multi.render(cam, W, H, SPP, BOUNCES, framebuffer=got)
    _, sw = fresh.render(cam, W, H, SPP, BOUNCES, framebuffer=want)
    assert same_bits(got, want) and sg["rays"] == sw["rays"]
    r0 = multi.bvh_arrays(0)
    check_structure(r0, new)
    for r in range(1, n_ranks):
        assert_arrays_equal(multi.bvh_arrays(r), r0, f"replica {r}")
    # the device variant on a multi-device scene: the vertices go device to device
    t = torch.from_numpy(smooth(tri0, a["emissive"], None)).cuda(devs[0])
    multi.update_triangles_device(t.data_ptr(), len(tri0))
    torch.cuda.synchronize()
    host = build_scene(rt, a, tri0, devices=devs)
    host.update_triangles(t.cpu().numpy())
    for r in range(n_ranks):
        assert_arrays_equal(multi.bvh_arrays(r), host.bvh_arrays(0), f"device variant, replica {r}")


# ---- 6: the device variant -----------------------------------------------------------------------------------------------------------------
def test_device_variant_orders_after_the_callers_stream(rt, golden_scenes, golden_cameras):
    import torch
    a = scene_arrays(golden_scenes, "mis")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    new = smooth(tri0, a["emissive"], None)
    want = build_scene(rt, a, tri0)
    want.update_triangles(new)
    sc = build_scene(rt, a, tri0)
    torch.cuda.set_device(0)
    base = torch.from_numpy(new).cuda()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(20_000_000)                   # the stream is busy; the copy below lands well after the call is issued
        dev = torch.empty_like(base)
        dev.copy_(base)
        st = sc.update_triangles_device(dev.data_ptr(), len(new), side.cuda_stream)
    assert torch.cuda.current_device() == 0
    assert st["h2d_bytes"] == 0 and st["kernel_ms"] > 0.0
    assert_arrays_equal(sc.bvh_arrays(), want.bvh_arrays(), "device variant")
    cam = rt.Camera.from_array17(golden_cameras["mis"])
    assert_same_outputs(outputs(rt, sc, cam, new), outputs(rt, want, cam, new), "device variant")


# ---- 7: refusals change nothing ------------------------------------------------------------------------------------------------------------
def test_refusals_change_nothing(rt, golden_scenes, golden_cameras):
    import torch
    L = rt.load_library()
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    moved = rigid(tri0, a["emissive"], None)
    sc.update_triangles(moved)
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    before, img = sc.bvh_arrays(), sc.render(cam, W, H, SPP, BOUNCES)[0]
    n = len(tri0)
    fp = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    assert L.b200rt_scene_update_triangles(sc._h, fp(tri0), n - 1, None) == 1
    assert L.b200rt_scene_update_triangles(sc._h, fp(tri0), n + 1, None) == 1
    assert L.b200rt_scene_update_triangles(sc._h, None, n, None) == 1
    assert L.b200rt_scene_update_triangles(None, fp(tri0), n, None) == 1
    assert L.b200rt_scene_update_triangles_device(sc._h, None, n, None, None) == 1
    for bad in (np.nan, np.inf, -np.inf):
        t = tri0.copy()
        t[-1, 7] = bad
        assert L.b200rt_scene_update_triangles(sc._h, fp(t), n, None) == 1
        assert b"NaN or infinite" in L.b200rt_last_error()
        d = torch.from_numpy(t).cuda()
        assert L.b200rt_scene_update_triangles_device(sc._h, C.c_void_p(d.data_ptr()), n, None, None) == 1
    with pytest.raises(ValueError):
        sc.update_triangles(tri0[:-1])
    after = sc.bvh_arrays()
    assert_arrays_equal(after, before, "after refusals")
    assert same_bits(sc.render(cam, W, H, SPP, BOUNCES)[0], img)


# ---- 8: accumulators and materials ----------------------------------------------------------------------------------------------------------
def test_accumulator_survives_an_update_and_materials_still_set(rt, golden_scenes, golden_cameras):
    a = scene_arrays(golden_scenes, "cornell")
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    acc = rt.Accumulator(sc, cam, W, H, 8, BOUNCES)
    new = smooth(tri0, a["emissive"], None)
    sc.update_triangles(new)
    for k in (3, 5):
        acc.add(k)
    fresh = build_scene(rt, a, new)
    want, _ = fresh.render(cam, W, H, 8, BOUNCES)
    assert same_bits(acc.resolve(), want)
    del acc
    gc.collect()
    mats = a["mats10"].copy()
    mats[:, 4:7] *= 0.5
    sc.set_materials(mats)
    fresh.set_materials(mats)
    assert same_bits(sc.render(cam, W, H, SPP, BOUNCES)[0], fresh.render(cam, W, H, SPP, BOUNCES)[0])


# ---- 9: SAH --------------------------------------------------------------------------------------------------------------------------------
def test_sah_cost_follows_the_deformation(rt):
    a = c3_small()
    tri0 = np.ascontiguousarray(a["tri9"], np.float32)
    sc = build_scene(rt, a, tri0)
    sc.update_triangles(tri0)
    s0 = sc.bvh_info()["sah_cost"]
    assert abs(s0 - sah_numpy(sc.bvh_arrays()["axis"])) <= 1e-9 * s0
    got = []
    for turns in (0.25, 1.0):
        sc.update_triangles(np.concatenate([twist(tri0[:-2], turns), tri0[-2:]]))
        s = sc.bvh_info()["sah_cost"]
        assert abs(s - sah_numpy(sc.bvh_arrays()["axis"])) <= 1e-9 * s
        got.append(s)
    assert s0 < got[0] < got[1], (s0, got)
