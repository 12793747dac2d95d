"""-m gpu, round 2: the configurations and entry points the first round left untested under the driver — BASELINE config 4 at
its sweep extremes, config 5's scene (fixture, the full 20 M-triangle scene, the wrapping 1024-spp seed, stacks deeper than
the shared-memory part), config 3 against the 2048x1024 sky, config 1 at full size; the region / single-pixel entry, the RGBA8
output stage, page-locked buffers, env tables built on the device, multi-device scenes behind the C ABI."""
import os

import numpy as np
import pytest

from conftest import brute_force_closest, load_golden, scene_arrays

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def image_stats(gpu, ref):
    a, b = gpu[..., :3].astype(np.float64), ref[..., :3].astype(np.float64)
    finite = np.isfinite(a) & np.isfinite(b)
    d = np.where(finite, a - b, 0.0)
    px_bad = (np.abs(d) > 1.0e-3).any(axis=-1)
    return dict(rmse=float(np.sqrt((d ** 2).mean())), max=float(np.abs(d).max()), frac_close=float(1.0 - px_bad.mean()),
                nan_gpu=int((~np.isfinite(a)).sum()), nan_ref=int((~np.isfinite(b)).sum()),
                mean_gpu=float(np.where(finite, a, 0).mean()), mean_ref=float(np.where(finite, b, 0).mean()))


def assert_radiance_parity(img, ref, what=""):
    """Stated tolerance of every radiance comparison against the reference (tone-mapped framebuffer RGB): >= 99 % of pixels
    within 1e-3 on every channel, RMSE <= 5e-3, means within 0.5 %, identical NaN counts."""
    s = image_stats(img, ref)
    print(what, s)
    assert s["frac_close"] >= 0.99, (what, s)
    assert s["rmse"] <= 5.0e-3, (what, s)
    assert abs(s["mean_gpu"] - s["mean_ref"]) <= 0.005 * max(s["mean_ref"], 1e-6), (what, s)
    assert s["nan_gpu"] == s["nan_ref"], (what, s)


def scene_of(rt, d, **kw):
    return rt.Scene(d["tri9"], d["mat_idx"], d["mats10"], d["emissive"], skysphere=d.get("env"), **kw)


# ---- BASELINE config 4: roughness / metalness sweep extremes against the compiled reference -----------------------------------------
@pytest.mark.parametrize("tag", ["r005_m1", "r005_m0", "r100_m1", "r100_m0"])
def test_c4_sweep_extremes_match_reference(rt, tag):
    from sycl_ray_tracing_b200 import scenes
    g = load_golden(f"render_c4_{tag}.npz")
    c = scenes.c3_scene(roughness=float(g["roughness"]), metalness=float(g["metalness"]), nu=int(g["nu"]), nv=int(g["nv"]),
                        sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    sc = scene_of(rt, c)
    w, h, spp, b = int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"])
    img, st = sc.render(c["camera"], w, h, spp, b)
    assert_radiance_parity(img, g["image"], f"c4 {tag}")
    mega, st_m = sc.render(c["camera"], w, h, spp, b, integrator=rt.INTEGRATOR_MEGAKERNEL)
    assert np.array_equal(bits(img), bits(mega)) and st["rays"] == st_m["rays"]
    # the same materials installed by b200rt_scene_set_materials on a scene created with another roughness (how the sweep runs)
    base = scenes.c3_scene(roughness=0.25, nu=int(g["nu"]), nv=int(g["nv"]), sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    sc2 = scene_of(rt, base)
    sc2.set_materials(c["mats10"])
    img2, _ = sc2.render(c["camera"], w, h, spp, b)
    assert np.array_equal(bits(img), bits(img2))


# ---- BASELINE config 5 -----------------------------------------------------------------------------------------------------------------
def c5_small(g):
    from sycl_ray_tracing_b200 import scenes
    return scenes.c5_scene(n_instances=int(g["n_instances"]), nu=int(g["nu"]), nv=int(g["nv"]), sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))


@pytest.mark.parametrize("on_device", [False, True])
def test_c5_small_matches_reference(rt, on_device):
    g = load_golden("render_c5small.npz")
    c5 = c5_small(g)
    bvh = rt.BVH(c5["tri9"], on_device=on_device)
    bvh.check()
    sc = scene_of(rt, c5, bvh=bvh)
    prim, t, _ = sc.trace_primary(c5["camera"], int(g["pw"]), int(g["ph"]))
    assert np.array_equal(bits(t), bits(g["t"])) and np.array_equal(prim, g["prim_brute"])
    assert (prim != g["prim"]).sum() == 0
    img, st = sc.render(c5["camera"], int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"]))
    assert_radiance_parity(img, g["image"], "c5small")
    mega, st_m = sc.render(c5["camera"], int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"]), integrator=rt.INTEGRATOR_MEGAKERNEL)
    assert np.array_equal(bits(img), bits(mega)) and st["rays"] == st_m["rays"]


def test_rng_streams_on_the_gpu(rt):
    """xorshift32_generator known answers (tests/golden/xorshift.npz, rng_wrap.npz: produced by the compiled reference) against
    the device's pixel_rng / xs_float, including config 5's seeds whose x*y*spp wraps int32 (render_kernel.cpp:77)."""
    k = load_golden("xorshift.npz")
    cases = {31: (0, 7, 64), 591: (560, 1, 1), 1: (-30, 1, 1), 0xFFFFFFFF: (-32, 1, 1),
             (31 + 3839 * 2159 * 1024) & 0xFFFFFFFF: (3839, 2159, 1024)}
    for seed, (x, y, spp) in cases.items():
        st, fl = rt.rng_stream(x, y, spp, 32)
        assert st == int(k[f"state_{seed}"][0]), (seed, hex(st))
        assert np.array_equal(bits(fl), bits(k[f"floats_{seed}"])), seed
    w = load_golden("rng_wrap.npz")
    for x, y in w["pixels"]:
        st, fl = rt.rng_stream(int(x), int(y), int(w["spp"]), 16)
        assert st == int(w[f"state_{x}_{y}"][0]) and np.array_equal(bits(fl), bits(w[f"floats_{x}_{y}"])), (x, y)
    assert 3000 * 2000 * 1024 >= 2 ** 32, "the fixture's pixels must wrap"


def test_c5_full_scene_crops_against_oracle(rt):
    """BASELINE config 5's own scene: 20 000 002 triangles (device-built BVH, 12 levels of 8-ary nodes: deeper than the 10
    shared-memory stack entries of the default trace kernel), 3840x2160. (a) a 64x36 crop of a full 4-spp frame and (b) an
    8x4 crop at the configuration's real 1024 spp, placed where x*y*spp wraps int32, against the live oracle's crops."""
    from oracle.oracle import best_oracle
    from sycl_ray_tracing_b200 import scenes
    c5 = scenes.c5_scene()
    assert len(c5["tri9"]) == 20_000_002
    sc = scene_of(rt, c5)                                    # >= 5 M triangles: b200rt_scene_create builds on the device
    info = sc.bvh_info()
    assert info["wide_max_depth"] > 10, info
    w, h, b = 3840, 2160, 8
    full, st = sc.render(c5["camera"], w, h, 4, b)
    assert st["samples"] == w * h * 4 and np.isfinite(full).all()
    x0, y0, cw, ch = 1890, 700, 64, 36
    reg, _ = sc.render_region(c5["camera"], w, h, 4, b, x0, y0, x0 + cw, y0 + ch)
    assert np.array_equal(bits(reg), bits(full[y0:y0 + ch, x0:x0 + cw])), "region == the same pixels of the full wavefront frame"
    o = best_oracle()
    os_ = o.scene_from_arrays(c5["tri9"], c5["mat_idx"], c5["mats10"], c5["emissive"])
    os_.set_env(c5["env"])
    cam17 = c5["camera"].as_array17()
    ref, _ = os_.render_crop(cam17, w, h, 4, b, x0, y0, x0 + cw, y0 + ch)
    assert_radiance_parity(reg, ref, "c5 crop 4 spp")
    assert reg[..., :3].std() > 0.01, "the crop must show geometry, not a flat field"
    # (b) 1024 spp where the seed wraps: x*y*spp >= 2^32
    x1, y1 = 3000, 1431
    assert x1 * y1 * 1024 >= 2 ** 32
    reg2, st2 = sc.render_region(c5["camera"], w, h, 1024, b, x1, y1, x1 + 8, y1 + 4)
    ref2, _ = os_.render_crop(cam17, w, h, 1024, b, x1, y1, x1 + 8, y1 + 4)
    d = np.abs(reg2[..., :3].astype(np.float64) - ref2[..., :3].astype(np.float64))
    print("c5 wrap crop 1024 spp: max |diff|", d.max(), "rays/sample", st2["rays"] / st2["samples"])
    assert d.max() <= 1.0e-3, d.max()


def test_deep_tree_exercises_the_stack_overflow_path(rt):
    """A geometric chain of nested triangles (sizes 1 .. 2e4) gives the SAH builder a deep tree (8-ary depth 14, binary 17): rays
    along the chain push more than the 10 stack entries the cooperative trace kernel keeps in shared memory, so its
    local-memory overflow runs. Closest hits against numpy brute force; wavefront == megakernel bit for bit."""
    n = 2000
    s = 1.005 ** np.arange(n)
    tri = np.zeros((n, 9))
    tri[:, 0] = 3 * s; tri[:, 1] = -s; tri[:, 2] = -s           # wound so that the geometric normal faces -x, towards the camera below
    tri[:, 3] = 3 * s; tri[:, 4] = -s; tri[:, 5] = 2 * s
    tri[:, 6] = 3 * s; tri[:, 7] = 2 * s; tri[:, 8] = -s
    tri = tri.astype(np.float32)
    bvh = rt.BVH(tri)
    bvh.check()
    info = bvh.info()
    assert info["wide_max_depth"] > 10, info
    mats = np.array([[1, 0, 1, 1, 0, 0, 0, 1, 0, 1], [0, 0, 0, 1, .9, .8, .7, 1, 1.0, 0.3]], np.float32)
    sc = rt.Scene(tri, np.ones(n, np.int32), mats, np.zeros(0, np.int32), skysphere=rt.constant_env(1.0), bvh=bvh)
    rng = np.random.default_rng(3)
    o = np.stack([np.full(400, -1.0), rng.uniform(-0.5, 0.5, 400), rng.uniform(-0.5, 0.5, 400)], 1)
    d = np.stack([np.ones(400), rng.normal(0, 0.05, 400), rng.normal(0, 0.05, 400)], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    # and from the far end, looking back through every triangle
    o2 = np.stack([np.full(200, 3.0 * s[-1] * 1.5), rng.uniform(-1, 1, 200), rng.uniform(-1, 1, 200)], 1)
    d2 = np.stack([-np.ones(200), rng.normal(0, 0.02, 200), rng.normal(0, 0.02, 200)], 1)
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True)
    rays = np.concatenate([np.concatenate([o, d], 1), np.concatenate([o2, d2], 1)]).astype(np.float32)
    bp, bt = brute_force_closest(tri, rays)
    for flags in (0, rt.FLAG_BVH2):
        prim, t, _ = sc.trace_rays(rays, flags=flags)
        assert np.array_equal(prim, bp) and np.array_equal(bits(np.where(prim >= 0, t, 0)), bits(np.where(bp >= 0, bt, 0))), flags
    assert (bp >= 0).sum() > 300
    # the integrators: camera at the origin looking down +x through the whole chain (view matrix columns = camera axes)
    cam = rt.Camera.from_array17(np.array([0, 0, 1, -1.0, 0, 1, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 2.41421342], np.float32))
    wave, st_w = sc.render(cam, 96, 64, 3, 6)
    mega, st_m = sc.render(cam, 96, 64, 3, 6, integrator=rt.INTEGRATOR_MEGAKERNEL)
    assert np.array_equal(bits(wave), bits(mega)) and st_w["rays"] == st_m["rays"]
    assert st_w["rays"] > 96 * 64 * 3 * 2, "the camera must see the chain"
    pers, st_p = sc.render(cam, 96, 64, 3, 6, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(wave), bits(pers)) and st_p["rays"] == st_w["rays"]
    simple, _ = sc.render(cam, 96, 64, 3, 6, flags=rt.FLAG_SIMPLE_TRACE)
    assert np.array_equal(bits(wave), bits(simple))


# ---- BASELINE config 3 with its real sky, config 1 at full size -------------------------------------------------------------------------
def test_c3_crop_with_the_full_sky_against_oracle(rt):
    """Config 3 exactly as the bench renders it — 1 000 002 triangles under the 2048x1024 sky, whose 8 MiB float running-sum
    CDF stagnates once the sum is large (DESIGN.md) — a 64x36 crop of the 1920x1080 frame at 4 spp against the live oracle. The
    CDF the integrator searches was computed ON THE DEVICE in the reference's serial order: it must equal numpy's serial
    float32 cumsum bit for bit."""
    from oracle.oracle import best_oracle
    from sycl_ray_tracing_b200 import scenes
    c3 = scenes.c3_scene()
    assert c3["env"].shape == (1024, 2048, 4)
    sc = scene_of(rt, c3)
    assert np.array_equal(bits(sc.env_cdf()), bits(rt.compute_env_map_cdf(c3["env"]))), "device CDF != serial float32 running sum"
    w, h, spp, b = 1920, 1080, 4, 8
    o = best_oracle()
    os_ = o.scene_from_arrays(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"])
    os_.set_env(c3["env"])
    assert np.array_equal(bits(sc.env_cdf()), bits(os_.env_cdf())), "device CDF != the oracle's compute_env_map_cdf"
    full, _ = sc.render(c3["camera"], w, h, spp, b)
    for x0, y0 in ((928, 520), (700, 300)):              # sphere silhouette + ground; ground with the sun's reflection lobe
        ref, _ = os_.render_crop(c3["camera"].as_array17(), w, h, spp, b, x0, y0, x0 + 64, y0 + 36)
        assert_radiance_parity(full[y0:y0 + 36, x0:x0 + 64], ref, f"c3 crop at {x0},{y0}")


def test_c1_full_size_against_oracle(rt, golden_scenes):
    """BASELINE config 1 in full: cornell_pbr.obj, 512x512, 16 spp, 4 bounces, constant 1e-20 env (SURVEY §8c), CORNELL_BOX_CAMERA,
    against the live oracle's whole frame (< 1 s of CPU)."""
    from oracle.oracle import best_oracle
    a = scene_arrays(golden_scenes, "cornell")
    env = rt.constant_env(1.0e-20)
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=env)
    cam = rt.Camera.CORNELL_BOX_CAMERA
    img, st = sc.render(cam, 512, 512, 16, 4)
    o = best_oracle()
    os_ = o.scene_from_arrays(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"])
    os_.set_env(env)
    ref, _ = os_.render(cam.as_array17(), 512, 512, 16, 4)
    assert_radiance_parity(img, ref, "c1 full")
    assert 6.5 < st["rays"] / st["samples"] < 7.6, st          # the reference: 7.09 rays per camera sample (SURVEY §3.2)
    # the ray counter restarts with every frame, also for tile groups that own no tile of a small frame
    small, st_s = sc.render(cam, 16, 16, 2, 4)
    mega, st_sm = sc.render(cam, 16, 16, 2, 4, integrator=rt.INTEGRATOR_MEGAKERNEL)
    assert st_s["rays"] == st_sm["rays"] and np.array_equal(bits(small), bits(mega))


# ---- entry points added in round 2 -----------------------------------------------------------------------------------------------------
def test_region_and_single_pixel_entry(rt, golden_scenes, golden_cameras):
    """b200rt_render_region == the same pixels of the full frame, bit for bit (both integrators); one pixel =
    RenderKernel::ray_trace_pixel(x, y) (render_kernel.h:56) and the mirror class writes it into the framebuffer in place."""
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h, spp, b = 100, 70, 4, 5
    full, _ = sc.render(c, w, h, spp, b)
    reg, st = sc.render_region(c, w, h, spp, b, 37, 11, 91, 64)
    assert np.array_equal(bits(reg), bits(full[11:64, 37:91])) and st["samples"] == (91 - 37) * (64 - 11) * spp
    px = sc.ray_trace_pixel(c, w, h, spp, b, 50, 35)
    assert np.array_equal(bits(px), bits(full[35, 50]))
    with pytest.raises(rt.B200RTError):
        sc.render_region(c, w, h, spp, b, 10, 10, 10, 20)
    with pytest.raises(rt.B200RTError):
        sc.render_region(c, w, h, spp, b, 0, 0, w + 1, h)
    image = rt.Image(w, h)
    k = rt.RenderKernel(w, h, spp, b, image, a["tri9"], a["mats10"], a["emissive"], a["mat_idx"], [], None, rt.Image(data=g["env"]), None)
    k.set_camera(c)
    k.ray_trace_pixel(50, 35)
    assert np.array_equal(bits(image.pixels[35, 50]), bits(full[35, 50])) and (image.pixels[0, 0] == (0, 0, 0, 1)).all()


def test_render_rgba8_and_pinned_buffers(rt, golden_scenes, golden_cameras):
    """b200rt_render_rgba8 == write_image_png's quantisation of b200rt_render's frame (bit-exact, both flips, incoming framebuffer
    honoured); page-locked and pageable caller buffers give the same frame."""
    from oracle.oracle import quantise_rgba8
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h, spp, b = 1000, 700, 2, 4                      # 11 MB of float pixels: several staging chunks
    img, st = sc.render(c, w, h, spp, b)
    for flip in (True, False):
        q, st8 = sc.render_rgba8(c, w, h, spp, b, flip_y=flip)
        assert np.array_equal(q, quantise_rgba8(img, flip_y=flip)), flip
        assert st8["d2h_bytes"] == w * h * 4 and st8["rays"] == st["rays"]
    rng = np.random.default_rng(1)
    fb0 = (rng.random((h, w, 4)) * 0.3).astype(np.float32)
    fb = fb0.copy()
    sc.render(c, w, h, spp, b, framebuffer=fb)
    assert not np.array_equal(bits(fb), bits(img)), "a non-black incoming framebuffer must change the result"
    q, _ = sc.render_rgba8(c, w, h, spp, b, framebuffer=fb0)
    assert np.array_equal(q, quantise_rgba8(fb, flip_y=True))
    pinned = rt.Image(w, h, pinned=True)
    pinned.pixels[...] = fb0
    sc.render(c, w, h, spp, b, framebuffer=pinned.pixels)
    assert np.array_equal(bits(pinned.pixels), bits(fb))
    prim, t, _ = sc.trace_primary(c, w, h)
    prim_p, t_p = rt.pinned_array((h, w), np.int32), rt.pinned_array((h, w), np.float32)
    import ctypes as C
    from sycl_ray_tracing_b200 import binding as B
    o = B.RenderOptions(0, 0, 0, 1)
    B.check(B.load_library().b200rt_trace_primary(sc._h, B.fptr(c.as_array17()), w, h, -1, 1, B.iptr(prim_p), B.fptr(t_p), C.byref(o), None))
    assert np.array_equal(prim, prim_p) and np.array_equal(bits(t), bits(t_p))


def test_env_tables_built_on_the_device(rt):
    """K5: (a) the CDF computed on the device equals the reference's (tests/golden/env_cdf.npz, from Utils::compute_env_map_cdf)
    bit for bit; (b) the alias table built on the device (prefix sums + binary searches) implies the same per-texel
    distribution lum/total as the host's Vose table to 1e-6 relative; (c) an RGB (3-channel, as stbi_loadf returns it) env map
    expanded on the device renders the same frame as the RGBA Image."""
    from sycl_ray_tracing_b200 import scenes
    g = load_golden("env_cdf.npz")
    c3 = scenes.c3_scene(nu=40, nv=20, sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    sc = scene_of(rt, c3)
    assert np.array_equal(bits(sc.env_cdf()), bits(g["cdf"]))
    for env in (c3["env"], scenes.procedural_sky(512, 256), rt.constant_env(0.7, 16, 8)):
        d = dict(c3, env=env)
        s2 = scene_of(rt, d)
        assert np.array_equal(bits(s2.env_cdf()), bits(rt.compute_env_map_cdf(env)))
        s2.build_env_alias()
        prob, alias, total = s2.env_alias()
        hprob, halias, htotal = rt.env_alias_table(env)
        n = prob.size
        assert abs(total - htotal) <= 1e-6 * htotal
        assert ((prob >= 0) & (prob <= 1)).all() and ((alias >= 0) & (alias < n)).all()

        def implied(p, a):
            m = p.astype(np.float64).copy()
            np.add.at(m, a, 1.0 - p.astype(np.float64))
            return m / n
        px = env.reshape(-1, 4).astype(np.float64)
        lum = (0.3086 * px[:, 0] + 0.6094 * px[:, 1] + 0.0820 * px[:, 2]).astype(np.float32).astype(np.float64)
        want = lum / lum.sum()
        got_d, got_h = implied(prob, alias), implied(hprob, halias)
        assert np.abs(got_d - want).max() <= 2e-6 * want.max() + 1e-12, np.abs(got_d - want).max()
        assert np.abs(got_d - got_h).max() <= 2e-6 * want.max() + 1e-12
    rgb = dict(c3, env=np.ascontiguousarray(c3["env"][..., :3]))
    s3 = scene_of(rt, rgb)
    a, _ = sc.render(c3["camera"], 64, 40, 2, 4)
    b, _ = s3.render(c3["camera"], 64, 40, 2, 4)
    assert np.array_equal(bits(a), bits(b))


def test_set_materials_must_cover_every_referenced_index(rt, golden_scenes):
    a = scene_arrays(golden_scenes, "cornell")
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"])
    with pytest.raises(rt.B200RTError):
        sc.set_materials(a["mats10"][: int(a["mat_idx"].max())])
    sc.set_materials(a["mats10"][: int(a["mat_idx"].max()) + 1])


# ---- multi-device scenes behind the C ABI ----------------------------------------------------------------------------------------------
def multi_devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % have for i in range(n)]


@pytest.mark.parametrize("n_ranks", [2, 3])
def test_multi_device_scene_equals_single_device(rt, golden_scenes, golden_cameras, n_ranks):
    """b200rt_scene_create_multi + b200rt_render: N ranks inside one process (on a one-GPU box they share the device),
    interleaved tiles rendered as mean radiance, peer copies into rank 0's gather buffer, `fb += final; tone map` there.
    Bit-identical to the single-device frame — with a non-black incoming framebuffer — and the same ray count."""
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    single = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    multi = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"], devices=multi_devices(n_ranks))
    assert multi.device_count() == n_ranks
    w, h, spp, b = 200, 150, 3, 5
    rng = np.random.default_rng(2)
    fb0 = (rng.random((h, w, 4)) * 0.2).astype(np.float32)
    for integ in (rt.INTEGRATOR_WAVEFRONT, rt.INTEGRATOR_MEGAKERNEL):
        fb_s, fb_m = fb0.copy(), fb0.copy()
        _, st_s = single.render(c, w, h, spp, b, framebuffer=fb_s, integrator=integ)
        _, st_m = multi.render(c, w, h, spp, b, framebuffer=fb_m, integrator=integ)
        assert np.array_equal(bits(fb_s), bits(fb_m)), f"{(bits(fb_s) != bits(fb_m)).sum()} words differ"
        assert st_s["rays"] == st_m["rays"] and st_m["samples"] == w * h * spp
    z_s, _ = single.render(c, w, h, spp, b)
    z_m, _ = multi.render(c, w, h, spp, b)
    assert np.array_equal(bits(z_s), bits(z_m))
    q_s, _ = single.render_rgba8(c, w, h, spp, b)
    q_m, _ = multi.render_rgba8(c, w, h, spp, b)
    assert np.array_equal(q_s, q_m)
    multi.set_materials(a["mats10"] * np.float32(0.5))
    single.set_materials(a["mats10"] * np.float32(0.5))
    assert np.array_equal(bits(single.render(c, w, h, 1, 3)[0]), bits(multi.render(c, w, h, 1, 3)[0]))
    with pytest.raises(rt.B200RTError):
        multi.render(c, w, h, 1, 1, rank=1, world=2)


def test_linear_tiles_and_accumulating_untile(rt, golden_scenes, golden_cameras):
    """The torchrun path's building blocks: B200RT_FLAG_LINEAR_TILES tile buffers + b200rt_untile_accumulate_device reproduce
    b200rt_render on a non-black framebuffer bit for bit."""
    import torch
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    w, h, spp, b, world = 120, 90, 2, 4, 3
    rng = np.random.default_rng(4)
    fb0 = (rng.random((h, w, 4)) * 0.2).astype(np.float32)
    want = fb0.copy()
    sc.render(c, w, h, spp, b, framebuffer=want)
    padded = rt.tiles_for_rank(w, h, 0, world)
    gathered = torch.zeros((world, padded * 256, 4), dtype=torch.float32, device="cuda")
    for r in range(world):
        sc.render_tiles_device(c, w, h, spp, b, gathered[r].data_ptr(), flags=rt.FLAG_LINEAR_TILES, rank=r, world=world)
    fb = torch.from_numpy(fb0).cuda()
    sc.untile_accumulate_device(gathered.data_ptr(), padded, world, w, h, fb.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(bits(fb.cpu().numpy()), bits(want))


# ---- persistent integrator (csrc/persist.cu) ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key,fixture", [("cornell", "render_cornell_c1.npz"), ("cornell", "render_cornell_env.npz"), ("mis", "render_mis_env.npz"),
                                         ("area", "render_area_c1.npz"), ("cornell", "sphere_cornell.npz")])
def test_persistent_integrator_equals_megakernel_bit_for_bit(rt, golden_scenes, golden_cameras, key, fixture):
    """One launch per frame, every warp its own wavefront machine: the same device functions on the same per-pixel RNG streams as the
    other two integrators -> identical framebuffers (NaN pixels included) and identical ray counts; and the reference's frame
    within the stated tolerance."""
    g = load_golden(fixture)
    w, h, spp, b = int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"])
    a = scene_arrays(golden_scenes, key)
    if fixture == "sphere_cornell.npz":
        n = len(a["tri9"])
        mat_idx = np.concatenate([a["mat_idx"], np.array([len(g["mats10"]) - 1], np.int32)])
        sph = [((float(g["spheres4"][0, 0]), float(g["spheres4"][0, 1]), float(g["spheres4"][0, 2])), float(g["spheres4"][0, 3]), n)]
        sc = rt.Scene(a["tri9"], mat_idx, g["mats10"], a["emissive"], spheres=sph, skysphere=g["env"])
    else:
        sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras[{"cornell": "cornell", "mis": "mis", "area": "cornell"}[key]])
    mega, st_m = sc.render(c, w, h, spp, b, integrator=rt.INTEGRATOR_MEGAKERNEL)
    pers, st_p = sc.render(c, w, h, spp, b, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(mega), bits(pers)), f"{(bits(mega) != bits(pers)).sum()} differing words"
    assert st_m["rays"] == st_p["rays"] and st_p["gpu_launches"] <= 3
    assert_radiance_parity(pers, g["image"], f"persistent {fixture}")
    # a non-black incoming framebuffer, a frame that is not a multiple of the tile size, interleaved ranks
    rng = np.random.default_rng(5)
    w2, h2 = 100, 70
    fb0 = (rng.random((h2, w2, 4)) * 0.2).astype(np.float32)
    want = fb0.copy(); sc.render(c, w2, h2, 2, 4, framebuffer=want)
    one = fb0.copy(); sc.render(c, w2, h2, 2, 4, framebuffer=one, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(want), bits(one)), f"non-black framebuffer: {(bits(want) != bits(one)).any(axis=-1).sum()} pixels differ"
    black_w, _ = sc.render(c, w2, h2, 2, 4)
    black = rt.Image(w2, h2).pixels
    for rank in range(3):
        sc.render(c, w2, h2, 2, 4, framebuffer=black, integrator=rt.INTEGRATOR_PERSISTENT, rank=rank, world=3)
    assert np.array_equal(bits(black_w), bits(black)), f"ranks: {(bits(black_w) != bits(black)).any(axis=-1).sum()} pixels differ"
    got = fb0.copy()
    for rank in range(3):
        sc.render(c, w2, h2, 2, 4, framebuffer=got, integrator=rt.INTEGRATOR_PERSISTENT, rank=rank, world=3)
    diff = (bits(want) != bits(got)).any(axis=-1)
    assert not diff.any(), f"ranks + non-black framebuffer: {diff.sum()} pixels differ, first at {np.argwhere(diff)[:5].tolist()}"
    zero, _ = sc.render(c, 40, 30, 0, 4, integrator=rt.INTEGRATOR_PERSISTENT)
    zero_w, _ = sc.render(c, 40, 30, 0, 4)
    assert np.array_equal(bits(zero), bits(zero_w))


def test_persistent_integrator_c3_and_multi_device(rt, golden_cameras):
    from sycl_ray_tracing_b200 import scenes
    g = load_golden("render_c3small.npz")
    c3 = scenes.c3_scene(roughness=float(g["roughness"]), nu=int(g["nu"]), nv=int(g["nv"]), sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    sc = scene_of(rt, c3)
    w, h, spp, b = int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"])
    wave, st_w = sc.render(c3["camera"], w, h, spp, b)
    pers, st_p = sc.render(c3["camera"], w, h, spp, b, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(wave), bits(pers)) and st_w["rays"] == st_p["rays"]
    skip, st_s = sc.render(c3["camera"], w, h, spp, b, integrator=rt.INTEGRATOR_PERSISTENT, flags=rt.FLAG_SKIP_DEAD_RAYS)
    assert np.array_equal(bits(wave), bits(skip)) and st_s["rays"] < st_p["rays"]
    # a larger frame than the persistent grid has slots: slots are re-used as pixels finish
    big_w, st_bw = sc.render(c3["camera"], 1280, 720, 2, 8)
    big_p, st_bp = sc.render(c3["camera"], 1280, 720, 2, 8, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(big_w), bits(big_p)) and st_bw["rays"] == st_bp["rays"]
    multi = scene_of(rt, c3, devices=multi_devices(2))
    m, st_mu = multi.render(c3["camera"], w, h, spp, b, integrator=rt.INTEGRATOR_PERSISTENT)
    assert np.array_equal(bits(wave), bits(m)) and st_mu["rays"] == st_w["rays"]
    # leaves of more than 3 triangles have no 8-ary layout: the persistent integrator must say so, not fall back
    fat = scene_of(rt, c3, bvh=rt.BVH(c3["tri9"], max_leaf_size=8))
    with pytest.raises(rt.B200RTError):
        fat.render(c3["camera"], 32, 32, 1, 2, integrator=rt.INTEGRATOR_PERSISTENT)


def test_progressive_accumulation_equals_one_shot(rt, golden_scenes, golden_cameras):
    """b200rt_accum_*: 16 spp streamed as 1 + 4 + 3 + 8 samples (each pixel's RNG stream continued across the chunks, linear sums
    kept on the device) == one b200rt_render(16), bit for bit, with a non-black incoming framebuffer; the intermediate resolves
    are proper running means; both barrier styles of the integrator."""
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h, spp, b = 100, 70, 16, 5
    rng = np.random.default_rng(6)
    fb0 = (rng.random((h, w, 4)) * 0.2).astype(np.float32)
    want = fb0.copy()
    _, st = sc.render(c, w, h, spp, b, framebuffer=want)
    for integ in (rt.INTEGRATOR_WAVEFRONT, rt.INTEGRATOR_PERSISTENT):
        acc = rt.Accumulator(sc, c, w, h, spp, b)
        rays, partial = 0, None
        for i, n in enumerate((1, 4, 3, 8)):
            rays += acc.add(n, integrator=integ)["rays"]
            if i == 1:
                partial = acc.resolve()
        assert acc.samples() == spp and rays == st["rays"]
        assert np.array_equal(bits(acc.resolve(fb0)), bits(want)), integ
        assert np.array_equal(bits(acc.resolve(fb0)), bits(want)), "resolve must not consume the accumulator"
        five, _ = sc.render(c, w, h, 5, b)          # a 5-spp frame uses another seed (31 + x*y*5): only statistically comparable
        assert abs(float(partial[..., :3].mean()) - float(five[..., :3].mean())) < 0.02
        with pytest.raises(rt.B200RTError):
            acc.add(1)


def test_env_cdf_search_guide_is_exact(rt):
    """env_map_cdf_search (render_kernel.cpp:532-567) on the device, through the guide table and without it, against a numpy
    restatement of the reference's two binary searches: the same texel for every value — random draws, every bucket boundary
    neighbourhood, exact table values, 0 and the largest draw — on the 2048x1024 sun+sky (whose float running sum stagnates)."""
    from sycl_ray_tracing_b200 import scenes
    c3 = scenes.c3_scene(nu=20, nv=10)
    sc = scene_of(rt, c3)
    cdf = rt.compute_env_map_cdf(c3["env"])
    h, w = c3["env"].shape[:2]
    total = cdf[-1]
    rng = np.random.default_rng(9)
    draws = np.minimum(rng.integers(0, 2 ** 32, 300000, dtype=np.uint64).astype(np.float32) * np.float32(2.0 ** -32), np.float32(1.0 - 1.0e-6))
    vals = [draws * total, cdf[rng.integers(0, cdf.size, 50000)], np.nextafter(cdf[rng.integers(0, cdf.size, 50000)], np.float32(0)),
            (np.arange(0, 65537, dtype=np.float64) / (65536.0 / float(total))).astype(np.float32),
            np.array([0.0, np.float32(1.0 - 1.0e-6) * total, total, np.nextafter(total, np.float32(0))], np.float32)]
    v = np.concatenate(vals).astype(np.float32)
    # the reference's searches: first row whose last column exceeds the value (else the last row), then first column in that row (else the last)
    rows = cdf.reshape(h, w)
    y = np.minimum(np.searchsorted(rows[:, -1], v, side="right"), h - 1)
    x = np.array([min(int(np.searchsorted(rows[yy], vv, side="right")), w - 1) for yy, vv in zip(y[:20000], v[:20000])])
    plain = sc.env_cdf_search(v, use_guide=False)
    guided = sc.env_cdf_search(v, use_guide=True)
    assert np.array_equal(plain, guided), f"{(plain != guided).any(axis=1).sum()} values pick another texel through the guide"
    assert np.array_equal(plain[:, 1], y) and np.array_equal(plain[:20000, 0], x)


def test_denoise_stage(rt, golden_cameras):
    """b200rt_denoise (the stage Utils::OIDN_denoise occupies, utils.cpp:144-196): not OIDN, so no parity claim — functional checks:
    a constant image is a fixed point, blend 0 returns the input, a clean step edge stays a step, and on a noisy 4-spp render the
    filtered frame is closer to the 1024-spp frame than the noisy one (RMSE), for float3 and RGBA layouts alike."""
    from sycl_ray_tracing_b200 import scenes
    const = np.full((40, 60, 3), 0.37, np.float32)
    assert np.allclose(rt.OIDN_denoise(const), const, atol=1e-6)
    step = np.zeros((64, 64, 4), np.float32); step[:, 32:, :3] = 0.9; step[..., 3] = 2.5
    out = rt.OIDN_denoise(step)
    assert np.abs(out[..., :3] - step[..., :3]).max() < 5e-3 and np.allclose(out[..., 3], 1.0), "edges survive; alpha -> 1 (utils.cpp:186)"
    c3 = scenes.c3_scene(nu=100, nv=50, sky_w=64, sky_h=32)
    sc = scene_of(rt, c3)
    noisy, _ = sc.render(c3["camera"], 320, 180, 4, 8)
    ref, _ = sc.render(c3["camera"], 320, 180, 1024, 8)
    assert np.array_equal(bits(rt.OIDN_denoise(noisy, blend_factor=0.0)[..., :3]), bits(noisy[..., :3]))
    den4 = rt.OIDN_denoise(noisy)
    den3 = rt.OIDN_denoise(np.ascontiguousarray(noisy[..., :3]))
    assert np.array_equal(bits(den4[..., :3]), bits(den3))
    rmse = lambda a: float(np.sqrt(((a[..., :3].astype(np.float64) - ref[..., :3]) ** 2).mean()))
    half = rt.OIDN_denoise(noisy, blend_factor=0.5)
    print("rmse noisy", rmse(noisy), "denoised", rmse(den4), "blend 0.5", rmse(half))
    assert rmse(den4) < 0.8 * rmse(noisy) and rmse(half) < rmse(noisy)
    assert np.allclose(half[..., :3], 0.5 * den4[..., :3] + 0.5 * noisy[..., :3], atol=1e-6)


# ---- barrier-free tail of a pass-synchronous frame (csrc/persist.cu) ----------------------------------------------------------------------
def test_tail_continuation_equals_passes_bit_for_bit(rt, golden_scenes, golden_cameras):
    """The default wavefront frame finishes each tile group's last few pixels with one barrier-free wf_tail launch (every warp runs a
    few slots to the end on its own): same device functions, same per-pixel RNG streams -> the frame and the ray count equal the pure
    pass-synchronous frame's (B200RT_FLAG_WF_PASSES_ONLY) and the megakernel's, bit for bit: groups that are barrier-free from the first
    pass (small frames), groups that switch once few pixels are left (a 1280x720 frame), interleaved ranks with a non-black incoming
    framebuffer, spheres, emissive triangles (MIS.obj), and the dead-ray elimination (slots that are alive without a ray)."""
    from sycl_ray_tracing_b200 import scenes
    for key, fixture in [("cornell", "render_cornell_env.npz"), ("mis", "render_mis_env.npz")]:
        g = load_golden(fixture)
        w, h, spp, b = int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"])
        a = scene_arrays(golden_scenes, key)
        sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
        c = rt.Camera.from_array17(golden_cameras[key])
        mega, st_m = sc.render(c, w, h, spp, b, integrator=rt.INTEGRATOR_MEGAKERNEL)
        pas, st_p = sc.render(c, w, h, spp, b, flags=rt.FLAG_WF_PASSES_ONLY)
        tail, st_t = sc.render(c, w, h, spp, b)
        for name, img, st in (("passes", pas, st_p), ("default", tail, st_t)):
            assert np.array_equal(bits(mega), bits(img)), f"{fixture} {name}: {(bits(mega) != bits(img)).any(axis=-1).sum()} pixels differ"
            assert st["rays"] == st_m["rays"], (fixture, name, st["rays"], st_m["rays"])
        assert st_t["gpu_launches"] < st_p["gpu_launches"], "the small frame is barrier-free from its first pass"
        assert_radiance_parity(tail, g["image"], f"default {fixture}")
        rng = np.random.default_rng(11)
        w2, h2 = 100, 70
        fb0 = (rng.random((h2, w2, 4)) * 0.2).astype(np.float32)
        want = fb0.copy(); sc.render(c, w2, h2, 3, 4, framebuffer=want, flags=rt.FLAG_WF_PASSES_ONLY)
        got = fb0.copy()
        for rank in range(3):
            sc.render(c, w2, h2, 3, 4, framebuffer=got, rank=rank, world=3)
        assert np.array_equal(bits(want), bits(got)), "ranks + non-black framebuffer"
    g = load_golden("render_c3small.npz")
    c3 = scenes.c3_scene(roughness=float(g["roughness"]), nu=int(g["nu"]), nv=int(g["nv"]), sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    sc = scene_of(rt, c3)
    for (w, h, spp) in ((640, 360, 6), (1280, 720, 4), (1920, 1080, 2)):
        pas, st_p = sc.render(c3["camera"], w, h, spp, 8, flags=rt.FLAG_WF_PASSES_ONLY)
        tail, st_t = sc.render(c3["camera"], w, h, spp, 8)
        assert np.array_equal(bits(pas), bits(tail)), f"c3 {w}x{h}: {(bits(pas) != bits(tail)).any(axis=-1).sum()} pixels differ"
        assert st_p["rays"] == st_t["rays"]
        skip_p, st_sp = sc.render(c3["camera"], w, h, spp, 8, flags=rt.FLAG_WF_PASSES_ONLY | rt.FLAG_SKIP_DEAD_RAYS)
        skip_t, st_st = sc.render(c3["camera"], w, h, spp, 8, flags=rt.FLAG_SKIP_DEAD_RAYS)
        assert np.array_equal(bits(pas), bits(skip_t)) and st_sp["rays"] == st_st["rays"] < st_p["rays"]
    # a longer chain (24 spp): same frame and ray count as passes only and as the megakernel; also as one rank of 2
    for kw in (dict(), dict(rank=1, world=2)):
        tail, st_t = sc.render(c3["camera"], 960, 540, 24, 8, **kw)
        pas, st_p = sc.render(c3["camera"], 960, 540, 24, 8, flags=rt.FLAG_WF_PASSES_ONLY, **kw)
        assert np.array_equal(bits(tail), bits(pas)), kw
        assert st_t["rays"] == st_p["rays"], (kw, st_t["rays"], st_p["rays"])
    mega, st_m = sc.render(c3["camera"], 960, 540, 24, 8, integrator=rt.INTEGRATOR_MEGAKERNEL)
    tail, st_t = sc.render(c3["camera"], 960, 540, 24, 8)
    assert np.array_equal(bits(tail), bits(mega)) and st_t["rays"] == st_m["rays"]
    # one rank of 8 of the 1080p frame (latency-bound passes: the shape the tail exists for), twice: the second frame starts from
    # whatever the first left in the group buffers
    want, st_w = sc.render(c3["camera"], 1920, 1080, 3, 8, rank=5, world=8, flags=rt.FLAG_WF_PASSES_ONLY)
    for _ in range(2):
        got, st_g = sc.render(c3["camera"], 1920, 1080, 3, 8, rank=5, world=8)
        assert np.array_equal(bits(want), bits(got)) and st_w["rays"] == st_g["rays"]
    # analytic spheres finish inside the tracer lanes
    gs = load_golden("sphere_cornell.npz")
    a = scene_arrays(golden_scenes, "cornell")
    n = len(a["tri9"])
    mat_idx = np.concatenate([a["mat_idx"], np.array([len(gs["mats10"]) - 1], np.int32)])
    sph = [((float(gs["spheres4"][0, 0]), float(gs["spheres4"][0, 1]), float(gs["spheres4"][0, 2])), float(gs["spheres4"][0, 3]), n)]
    scs = rt.Scene(a["tri9"], mat_idx, gs["mats10"], a["emissive"], spheres=sph, skysphere=gs["env"])
    cs = rt.Camera.from_array17(golden_cameras["cornell"])
    ws, hs, spps, bs = int(gs["w"]), int(gs["h"]), int(gs["spp"]), int(gs["bounces"])
    m, st_m = scs.render(cs, ws, hs, spps, bs, integrator=rt.INTEGRATOR_MEGAKERNEL)
    s_t, st_t = scs.render(cs, ws, hs, spps, bs)
    assert np.array_equal(bits(m), bits(s_t)) and st_m["rays"] == st_t["rays"]
