"""-m gpu: progressive accumulation on multi-device scenes (b200rt_accum_* on a b200rt_scene_create_multi scene) and the RGBA8 resolve
(b200rt_accum_resolve_rgba8). A pixel depends only on (x, y, spp, scene, camera), never on which device or tile split renders it, so
every result here has an exact oracle: the single-device render or the single-device accumulator, bit for bit, ray counts included.
On a one-GPU box the ranks share device 0; with several GPUs they run on distinct devices."""
import ctypes as C
import gc

import numpy as np
import pytest

from conftest import load_golden, scene_arrays

pytestmark = pytest.mark.gpu

W, H, SPP, BOUNCES = 100, 70, 16, 5          # not a multiple of the 16x16 tile
CHUNKS = (1, 4, 3, 8)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same_bits(got, want, what=""):
    diff = (bits(got) != bits(want)).any(axis=-1)
    assert not diff.any(), f"{what}: {diff.sum()} pixels differ, first at {np.argwhere(diff)[:5].tolist()}"


def multi_devices(n):
    import torch
    have = torch.cuda.device_count()
    return [i % have for i in range(n)]


def cornell(rt, golden_scenes, devices=None):
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    return rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"], devices=devices)


def incoming_framebuffer(w=W, h=H, seed=6):
    rng = np.random.default_rng(seed)
    return (rng.random((h, w, 4)) * 0.2).astype(np.float32)


def integrator_of(rt, name):
    return {"wavefront": rt.INTEGRATOR_WAVEFRONT, "persistent": rt.INTEGRATOR_PERSISTENT}[name]


@pytest.mark.parametrize("integrator", ["wavefront", "persistent"])
@pytest.mark.parametrize("n_ranks", [2, 3])
def test_multi_device_chunks_equal_one_render(rt, golden_scenes, golden_cameras, n_ranks, integrator):
    """16 spp streamed as 1 + 4 + 3 + 8 samples on N ranks, resolved onto a non-black framebuffer == b200rt_render(16) on a
    single-device scene and on the same multi-device scene; the chunks' summed ray count == the single-device render's."""
    integ = integrator_of(rt, integrator)
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    single = cornell(rt, golden_scenes)
    multi = cornell(rt, golden_scenes, devices=multi_devices(n_ranks))
    assert multi.device_count() == n_ranks
    fb0 = incoming_framebuffer()
    want = fb0.copy()
    _, st = single.render(c, W, H, SPP, BOUNCES, framebuffer=want)
    want_multi = fb0.copy()
    multi.render(c, W, H, SPP, BOUNCES, framebuffer=want_multi)
    acc = rt.Accumulator(multi, c, W, H, SPP, BOUNCES)
    rays = 0
    for n in CHUNKS:
        s = acc.add(n, integrator=integ)
        assert s["samples"] == W * H * n and s["gpu_launches"] >= n_ranks and s["kernel_ms"] > 0.0, s
        rays += s["rays"]
    assert acc.samples() == SPP and rays == st["rays"], (rays, st["rays"])
    got = acc.resolve(fb0)
    assert_same_bits(got, want, f"{n_ranks} ranks, {integrator} vs single-device render")
    assert_same_bits(got, want_multi, f"{n_ranks} ranks, {integrator} vs multi-device render")


@pytest.mark.parametrize("n_ranks", [2, 3])
def test_intermediate_resolves_equal_single_device_accumulator(rt, golden_scenes, golden_cameras, n_ranks):
    """After 1 and after 5 samples the multi-device resolve equals the single-device accumulator's resolve after the same chunks,
    bit for bit, with and without an incoming framebuffer; resolving again gives the same bits (a resolve consumes nothing)."""
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    single = cornell(rt, golden_scenes)
    multi = cornell(rt, golden_scenes, devices=multi_devices(n_ranks))
    acc_s = rt.Accumulator(single, c, W, H, SPP, BOUNCES)
    acc_m = rt.Accumulator(multi, c, W, H, SPP, BOUNCES)
    fb0 = incoming_framebuffer(seed=7)
    for n in CHUNKS[:2]:
        st_s, st_m = acc_s.add(n), acc_m.add(n)
        assert st_s["rays"] == st_m["rays"] and st_s["samples"] == st_m["samples"]
        for fb in (None, fb0):
            want = acc_s.resolve(fb)
            first = acc_m.resolve(fb)
            assert_same_bits(first, want, f"after {acc_m.samples()} samples, fb {'given' if fb is not None else 'black'}")
            assert_same_bits(acc_m.resolve(fb), first, "a second resolve")


def test_rank_without_tiles(rt, golden_scenes, golden_cameras):
    """A 24x8 frame has 2 tiles: on 3 ranks the third owns none. The accumulation still equals the single-device render, float and
    RGBA8, for both integrators."""
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h, spp = 24, 8, 4
    assert rt.tiles_for_rank(w, h, 2, 3) == 0
    single = cornell(rt, golden_scenes)
    multi = cornell(rt, golden_scenes, devices=multi_devices(3))
    fb0 = incoming_framebuffer(w, h, seed=8)
    want = fb0.copy()
    _, st = single.render(c, w, h, spp, BOUNCES, framebuffer=want)
    want8, _ = single.render_rgba8(c, w, h, spp, BOUNCES, framebuffer=fb0)
    for integ in (rt.INTEGRATOR_WAVEFRONT, rt.INTEGRATOR_PERSISTENT):
        acc = rt.Accumulator(multi, c, w, h, spp, BOUNCES)
        rays = acc.add(1, integrator=integ)["rays"] + acc.add(spp - 1, integrator=integ)["rays"]
        assert rays == st["rays"]
        assert_same_bits(acc.resolve(fb0), want, f"integrator {integ}")
        assert np.array_equal(acc.resolve_rgba8(fb0), want8)


def test_c3_small_on_two_ranks(rt):
    """The C3-small fixture's frame (the C3 scene at the fixture's tessellation, its sky, the default wavefront with its barrier-free
    tail) on 2 ranks, accumulated in 2 chunks == the one-shot single-device wavefront frame, bit for bit."""
    from sycl_ray_tracing_b200 import scenes
    g = load_golden("render_c3small.npz")
    c3 = scenes.c3_scene(roughness=float(g["roughness"]), nu=int(g["nu"]), nv=int(g["nv"]), sky_w=int(g["sky_w"]), sky_h=int(g["sky_h"]))
    w, h, spp, b = int(g["w"]), int(g["h"]), int(g["spp"]), int(g["bounces"])
    single = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"])
    multi = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"], devices=multi_devices(2))
    want, st = single.render(c3["camera"], w, h, spp, b)
    acc = rt.Accumulator(multi, c3["camera"], w, h, spp, b)
    rays = acc.add(spp // 2)["rays"] + acc.add(spp - spp // 2)["rays"]
    assert rays == st["rays"]
    assert_same_bits(acc.resolve(), want, "c3 small, 2 ranks")


def test_renders_between_adds_leave_the_accumulation_alone(rt, golden_scenes, golden_cameras):
    """Scene.render and Scene.render_rgba8 on the same multi-device scene between two adds (same frame size, and a larger one that
    regrows the scene's gather buffer) leave the final resolve bit-identical."""
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    single = cornell(rt, golden_scenes)
    multi = cornell(rt, golden_scenes, devices=multi_devices(3))
    fb0 = incoming_framebuffer(seed=9)
    want = fb0.copy()
    single.render(c, W, H, SPP, BOUNCES, framebuffer=want)
    acc = rt.Accumulator(multi, c, W, H, SPP, BOUNCES)
    acc.add(5)
    partial = acc.resolve(fb0)
    multi.render(c, W, H, 3, 4)
    multi.render_rgba8(c, W, H, 2, 3, framebuffer=fb0)
    multi.render(c, 2 * W, 2 * H, 1, 3)
    multi.render_rgba8(c, 2 * W, 2 * H, 1, 3)
    assert_same_bits(acc.resolve(fb0), partial, "partial resolve after renders")
    acc.add(SPP - 5)
    assert_same_bits(acc.resolve(fb0), want, "final resolve")


def test_refused_calls_change_nothing(rt, golden_scenes, golden_cameras):
    """rank/world other than 0/1, the megakernel, more samples than spp_total and a resolve before any add are refused with
    B200RTError, before any rank launches; completing the accumulation afterwards still gives the exact frame."""
    from sycl_ray_tracing_b200 import binding as B
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    single = cornell(rt, golden_scenes)
    multi = cornell(rt, golden_scenes, devices=multi_devices(2))
    fb0 = incoming_framebuffer(seed=10)
    want = fb0.copy()
    single.render(c, W, H, SPP, BOUNCES, framebuffer=want)
    acc = rt.Accumulator(multi, c, W, H, SPP, BOUNCES)

    def refusals():
        before = acc.samples()
        with pytest.raises(rt.B200RTError):
            o, st = B.RenderOptions(rt.INTEGRATOR_WAVEFRONT, 0, 1, 2), B.Stats()
            B.check(B.load_library().b200rt_accum_add(acc._h, 1, C.byref(o), C.byref(st)))
        with pytest.raises(rt.B200RTError):
            acc.add(1, integrator=rt.INTEGRATOR_MEGAKERNEL)
        with pytest.raises(rt.B200RTError):
            acc.add(SPP - before + 1)
        assert acc.samples() == before

    with pytest.raises(rt.B200RTError):
        acc.resolve()
    with pytest.raises(rt.B200RTError):
        acc.resolve_rgba8()
    refusals()
    acc.add(6)
    refusals()
    acc.add(SPP - 6)
    refusals()
    assert_same_bits(acc.resolve(fb0), want, "after refused calls")


@pytest.mark.parametrize("n_ranks", [1, 2])
def test_rgba8_resolve(rt, golden_scenes, golden_cameras, n_ranks):
    """resolve_rgba8(fb) == quantise_rgba8(resolve(fb)) byte for byte, partial and complete, both flips, with and without an incoming
    framebuffer; complete, it equals render_rgba8(spp_total)."""
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    sc = cornell(rt, golden_scenes, devices=None if n_ranks == 1 else multi_devices(n_ranks))
    fb0 = incoming_framebuffer(seed=11)
    acc = rt.Accumulator(sc, c, W, H, SPP, BOUNCES)
    for n in (5, SPP - 5):
        acc.add(n)
        for fb in (None, fb0):
            img = acc.resolve(fb)
            for flip in (False, True):
                assert np.array_equal(acc.resolve_rgba8(fb, flip_y=flip), rt.quantise_rgba8(img, flip_y=flip)), (acc.samples(), flip)
    for fb in (None, fb0):
        for flip in (False, True):
            want, _ = sc.render_rgba8(c, W, H, SPP, BOUNCES, framebuffer=fb, flip_y=flip)
            assert np.array_equal(acc.resolve_rgba8(fb, flip_y=flip), want), flip


def test_current_device_is_restored(rt, golden_scenes, golden_cameras):
    """With ranks on distinct devices, create / add / resolve / destroy leave the calling thread's current device as they found it,
    whichever device that is."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    multi = cornell(rt, golden_scenes, devices=[1, 0])
    for cur in (0, 1):
        torch.cuda.set_device(cur)
        acc = rt.Accumulator(multi, c, W, H, 4, BOUNCES)
        assert torch.cuda.current_device() == cur
        acc.add(2)
        assert torch.cuda.current_device() == cur
        acc.resolve()
        acc.resolve_rgba8()
        assert torch.cuda.current_device() == cur
        del acc
        gc.collect()
        assert torch.cuda.current_device() == cur
    torch.cuda.set_device(0)
