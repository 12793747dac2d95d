"""Feature buffers for a denoiser (b200rt_render_aovs) and the à-trous filter guided by them (b200rt_denoise_guided, the OIDN drop-in's
"albedo" / "normal" images). The GPU tests are marked gpu; the argument and no-device checks at the end run anywhere."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, load_golden, scene_arrays

gpu = pytest.mark.gpu
CAM_OF = {"cornell": "cornell", "mis": "mis", "area": "cornell"}
f32 = np.float32


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def make_scene(rt, golden_scenes, key, **kw):
    a = scene_arrays(golden_scenes, key)
    return rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], **kw), a


def geometric_normals(tri9):
    """normalize(cross(b - a, c - a)) in float32, in the operation order of triangle.h / vec.h."""
    t = np.asarray(tri9, f32).reshape(-1, 9)
    u = (t[:, 3:6] - t[:, 0:3]).astype(f32)
    v = (t[:, 6:9] - t[:, 0:3]).astype(f32)
    c = np.stack([u[:, 1] * v[:, 2] - u[:, 2] * v[:, 1], u[:, 2] * v[:, 0] - u[:, 0] * v[:, 2], u[:, 0] * v[:, 1] - u[:, 1] * v[:, 0]], 1).astype(f32)
    length = np.sqrt((c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]).astype(f32) + c[:, 2] * c[:, 2]).astype(f32)
    return ((f32(1.0) / length)[:, None] * c).astype(f32)


def neighbourhood_labels(label, h, w):
    """for every pixel, the number of distinct labels in its 3x3 neighbourhood (clamped at the frame border)"""
    pad = np.pad(label.reshape(h, w), 1, mode="edge")
    stack = np.stack([pad[dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3)], -1)
    return np.array([len(np.unique(s)) for s in stack.reshape(h * w, 9)]).reshape(h, w)


# ---- feature buffers ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("key", ["cornell", "mis", "area"])
def test_aov_one_ray_per_pixel_is_the_primary_hit(rt, golden_scenes, golden_cameras, key):
    """k = 1 traces exactly b200rt_trace_primary's un-jittered ray: the albedo is the hit material's diffuse colour bit for bit, the
    normal the triangle's geometric normal; misses are 0. Every BVH layout gives the same buffers."""
    g = load_golden(f"primary_{key}.npz")
    w, h = int(g["w"]), int(g["h"])
    sc, a = make_scene(rt, golden_scenes, key)
    c = rt.Camera.from_array17(golden_cameras[CAM_OF[key]])
    prim, _, _ = sc.trace_primary(c, w, h)
    albedo, normal, st = sc.render_aovs(c, w, h, samples_per_axis=1)
    assert st["rays"] == w * h
    hit = prim >= 0
    assert hit.any() and albedo.shape == (h, w, 3) and normal.shape == (h, w, 3)
    want_albedo = np.zeros((h, w, 3), f32)
    want_albedo[hit] = a["mats10"][a["mat_idx"][prim[hit]], 4:7]
    assert np.array_equal(bits(albedo), bits(want_albedo))
    want_normal = np.zeros((h, w, 3), f32)
    want_normal[hit] = geometric_normals(a["tri9"])[prim[hit]]
    assert np.abs(normal - want_normal).max() <= 2e-7
    assert not normal[~hit].any()
    for flags in (rt.FLAG_BVH8, rt.FLAG_DIAG_SLABS):
        a2, n2, _ = sc.render_aovs(c, w, h, samples_per_axis=1, flags=flags)
        assert np.array_equal(bits(a2), bits(albedo)) and np.array_equal(bits(n2), bits(normal)), flags


@gpu
def test_aov_spheres(rt, golden_scenes, golden_cameras):
    g = load_golden("sphere_cornell.npz")
    a = scene_arrays(golden_scenes, "cornell")
    n = len(a["tri9"])
    mat_idx = np.concatenate([a["mat_idx"], np.array([len(g["mats10"]) - 1], np.int32)])
    sph = [((float(g["spheres4"][0, 0]), float(g["spheres4"][0, 1]), float(g["spheres4"][0, 2])), float(g["spheres4"][0, 3]), n)]
    sc = rt.Scene(a["tri9"], mat_idx, g["mats10"], a["emissive"], spheres=sph, skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    prim, _, _ = sc.trace_primary(c, 128, 128)
    albedo, normal, _ = sc.render_aovs(c, 128, 128, samples_per_axis=1)
    on_sphere = prim == n
    assert on_sphere.sum() > 100
    length = np.linalg.norm(normal[on_sphere].astype(np.float64), axis=-1)
    assert np.abs(length - 1.0).max() <= 1e-6
    assert np.array_equal(bits(albedo[on_sphere]), bits(np.broadcast_to(g["mats10"][-1, 4:7], (int(on_sphere.sum()), 3))))


@gpu
def test_aov_stratified_rays_antialias(rt, golden_scenes, golden_cameras):
    """k = 4: means of 16 hits. Albedos stay inside the materials' range, normals inside the unit ball; where the one-ray buffers see a
    single material around a pixel the mean is that material's colour; along edges some pixels blend two (partial coverage)."""
    sc, a = make_scene(rt, golden_scenes, "cornell")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h = 256, 256
    prim, _, _ = sc.trace_primary(c, w, h)
    albedo, normal, st = sc.render_aovs(c, w, h, samples_per_axis=4)
    assert st["rays"] == w * h * 16
    diffuse = a["mats10"][np.unique(a["mat_idx"]), 4:7]
    if (prim < 0).any():                       # a miss contributes albedo 0
        diffuse = np.concatenate([diffuse, np.zeros((1, 3), f32)])
    assert (albedo >= diffuse.min(0) - 1e-6).all() and (albedo <= diffuse.max(0) + 1e-6).all()
    assert (np.linalg.norm(normal.astype(np.float64), axis=-1) <= 1 + 1e-6).all()
    mat = np.where(prim >= 0, a["mat_idx"][np.maximum(prim, 0)], -1)
    single = neighbourhood_labels(mat, h, w) == 1
    want = np.where((mat >= 0)[..., None], a["mats10"][np.maximum(mat, 0), 4:7], 0.0)
    exact = np.abs(albedo - want).max(-1) <= 1e-6
    frac = float(exact[single].mean())
    print(f"{single.sum()} single-material pixels, {frac * 100:.3f} % of them at that material's albedo")
    assert frac >= 0.999
    nearest = np.abs(albedo.reshape(-1, 1, 3) - diffuse[None]).max(-1).min(-1)
    assert (nearest > 1e-6).sum() > 0, "no pixel is partly covered by two materials"


@gpu
def test_aov_host_device_multi_device_and_stats(rt, golden_scenes, golden_cameras):
    import torch
    sc, a = make_scene(rt, golden_scenes, "cornell")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    w, h, k = 200, 150, 2
    albedo, normal, st = sc.render_aovs(c, w, h, samples_per_axis=k)
    assert st["rays"] == w * h * k * k and st["samples"] == w * h * k * k
    a2, n2, _ = sc.render_aovs(c, w, h, samples_per_axis=k)
    assert np.array_equal(bits(a2), bits(albedo)) and np.array_equal(bits(n2), bits(normal))
    da = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    dn = torch.empty_like(da)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        st_d = sc.render_aovs_device(c, w, h, da.data_ptr(), dn.data_ptr(), samples_per_axis=k, stream_ptr=side.cuda_stream, want_stats=True)
    side.synchronize()
    assert st_d["rays"] == w * h * k * k
    assert np.array_equal(bits(da.cpu().numpy()), bits(albedo)) and np.array_equal(bits(dn.cpu().numpy()), bits(normal))
    only = torch.zeros_like(da)
    sc.render_aovs_device(c, w, h, 0, only.data_ptr(), samples_per_axis=k)
    torch.cuda.synchronize()
    assert np.array_equal(bits(only.cpu().numpy()), bits(normal))
    multi = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], devices=[0, 0])
    ma, mn, _ = multi.render_aovs(c, w, h, samples_per_axis=k)
    assert np.array_equal(bits(ma), bits(albedo)) and np.array_equal(bits(mn), bits(normal))


@gpu
def test_aov_argument_errors(rt, golden_scenes, golden_cameras):
    import torch
    sc, _ = make_scene(rt, golden_scenes, "cornell")
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    buf = torch.empty((16, 16, 3), dtype=torch.float32, device="cuda")
    for k in (0, 17):
        with pytest.raises(rt.B200RTError, match="samples_per_axis"):
            sc.render_aovs(c, 16, 16, samples_per_axis=k)
    with pytest.raises(rt.B200RTError, match="at least one"):
        sc.render_aovs_device(c, 16, 16, 0, 0, samples_per_axis=1)
    with pytest.raises(rt.B200RTError, match="rank/world"):
        sc.render_aovs_device(c, 16, 16, buf.data_ptr(), 0, samples_per_axis=1, rank=0, world=2)
    with pytest.raises(rt.B200RTError):
        sc.render_aovs(c, 0, 16)


# ---- guided denoise ---------------------------------------------------------------------------------------------------------------------
def denoise_raw(rt, img, albedo=None, normal=None, blend=1.0, guided=True):
    """b200rt_denoise_guided (guided=True, NULL guides allowed) or b200rt_denoise straight through the C ABI"""
    L = rt.load_library()
    img = np.ascontiguousarray(img, f32)
    h, w, ch = img.shape
    out = np.empty_like(img)
    fp = rt.binding.fptr
    if guided:
        rt.binding.check(L.b200rt_denoise_guided(fp(img), ch, fp(albedo), fp(normal), w, h, blend, 0, 0.0, fp(out)))
    else:
        rt.binding.check(L.b200rt_denoise(fp(img), ch, w, h, blend, 0, 0.0, fp(out)))
    return out


@gpu
@pytest.mark.parametrize("channels", [3, 4])
def test_guided_denoise_without_guides_is_the_colour_filter(rt, channels):
    rng = np.random.default_rng(11)
    img = (rng.random((61, 97, channels)) * 1.2).astype(f32)
    img[10:40, 20:60, :3] = 0.8
    for blend in (1.0, 0.5, 0.0):
        want = denoise_raw(rt, img, blend=blend, guided=False)
        got = denoise_raw(rt, img, blend=blend)
        assert np.array_equal(bits(got), bits(want)), blend


def checker_case(h=128, w=128, seed=3):
    cell = ((np.arange(h)[:, None] // 4) + (np.arange(w)[None, :] // 4)) % 2
    albedos = np.array([[0.8, 0.5, 0.2], [0.2, 0.4, 0.9]], f32)
    albedo = albedos[cell].astype(f32)
    clean = (albedo * f32(0.6)).astype(f32)
    noisy = (clean * (1.0 + 0.3 * np.random.default_rng(seed).standard_normal((h, w, 3)))).astype(f32)
    normal = np.broadcast_to(np.array([0.0, 0.0, 1.0], f32), (h, w, 3)).copy()
    return clean, noisy, albedo, normal, cell


def rmse(a, b):
    return float(np.sqrt(((a[..., :3].astype(np.float64) - b[..., :3].astype(np.float64)) ** 2).mean()))


@gpu
def test_guided_denoise_keeps_texture_detail(rt):
    """A 4x4-pixel checker of two albedos under constant lighting and 30 % multiplicative noise: the colour-only filter either blurs
    the checker or leaves the noise; with the albedo guide the filter averages within cells and the cell edges stay."""
    clean, noisy, albedo, normal, cell = checker_case()
    colour = rt.OIDN_denoise(noisy)
    guided = rt.OIDN_denoise(noisy, albedo=albedo, normal=normal)
    r_noisy, r_colour, r_guided = rmse(noisy, clean), rmse(colour, clean), rmse(guided, clean)
    print(f"checker rmse: noisy {r_noisy:.5f} colour-only {r_colour:.5f} guided {r_guided:.5f} ratio {r_guided / r_colour:.3f}")
    assert r_guided < 0.7 * r_colour
    # edges: across every vertical cell border the filtered step keeps >= 80 % of the clean step
    left, right = np.s_[:, 3:-1:4], np.s_[:, 4::4]
    step = (clean[right] - clean[left]).astype(np.float64)
    kept = ((guided[right] - guided[left]) * np.sign(step)).mean() / np.abs(step).mean()
    print(f"checker edge contrast kept: {kept:.3f}")
    assert kept >= 0.8


def edge_pixels(albedo1, normal1):
    """pixels whose 3x3 neighbourhood of one-ray feature buffers holds more than one (albedo, normal)"""
    h, w = albedo1.shape[:2]
    key = np.concatenate([albedo1, normal1], -1).reshape(h * w, 6)
    _, label = np.unique(key, axis=0, return_inverse=True)
    return neighbourhood_labels(label.reshape(-1), h, w) > 1


@gpu
def test_guided_denoise_on_rendered_frames(rt, golden_scenes, golden_cameras):
    """4 spp against 1024 spp, guides from render_aovs(k=2): the guided filter is closer to the converged frame than the colour-only
    one on the whole frame, and on Cornell's edge pixels (where the one-ray feature buffers change)."""
    from sycl_ray_tracing_b200 import scenes
    g = load_golden("render_cornell_env.npz")
    sc, _ = make_scene(rt, golden_scenes, "cornell", skysphere=g["env"])
    c = rt.Camera.from_array17(golden_cameras["cornell"])
    c3 = scenes.c3_scene(nu=100, nv=50, sky_w=64, sky_h=32)
    sc3 = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"])
    for name, s, cam, w, h, bounces in (("cornell", sc, c, 256, 256, 5), ("c3small", sc3, c3["camera"], 320, 180, 8)):
        noisy, _ = s.render(cam, w, h, 4, bounces)
        ref, _ = s.render(cam, w, h, 1024, bounces)
        noisy = np.ascontiguousarray(noisy[..., :3])
        albedo, normal, _ = s.render_aovs(cam, w, h, samples_per_axis=2)
        colour = rt.OIDN_denoise(noisy)
        guided = rt.OIDN_denoise(noisy, albedo=albedo, normal=normal)
        r = dict(noisy=rmse(noisy, ref), colour=rmse(colour, ref), guided=rmse(guided, ref))
        print(name, "frame rmse", r, f"guided / colour {r['guided'] / r['colour']:.3f}")
        assert r["guided"] < r["colour"], name
        if name == "cornell":
            a1, n1, _ = s.render_aovs(cam, w, h, samples_per_axis=1)
            e = edge_pixels(a1, n1)
            re = dict(noisy=rmse(noisy[e], ref[e]), colour=rmse(colour[e], ref[e]), guided=rmse(guided[e], ref[e]))
            print(name, f"{int(e.sum())} edge pixels rmse", re, f"guided / colour {re['guided'] / re['colour']:.3f}")
            assert re["guided"] < re["colour"]


# ---- OIDN entry points ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_oidn_dropin_passes_albedo_and_normal(rt, tmp_path):
    import subprocess
    libdir = os.path.join(ROOT, "sycl-ray-tracing_b200")
    so = tmp_path / "libb200rt_oidn.so"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"),
                    os.path.join(libdir, "host", "dropin", "b200rt_oidn.c"), "-o", str(so), "-L", libdir, "-lb200rt", f"-Wl,-rpath,{libdir}"],
                   check=True)
    O = C.CDLL(str(so))
    VP, SZ = C.c_void_p, C.c_size_t
    O.oidnNewDevice.restype = VP
    O.oidnNewDevice.argtypes = [C.c_int]
    O.oidnCommitDevice.argtypes = [VP]
    O.oidnNewBuffer.restype = VP
    O.oidnNewBuffer.argtypes = [VP, SZ]
    O.oidnGetBufferData.restype = VP
    O.oidnGetBufferData.argtypes = [VP]
    O.oidnNewFilter.restype = VP
    O.oidnNewFilter.argtypes = [VP, C.c_char_p]
    O.oidnSetFilterImage.argtypes = [VP, C.c_char_p, VP, C.c_int, SZ, SZ, SZ, SZ, SZ]
    O.oidnSetFilterBool.argtypes = [VP, C.c_char_p, C.c_int]
    O.oidnCommitFilter.argtypes = [VP]
    O.oidnExecuteFilter.argtypes = [VP]
    O.oidnGetDeviceError.argtypes = [VP, C.POINTER(C.c_char_p)]
    O.oidnReleaseBuffer.argtypes = [VP]
    O.oidnReleaseFilter.argtypes = [VP]
    O.oidnReleaseDevice.argtypes = [VP]
    _, noisy, albedo, normal, _ = checker_case(64, 96)
    h, w = noisy.shape[:2]
    nbytes = noisy.nbytes
    FLOAT3 = 3                                   # OIDN_FORMAT_FLOAT3

    def run(images):
        dev = O.oidnNewDevice(0)
        O.oidnCommitDevice(dev)
        bufs = {}
        for name, arr in images.items():
            b = O.oidnNewBuffer(dev, nbytes)
            C.memmove(O.oidnGetBufferData(b), arr.ctypes.data, nbytes)
            bufs[name] = b
        flt = O.oidnNewFilter(dev, b"RT")
        for name, b in bufs.items():
            O.oidnSetFilterImage(flt, name.encode(), b, FLOAT3, w, h, 0, 0, 0)
        O.oidnSetFilterImage(flt, b"output", bufs["color"], FLOAT3, w, h, 0, 0, 0)      # in place, as utils.cpp:158-159
        O.oidnSetFilterBool(flt, b"hdr", 0)
        O.oidnSetFilterBool(flt, b"cleanAux", 1)
        O.oidnCommitFilter(flt)
        O.oidnExecuteFilter(flt)
        msg = C.c_char_p()
        assert O.oidnGetDeviceError(dev, C.byref(msg)) == 0, msg.value
        out = np.empty_like(noisy)
        C.memmove(out.ctypes.data, O.oidnGetBufferData(bufs["color"]), nbytes)
        O.oidnReleaseFilter(flt)
        for b in bufs.values():
            O.oidnReleaseBuffer(b)
        O.oidnReleaseDevice(dev)
        return out

    assert np.array_equal(bits(run({"color": noisy})), bits(denoise_raw(rt, noisy, guided=False)))
    want = denoise_raw(rt, noisy, albedo, normal)
    assert not np.array_equal(bits(want), bits(denoise_raw(rt, noisy, guided=False)))
    assert np.array_equal(bits(run({"color": noisy, "albedo": albedo, "normal": normal})), bits(want))


# ---- without a GPU ---------------------------------------------------------------------------------------------------------------------------
NO_GPU_GUIDED = """
import numpy as np
import pytest
import sycl_ray_tracing_b200 as rt
img = np.zeros((8, 8, 3), np.float32)
with pytest.raises(rt.B200RTError, match="no CUDA device"):
    rt.OIDN_denoise(img, albedo=img, normal=img)
"""


def test_guided_denoise_fails_loudly_without_a_gpu():
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join(p for p in (ROOT, os.environ.get("PYTHONPATH")) if p))
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", NO_GPU_GUIDED], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_guided_denoise_rejects_a_null_image(rt):
    L = rt.load_library()
    out = np.empty((4, 4, 3), f32)
    assert L.b200rt_denoise_guided(None, 3, None, None, 4, 4, 1.0, 0, 0.0, rt.binding.fptr(out)) == 1       # B200RT_ERR_ARG
    assert "bad denoise arguments" in L.b200rt_last_error().decode()


def test_guide_shapes_are_checked(rt):
    img = np.zeros((8, 10, 3), np.float32)
    for kw in (dict(albedo=np.zeros((10, 8, 3), np.float32)), dict(normal=np.zeros((8, 10, 4), np.float32)),
               dict(albedo=img, normal=np.zeros((8, 10), np.float32))):
        with pytest.raises(ValueError, match="guide has shape"):
            rt.OIDN_denoise(img, **kw)
