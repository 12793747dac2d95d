"""The output stage against plain restatements: the à-trous denoiser (csrc/denoise.cu, b200rt_denoise_guided) against a float64 numpy
reference of the documented filter, its non-finite policy, k_aov's k x k feature buffers against the port's camera rays and the
library's own closest hits, and the OIDN drop-in's refusal of image layouts it cannot read.

The reference restates the filter from its documentation, not from the library:
* passes i = 0 .. iterations - 1 with holes of 1 << i pixels and sigma_i = sigma / 2^i; a tap's weight is the 5x5 B3 spline weight
  (1/16, 1/4, 3/8, 1/4, 1/16 per axis) times exp(-|c_q - c_p|^2 / sigma_i^2 * noise_scale), with (2 sigma_i)^2 in place of sigma_i^2
  when guides are given; samples clamp to the image's edge;
* pass 0 only: noise_scale = 1 / (1 + 16 max(E[l^2] - E[l]^2, 0)) over the clamped 3x3 neighbourhood, l = 0.2126 r + 0.7152 g + 0.0722 b
  (1 in every later pass);
* guides: albedo weighs exp(-|a_q - a_p|^2 / 0.1^2); normal weighs max(0, n_p . n_q)^128 of the normalised normals, and a zero
  normal (zero float32 squared length) matches only a zero normal;
* each pass copies the input's alpha; the blend writes blend * denoised + (1 - blend) * noisy and alpha 1;
* host defaults: iterations <= 0 -> 5, > 8 -> 8; sigma <= 0 or NaN -> 0.45;
* non-finite pixels (NaN or +-Inf in R, G or B) are missing: no tap, left out of the 3x3 statistic (divided by the number of finite
  neighbours; none finite -> noise_scale 1), filtered without the colour term as a centre, and the blend takes the denoised value.

The GPU tests are marked gpu; the reference's own checks and the drop-in's format checks run anywhere."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, brute_force_closest, load_golden, scene_arrays

gpu = pytest.mark.gpu
f32, f64 = np.float32, np.float64
B3 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
LUMA = np.array([0.2126, 0.7152, 0.0722])
SIGMA_ALBEDO = 0.1
NORMAL_EXPONENT = 128
GUIDED_COLOUR_RELAX = 2.0

# max |GPU - reference| over a case family, for images whose values are at most 1 (the HDR case and the renders are divided by their
# peak). The bounds allow for float32 arithmetic and __expf / __powf (whose log2 error __powf(x, 128) multiplies by 128); they are
# not yet set from errors measured on a B200 — the tests print the errors they see. Each stays at least 20x below the smallest effect
# of a one-constant change of the filter in the numpy reference (sigma_albedo 0.1 -> 0.12 on the albedo-guided case moves the output
# by 0.11).
TOL_COLOUR = 5e-5
TOL_GUIDED = 5e-4


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


# ---- the reference ----------------------------------------------------------------------------------------------------------------------
def host_defaults(iterations, sigma):
    it = 5 if iterations <= 0 else min(iterations, 8)
    sigma = f32(sigma)
    return it, float(sigma if sigma > 0 else f32(0.45))


def clamped(a, r):
    """a padded by r pixels on each side with its edge values: view [r + dy : r + dy + h, r + dx : r + dx + w] of it is
    a[clamp(y + dy), clamp(x + dx)] for every pixel (clamp-to-edge sampling), however wide r is"""
    pad = ((r, r), (r, r)) + ((0, 0),) * (a.ndim - 2)
    padded = np.pad(a, pad, mode="edge")
    h, w = a.shape[:2]
    return lambda dy, dx: padded[r + dy: r + dy + h, r + dx: r + dx + w]


def unit_or_zero(normal):
    """(normalised normals in float64, zero mask); "zero" is decided on the float32 squared length, as the kernel does"""
    n = np.asarray(normal, f32)
    l2 = ((n[..., 0] * n[..., 0] + n[..., 1] * n[..., 1]).astype(f32) + n[..., 2] * n[..., 2]).astype(f32)
    zero = l2 == 0
    n64 = n.astype(f64)
    length = np.sqrt((n64 ** 2).sum(-1))
    unit = np.where(zero[..., None], 0.0, n64 / np.where(zero, 1.0, length)[..., None])
    return unit, zero


def atrous_pass(img, step, inv_sigma2, local_noise, albedo, normal):
    rgb = img[..., :3]
    ok = np.isfinite(rgb).all(-1)
    noise_scale = 1.0
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        if local_noise:
            lum_at, ok_at = clamped(np.where(ok, rgb @ LUMA, 0.0), 1), clamped(ok, 1)
            s, s2, n = np.zeros(ok.shape), np.zeros(ok.shape), np.zeros(ok.shape)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    lum = lum_at(dy, dx)
                    s += lum
                    s2 += lum * lum
                    n += ok_at(dy, dx)
            var = np.maximum(s2 / n - (s / n) ** 2, 0.0)
            noise_scale = np.where(n > 0, 1.0 / (1.0 + 16.0 * var), 1.0)
        r = 2 * step
        rgb_at, ok_at = clamped(np.where(ok[..., None], rgb, 0.0), r), clamped(ok, r)
        if albedo is not None:
            albedo_at = clamped(albedo, r)
        if normal is not None:
            unit, zero = normal
            unit_at, zero_at = clamped(unit, r), clamped(zero, r)
        acc, wsum = np.zeros(rgb.shape), np.zeros(ok.shape)
        for j in range(5):
            for i in range(5):
                dy, dx = (j - 2) * step, (i - 2) * step
                q, q_ok = rgb_at(dy, dx), ok_at(dy, dx)
                d2 = ((q - rgb) ** 2).sum(-1)
                wgt = B3[i] * B3[j] * np.where(ok, np.exp(-d2 * inv_sigma2 * noise_scale), 1.0)
                if albedo is not None:
                    wgt *= np.exp(-((albedo_at(dy, dx) - albedo) ** 2).sum(-1) / SIGMA_ALBEDO ** 2)
                if normal is not None:
                    q_zero = zero_at(dy, dx)
                    cos = np.maximum(0.0, (unit_at(dy, dx) * unit).sum(-1))
                    wgt *= np.where(zero | q_zero, (zero == q_zero).astype(f64), cos ** NORMAL_EXPONENT)
                wgt = np.where(q_ok, wgt, 0.0)
                acc += wgt[..., None] * q
                wsum += wgt
        out = img.copy()
        out[..., :3] = acc / wsum[..., None]
    return out


def denoise_reference(img, iterations=0, sigma=0.0, blend=1.0, albedo=None, normal=None):
    """float64 restatement of b200rt_denoise_guided (the module docstring lists what it restates)"""
    it, sigma = host_defaults(iterations, sigma)
    noisy = np.asarray(img, f32).astype(f64)
    guides = dict(albedo=None if albedo is None else np.asarray(albedo, f32).astype(f64),
                  normal=None if normal is None else unit_or_zero(normal))
    guided = albedo is not None or normal is not None
    cur = noisy
    for i in range(it):
        s = sigma / 2 ** i * (GUIDED_COLOUR_RELAX if guided else 1.0)
        cur = atrous_pass(cur, 1 << i, 1.0 / (s * s), i == 0, **guides)
    b = float(f32(blend))
    keep = float(f32(1.0) - f32(blend))
    out = noisy.copy()
    with np.errstate(invalid="ignore", over="ignore"):
        out[..., :3] = np.where(np.isfinite(noisy[..., :3]).all(-1)[..., None], b * cur[..., :3] + keep * noisy[..., :3], cur[..., :3])
    if out.shape[-1] == 4:
        out[..., 3] = 1.0
    return out


# ---- the library ------------------------------------------------------------------------------------------------------------------------
def denoise_gpu(rt, img, iterations=0, sigma=0.0, blend=1.0, albedo=None, normal=None, in_place=False):
    """b200rt_denoise_guided straight through the C ABI (NULL guides: the colour-only filter)"""
    L = rt.load_library()
    img = np.array(img, f32, order="C")
    h, w, ch = img.shape
    out = img if in_place else np.empty_like(img)
    g = [None if a is None else np.ascontiguousarray(a, f32) for a in (albedo, normal)]
    fp = rt.binding.fptr
    rt.binding.check(L.b200rt_denoise_guided(fp(img), ch, fp(g[0]), fp(g[1]), w, h, float(blend), int(iterations), float(sigma), fp(out)))
    return out


def max_err(got, want, scale=1.0):
    got, want = np.asarray(got, f64), np.asarray(want, f64)
    assert np.array_equal(np.isfinite(got), np.isfinite(want)), f"{(np.isfinite(got) != np.isfinite(want)).sum()} finiteness mismatches"
    fin = np.isfinite(want)
    return float(np.abs(got[fin] - want[fin]).max() / scale) if fin.any() else 0.0


def check(rt, img, tol, scale=1.0, **kw):
    got = denoise_gpu(rt, img, **kw)
    want = denoise_reference(img, **{k: v for k, v in kw.items() if k != "in_place"})
    err = max_err(got, want, scale)
    assert err <= tol, f"max |gpu - reference| = {err:.3g} > {tol:.3g}"
    return err, got


# ---- inputs --------------------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1), (1, 57), (57, 1), (9, 31), (8, 33), (61, 97), (360, 640), (1080, 1920)]     # (h, w)


def noise_image(h, w, channels=3, seed=0):
    rng = np.random.default_rng(seed)
    img = rng.random((h, w, channels)).astype(f32)
    if channels == 4:
        img[..., 3] = rng.random((h, w)) * 3.0 - 1.0          # random alpha, copied through every pass
    return img


def steps_image(h=61, w=97, seed=1):
    """piecewise constant: four flat blocks with steps between them, plus a little noise"""
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w, 3), f32)
    img[:, : w // 3] = (0.1, 0.2, 0.3)
    img[:, w // 3:] = (0.9, 0.5, 0.1)
    img[h // 2:, w // 2:] = (0.05, 0.8, 0.6)
    img[h // 4: h // 4 + 5, :] = (1.0, 1.0, 1.0)
    return (img + 0.02 * rng.standard_normal(img.shape)).astype(f32)


def hdr_image(h=61, w=97, seed=2):
    """values up to ~50: most colour weights underflow to 0"""
    rng = np.random.default_rng(seed)
    return (np.exp(rng.random((h, w, 3)) * np.log(50.0)) * (rng.random((h, w, 1)) < 0.7)).astype(f32)


def c3_frame(rt):
    from sycl_ray_tracing_b200 import scenes
    c3 = scenes.c3_scene(nu=100, nv=50, sky_w=64, sky_h=32)
    sc = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"])
    img, _ = sc.render(c3["camera"], 320, 180, 4, 8)
    return img


def synthetic_guides(h=61, w=97, seed=4):
    """albedo: a 4x4-pixel checker of two colours with +-0.05 noise (differences where exp(-d^2 / 0.01) is neither 0 nor 1); normals:
    unit normals jittered around +z (cosines near 0.98, where ^128 matters), unnormalised means of length 0.3 .. 1 (what k_aov gives on
    edges), an antiparallel block, an exact-zero block (misses) and a tiny (1e-30, a miss in float32) block"""
    rng = np.random.default_rng(seed)
    cell = ((np.arange(h)[:, None] // 4) + (np.arange(w)[None, :] // 4)) % 2
    albedo = (np.array([[0.8, 0.5, 0.2], [0.2, 0.4, 0.9]])[cell] + 0.05 * rng.standard_normal((h, w, 3))).astype(f32)
    n = np.array([0.0, 0.0, 1.0]) + 0.12 * rng.standard_normal((h, w, 3))
    n /= np.linalg.norm(n, axis=-1, keepdims=True)
    n[:, w // 2: w // 2 + 12] *= rng.uniform(0.3, 1.0, (h, 12, 1))
    n[h // 2: h // 2 + 10, : w // 4] = (0.0, 0.0, -1.0)
    n[: h // 4, w // 4: w // 2] = 0.0
    n[h - 8:, w - 20:] = 1e-30
    return albedo, n.astype(f32)


def finite_cases():
    """(name, image, keyword arguments) of the finite colour-only and synthetic-guided cases: their outputs are fixed bit for bit"""
    for h, w in SHAPES:
        for ch in (3, 4):
            yield f"noise_{h}x{w}x{ch}", noise_image(h, w, ch), {}
    base = noise_image(61, 97, 4, seed=5)
    for it in (0, 1, 2, 5, 8, 12):
        for sigma in (0.1, 0.45, 2.0, 0.0, -1.0, float("nan")):
            for blend in (0.0, 0.37, 1.0):
                yield f"schedule_{it}_{sigma}_{blend}", base, dict(iterations=it, sigma=sigma, blend=blend)
    yield "steps", steps_image(), {}
    yield "hdr", hdr_image(), {}
    albedo, normal = synthetic_guides()
    img = noise_image(61, 97, 3, seed=6)
    for name, g in (("albedo", dict(albedo=albedo)), ("normal", dict(normal=normal)), ("both", dict(albedo=albedo, normal=normal))):
        yield f"guided_{name}", img, g


# ---- the reference on its own (no GPU) -------------------------------------------------------------------------------------------------
def test_reference_keeps_a_constant_image():
    img = np.full((9, 31, 4), 0.37, f32)
    img[..., 3] = 0.5
    out = denoise_reference(img, blend=0.37)
    assert np.allclose(out[..., :3], 0.37, atol=1e-7, rtol=0) and (out[..., 3] == 1.0).all()       # f32(0.37) + f32(0.63) != 1
    assert np.abs(denoise_reference(img, iterations=8)[..., :3] - f64(f32(0.37))).max() < 1e-15


def test_reference_fills_the_golden_mis_frame():
    """The reference's MIS + environment frame holds 3 NaN pixels (reference quirk 6); filtered as missing data they are filled from
    their finite neighbours and no other pixel changes finiteness."""
    img = load_golden("render_mis_env.npz")["image"]
    assert (~np.isfinite(img[..., :3]).all(-1)).sum() == 3
    out = denoise_reference(img)
    assert np.isfinite(out).all()
    assert np.isfinite(denoise_reference(img, albedo=np.zeros(img.shape[:2] + (3,), f32))).all()


def test_reference_fills_a_single_nan():
    """one NaN tap, if it counted, would reach 2 * (1 + 2 + 4 + 8 + 16) = 62 pixels in each direction: the reference fills that pixel
    from its neighbours' range and is finite everywhere"""
    img = steps_image()
    img[30, 40, 1] = np.nan
    out = denoise_reference(img, blend=0.0)
    assert np.isfinite(out).all()
    lo, hi = np.nanmin(img[26:35, 36:45], axis=(0, 1)), np.nanmax(img[26:35, 36:45], axis=(0, 1))
    assert (out[30, 40] >= lo - 0.2).all() and (out[30, 40] <= hi + 0.2).all()


# ---- colour-only filter ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("channels", [3, 4])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
def test_colour_filter_matches_reference(rt, shape, channels):
    """every shape's small or odd edge (1x1, 1 x 57, one pixel past a 32x8 block) clamps the wide holes; 4 channels carry a random
    alpha through the passes; in == out gives the same bits as separate buffers"""
    img = noise_image(*shape, channels)
    err, got = check(rt, img, TOL_COLOUR, blend=0.37)
    print(f"{shape} x {channels}: max err {err:.3g}")
    assert np.array_equal(bits(denoise_gpu(rt, img, blend=0.37, in_place=True)), bits(got))


@gpu
@pytest.mark.parametrize("iterations", [0, 1, 2, 5, 8, 12])
@pytest.mark.parametrize("sigma", [0.1, 0.45, 2.0, 0.0, -1.0, float("nan")])
def test_pass_schedule_and_defaults_match_reference(rt, iterations, sigma):
    """sigma_i = sigma / 2^i, holes 1 << i, the noise scale in pass 0 only, iterations <= 0 -> 5 and > 8 -> 8, sigma <= 0 or NaN
    -> 0.45, for blends 0, 0.37 and 1 on a 97x61 RGBA noise image"""
    img = noise_image(61, 97, 4, seed=5)
    worst = 0.0
    for blend in (0.0, 0.37, 1.0):
        err, _ = check(rt, img, TOL_COLOUR, iterations=iterations, sigma=sigma, blend=blend)
        worst = max(worst, err)
    print(f"iterations {iterations} sigma {sigma}: max err {worst:.3g}")


@gpu
def test_colour_filter_on_steps_hdr_and_a_render(rt):
    err = check(rt, steps_image(), TOL_COLOUR)[0]
    hdr = hdr_image()
    err_hdr = check(rt, hdr, TOL_COLOUR, scale=float(hdr.max()))[0]
    frame = c3_frame(rt)
    err_c3 = check(rt, frame, TOL_COLOUR, scale=max(1.0, float(frame[..., :3].max())))[0]
    print(f"steps {err:.3g}, hdr (over its peak) {err_hdr:.3g}, 4-spp C3 {err_c3:.3g}")


# ---- guided filter ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("guides", ["albedo", "normal", "both"])
def test_guided_filter_matches_reference(rt, guides):
    albedo, normal = synthetic_guides()
    img = noise_image(61, 97, 3, seed=6)
    kw = dict(albedo=albedo if guides != "normal" else None, normal=normal if guides != "albedo" else None)
    err = max(check(rt, img, TOL_GUIDED, blend=blend, **kw)[0] for blend in (1.0, 0.37))
    err4 = check(rt, noise_image(61, 97, 4, seed=7), TOL_GUIDED, iterations=3, sigma=0.3, **kw)[0]
    print(f"guided by {guides}: max err {err:.3g}, RGBA {err4:.3g}")


@gpu
def test_guided_filter_with_rendered_guides(rt, golden_scenes, golden_cameras):
    """Cornell at 4 spp with render_aovs(k=2) albedo and normal: the guides of a real frame (misses, partly covered edge pixels)"""
    g = load_golden("render_cornell_env.npz")
    a = scene_arrays(golden_scenes, "cornell")
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"], skysphere=g["env"])
    cam = rt.Camera.from_array17(golden_cameras["cornell"])
    noisy, _ = sc.render(cam, 128, 128, 4, 5)
    noisy = np.ascontiguousarray(noisy[..., :3])
    albedo, normal, _ = sc.render_aovs(cam, 128, 128, samples_per_axis=2)
    scale = max(1.0, float(noisy.max()))
    errs = [check(rt, noisy, TOL_GUIDED, scale=scale, **kw)[0]
            for kw in (dict(albedo=albedo), dict(normal=normal), dict(albedo=albedo, normal=normal))]
    print(f"Cornell with rendered guides: max err {max(errs):.3g}")


# ---- non-finite pixels -------------------------------------------------------------------------------------------------------------------
@gpu
def test_golden_mis_frame_is_denoised_finite(rt):
    """The MIS + environment frame's 3 NaN pixels (29, 49), (32, 51), (54, 62) must not spread through the filter; each is filled
    from its finite neighbours, as the reference does."""
    img = load_golden("render_mis_env.npz")["image"]
    for blend in (1.0, 0.5):
        got = denoise_gpu(rt, img, blend=blend)
        assert np.isfinite(got).all(), f"{(~np.isfinite(got[..., :3]).all(-1)).sum()} of 4096 pixels are not finite"
        err = max_err(got, denoise_reference(img, blend=blend))
        assert err <= TOL_COLOUR, err


def nan_cases():
    base = steps_image()
    cases = {}
    one = base.copy(); one[30, 40, 1] = np.nan; cases["one_nan"] = one
    inf = base.copy(); inf[20, 70, 0] = np.inf; inf[40, 10, 2] = -np.inf; cases["inf"] = inf
    block = base.copy(); block[20:30, 30:38] = np.nan; cases["nan_block"] = block
    corner = base.copy(); corner[0, 0] = np.nan; corner[-1, -1, 2] = np.nan; cases["corner"] = corner
    return cases


@gpu
@pytest.mark.parametrize("name", ["one_nan", "inf", "nan_block", "corner"])
def test_non_finite_pixels_are_missing_data(rt, name):
    """a missing pixel gives no tap, is left out of the 3x3 statistic and is filled from its finite neighbours, for colour-only and
    guided filtering and every blend; a block wider than the 5x5 footprint is filled by the later, wider passes"""
    img = nan_cases()[name]
    albedo, normal = synthetic_guides()
    for kw in (dict(blend=1.0), dict(blend=0.0), dict(blend=0.37, iterations=2), dict(albedo=albedo, normal=normal, blend=0.37)):
        tol = TOL_GUIDED if "albedo" in kw else TOL_COLOUR
        got = check(rt, img, tol, **kw)[1]
        assert np.isfinite(got).all(), kw


@gpu
def test_nan_in_alpha_only_is_not_missing(rt):
    img = noise_image(61, 97, 4, seed=8)
    img[30, 40, 3] = np.nan
    got = denoise_gpu(rt, img, iterations=2)
    assert np.array_equal(bits(got[..., :3]), bits(denoise_gpu(rt, np.nan_to_num(img), iterations=2)[..., :3]))
    assert (got[..., 3] == 1.0).all()
    assert max_err(got, denoise_reference(img, iterations=2)) <= TOL_COLOUR


@gpu
def test_all_nan_image_stays_nan(rt):
    img = np.full((19, 45, 4), np.nan, f32)
    got = denoise_gpu(rt, img, blend=0.37)
    assert np.isnan(got[..., :3]).all() and (got[..., 3] == 1.0).all()


# ---- k_aov at k > 1 ------------------------------------------------------------------------------------------------------------------------
CAM_OF = {"cornell": "cornell", "mis": "mis", "area": "cornell"}


def geometric_normals(tri9):
    """normalize(cross(b - a, c - a)) in float32, in the operation order of triangle.h / vec.h (as in test_gpu_aov.py)"""
    t = np.asarray(tri9, f32).reshape(-1, 9)
    u = (t[:, 3:6] - t[:, 0:3]).astype(f32)
    v = (t[:, 6:9] - t[:, 0:3]).astype(f32)
    c = np.stack([u[:, 1] * v[:, 2] - u[:, 2] * v[:, 1], u[:, 2] * v[:, 0] - u[:, 0] * v[:, 2], u[:, 0] * v[:, 1] - u[:, 1] * v[:, 0]], 1).astype(f32)
    length = np.sqrt((c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]).astype(f32) + c[:, 2] * c[:, 2]).astype(f32)
    return ((f32(1.0) / length)[:, None] * c).astype(f32)


@gpu
@pytest.mark.parametrize("key", ["cornell", "mis", "area"])
@pytest.mark.parametrize("size", [(37, 23), (256, 256)], ids=["37x23", "256x256"])
@pytest.mark.parametrize("k", [2, 3, 5, 16])
def test_aov_grid_matches_restatement(rt, golden_scenes, golden_cameras, key, size, k):
    """Pixel (x, y) traces the sub-pixel positions x + ((i + 0.5) / k - 0.5), y + ((j + 0.5) / k - 0.5) in float32, j outer and i inner;
    the port's camera rays through them, closest hits from Scene.trace_rays. The albedo is the sum of the hit materials' diffuse
    colours in that order over float32(k * k), bit for bit; the normal the same sum of the hits' normals (bit for bit against
    trace_rays' hit normals, within 3e-7 of the float32 geometric normals)."""
    from oracle.oracle import PortOracle
    w, h = size
    a = scene_arrays(golden_scenes, key)
    sc = rt.Scene(a["tri9"], a["mat_idx"], a["mats10"], a["emissive"])
    cam17 = np.asarray(golden_cameras[CAM_OF[key]], f32)
    albedo, normal, _ = sc.render_aovs(rt.Camera.from_array17(cam17), w, h, samples_per_axis=k)
    port = PortOracle()
    xs, ys = np.meshgrid(np.arange(w, dtype=f32), np.arange(h, dtype=f32))
    off = ((np.arange(k, dtype=f32) + f32(0.5)) / f32(k) - f32(0.5)).astype(f32)
    geo = geometric_normals(a["tri9"])
    want_a = np.zeros((h, w, 3), f32)
    want_n = np.zeros((h, w, 3), f32)
    want_g = np.zeros((h, w, 3), f32)
    for j in range(k):
        fx = (xs[..., None] + off[None, None, :]).astype(f32)                       # (h, w, k): i is the last axis
        fy = np.broadcast_to((ys + off[j]).astype(f32)[..., None], fx.shape)
        rays = port.camera_rays(cam17, w, h, np.stack([fx, fy], -1).reshape(-1, 2))
        prim, _, extra = sc.trace_rays(rays)
        if j == 0 and w * h <= 1024 and k <= 3:
            bprim, _ = brute_force_closest(a["tri9"], rays)
            assert np.array_equal(prim, bprim)
        prim, extra = prim.reshape(h, w, k), extra.reshape(h, w, k, 8)
        hit = (prim >= 0)[..., None]
        alb = np.where(hit, a["mats10"][a["mat_idx"][np.maximum(prim, 0)], 4:7], f32(0)).astype(f32)
        gn = np.where(hit, geo[np.maximum(prim, 0)], f32(0)).astype(f32)
        for i in range(k):
            want_a = (want_a + alb[:, :, i]).astype(f32)
            want_n = (want_n + extra[:, :, i, 3:6]).astype(f32)
            want_g = (want_g + gn[:, :, i]).astype(f32)
    rays_n = f32(k * k)
    want_a, want_n, want_g = (want_a / rays_n).astype(f32), (want_n / rays_n).astype(f32), (want_g / rays_n).astype(f32)
    assert np.array_equal(bits(albedo), bits(want_a)), f"{(bits(albedo) != bits(want_a)).any(-1).sum()} pixels differ"
    assert np.array_equal(bits(normal), bits(want_n)), f"{(bits(normal) != bits(want_n)).any(-1).sum()} pixels differ"
    assert np.abs(normal - want_g).max() <= 3e-7


# ---- the OIDN drop-in's image layouts (no GPU: refused before any CUDA call) ----------------------------------------------------------------
def load_dropin(tmp_path):
    libdir = os.path.join(ROOT, "sycl-ray-tracing_b200")
    so = tmp_path / "libb200rt_oidn.so"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"),
                    os.path.join(libdir, "host", "dropin", "b200rt_oidn.c"), "-o", str(so), "-L", libdir, "-lb200rt", f"-Wl,-rpath,{libdir}"],
                   check=True)
    O = C.CDLL(str(so))
    VP, SZ = C.c_void_p, C.c_size_t
    for name, res, args in (("oidnNewDevice", VP, [C.c_int]), ("oidnNewBuffer", VP, [VP, SZ]), ("oidnNewFilter", VP, [VP, C.c_char_p]),
                            ("oidnSetFilterImage", None, [VP, C.c_char_p, VP, C.c_int, SZ, SZ, SZ, SZ, SZ]),
                            ("oidnExecuteFilter", None, [VP]), ("oidnGetDeviceError", C.c_int, [VP, C.POINTER(C.c_char_p)]),
                            ("oidnReleaseBuffer", None, [VP]), ("oidnReleaseFilter", None, [VP])):
        fn = getattr(O, name)
        fn.restype, fn.argtypes = res, args
    return O


def test_oidn_dropin_refuses_image_layouts_it_would_misread(rt, tmp_path):
    """Only packed float3 is read: another format (FLOAT4, HALF3), a byte offset, or a pixel / row stride other than packed is a
    device error, and the filter then refuses to run (no CUDA call, so this holds without a GPU). Packed strides given explicitly, or
    as 0 (the reference's calls), are accepted."""
    O = load_dropin(tmp_path)
    w, h = 9, 5
    FLOAT3, FLOAT4, HALF3 = 3, 4, 0x103
    dev = O.oidnNewDevice(0)
    buf = O.oidnNewBuffer(dev, w * h * 16)

    def error():
        msg = C.c_char_p()
        return O.oidnGetDeviceError(dev, C.byref(msg)), (msg.value or b"").decode()

    assert error()[0] == 0
    for fmt, off, ps, rs in ((FLOAT3, 0, 0, 0), (FLOAT3, 0, 12, 12 * w), (FLOAT3, 0, 12, 0), (FLOAT3, 0, 0, 12 * w)):
        flt = O.oidnNewFilter(dev, b"RT")
        for name in (b"color", b"output", b"albedo", b"normal"):
            O.oidnSetFilterImage(flt, name, buf, fmt, w, h, off, ps, rs)
        assert error() == (0, ""), (fmt, off, ps, rs)
        O.oidnReleaseFilter(flt)
    for fmt, off, ps, rs, what in ((FLOAT4, 0, 0, 0, "format"), (HALF3, 0, 0, 0, "format"), (FLOAT3, 12, 0, 0, "offset"),
                                   (FLOAT3, 0, 16, 0, "pixel stride"), (FLOAT3, 0, 0, 12 * w + 4, "row stride"),
                                   (FLOAT3, 0, 12, 16 * w, "row stride")):
        for bad_name in (b"color", b"normal"):
            flt = O.oidnNewFilter(dev, b"RT")
            for name in (b"color", b"output"):
                O.oidnSetFilterImage(flt, name, buf, FLOAT3, w, h, 0, 0, 0)
            O.oidnSetFilterImage(flt, bad_name, buf, fmt, w, h, off, ps, rs)
            code, msg = error()
            assert code != 0 and what in msg, (fmt, off, ps, rs, msg)
            O.oidnExecuteFilter(flt)
            code, msg = error()
            assert code != 0 and what in msg, ("execute", fmt, off, ps, rs, msg)
            O.oidnReleaseFilter(flt)
    O.oidnReleaseBuffer(buf)
