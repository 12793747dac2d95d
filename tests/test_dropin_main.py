"""-m gpu: the reference's UNMODIFIED source/main.cpp, linked against the drop-in RenderKernel
(sycl-ray-tracing_b200/host/dropin, built in the build container where /root/reference exists; the binary travels with
the repo snapshot), renders an OBJ + MTL + HDR from disk on the GPU, denoises on the GPU and writes its four PNGs. The PNG must match a render
of the same scene through the Python mirror."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

BIN = os.path.join(ROOT, "sycl-ray-tracing_b200", "host", "dropin", "_build", "SYCL_RayTracing_b200")


def write_obj(path, tri9, mat_idx, mats10):
    names = [f"m{i}" for i in range(len(mats10))]
    with open(path + ".mtl", "w") as f:
        for i in range(1, len(mats10)):            # slot 0 is parse_obj's built-in default material (utils.cpp:75)
            m = mats10[i]
            f.write(f"newmtl {names[i]}\nKe {m[0]:.9g} {m[1]:.9g} {m[2]:.9g}\nKd {m[4]:.9g} {m[5]:.9g} {m[6]:.9g}\n"
                    f"Pm {m[8]:.9g}\nPr {m[9]:.9g}\nillum 2\n\n")
    with open(path + ".obj", "w") as f:
        f.write(f"mtllib {os.path.basename(path)}.mtl\n")
        for t in tri9:
            for v in range(3):
                f.write(f"v {t[3 * v]:.9g} {t[3 * v + 1]:.9g} {t[3 * v + 2]:.9g}\n")
        cur = -1
        for i in range(len(tri9)):
            if mat_idx[i] != cur:
                cur = int(mat_idx[i])
                f.write(f"usemtl {names[cur]}\n")
            f.write(f"f {3 * i + 1} {3 * i + 2} {3 * i + 3}\n")


def write_hdr_and_decode(path, env_rgb):
    """Flat (non-RLE) Radiance RGBE; returns the float image exactly as stb_image decodes it and
    Utils::read_image_float stores it (vertical flip on load, alpha 0; utils.cpp:100-124)."""
    h, w, _ = env_rgb.shape
    m = env_rgb.max(axis=-1)
    mant, ex = np.frexp(m.astype(np.float64))
    scale = np.where(m > 1e-32, mant * 256.0 / np.maximum(m, 1e-38), 0.0)
    rgbe = np.zeros((h, w, 4), np.uint8)
    rgbe[..., :3] = np.clip(env_rgb * scale[..., None], 0, 255).astype(np.uint8)
    rgbe[..., 3] = np.where(m > 1e-32, ex + 128, 0).astype(np.uint8)
    file_rows = rgbe[::-1]                                   # file row 0 = top = last row in memory after the flip
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n" + f"-Y {h} +X {w}\n".encode())
        f.write(file_rows.tobytes())
    f1 = np.ldexp(np.float32(1.0), rgbe[..., 3].astype(np.int32) - 136).astype(np.float32)
    dec = np.zeros((h, w, 4), np.float32)
    dec[..., :3] = np.where(rgbe[..., 3:4] != 0, rgbe[..., :3].astype(np.float32) * f1[..., None], 0.0)
    return dec


@pytest.mark.skipif(not os.path.exists(BIN), reason="drop-in main.cpp binary not built: it needs the reference project's sources (REF_DIR), which are not part of this repository")
def test_reference_main_cpp_drives_the_b200_path(rt, tmp_path):
    from PIL import Image as PILImage
    from sycl_ray_tracing_b200 import scenes
    c3 = scenes.c3_scene(nu=100, nv=50, sky_w=64, sky_h=32)
    base = str(tmp_path / "scene")
    write_obj(base, c3["tri9"], c3["mat_idx"], c3["mats10"])
    env = write_hdr_and_decode(str(tmp_path / "sky.hdr"), c3["env"][..., :3])
    w, h, spp, bounces = 96, 54, 4, 4
    r = subprocess.run([BIN, f"--sky={tmp_path / 'sky.hdr'}", f"--w={w}", f"--h={h}", f"--samples={spp}", f"--bounces={bounces}", base + ".obj"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    png = np.asarray(PILImage.open(tmp_path / "RT_output.png").convert("RGBA"))
    assert png.shape == (h, w, 4)
    # the same scene through the Python mirror; main.cpp hard-codes PBRT_DRAGON_CAMERA (main.cpp:110)
    sc = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=env)
    img, _ = sc.render(rt.Camera.PBRT_DRAGON_CAMERA, w, h, spp, bounces)
    expect = np.clip(img * np.float32(255.0), 0, 255).astype(np.uint8)[::-1]          # write_image_png: *255, clamp, flip (image_io.cpp:165-182)
    diff = np.abs(png.astype(np.int32) - expect.astype(np.int32))
    assert (diff <= 1).mean() > 0.995, f"{(diff > 1).sum()} of {diff.size} bytes differ by more than one level"
    assert png[..., :3].std() > 10, "the frame must not be blank"
    # main.cpp:118-125 ran to the end: three blends of the denoised frame. The OIDN entry points are served by the library's GPU denoise
    # stage (host/dropin/b200rt_oidn.c): blend 1 must equal b200rt_denoise of the frame, the others lie between it and the noisy frame
    den = rt.OIDN_denoise(np.ascontiguousarray(img[..., :3]))
    for name, blend in (("RT_output_denoised_1.png", 1.0), ("RT_output_denoised_0.75.png", 0.75), ("RT_output_denoised_0.5.png", 0.5)):
        assert os.path.exists(tmp_path / name)
        p = np.asarray(PILImage.open(tmp_path / name).convert("RGBA")).astype(np.int32)
        want = np.clip((blend * den + (1.0 - blend) * img[..., :3]) * np.float32(255.0), 0, 255).astype(np.uint8)[::-1].astype(np.int32)
        assert (np.abs(p[..., :3] - want) <= 1).mean() > 0.995, name
    assert (np.asarray(PILImage.open(tmp_path / "RT_output_denoised_1.png").convert("RGBA")) != png).mean() > 0.05, "the denoised frame is really filtered"
    # the same unmodified main.cpp on several ranks behind the boundary (b200rt_scene_create_multi): B200RT_GPUS=2 when the box has two
    # GPUs, and B200RT_DEVICE_LIST=0,0,0 (three ranks sharing the one device) everywhere. The PNG must be byte-identical.
    import torch
    variants = [{"B200RT_DEVICE_LIST": "0,0,0"}] + ([{"B200RT_GPUS": "2"}] if torch.cuda.device_count() >= 2 else [])
    for extra in variants:
        out = tmp_path / ("multi_" + "_".join(extra.values()).replace(",", ""))
        out.mkdir()
        r2 = subprocess.run([BIN, f"--sky={tmp_path / 'sky.hdr'}", f"--w={w}", f"--h={h}", f"--samples={spp}", f"--bounces={bounces}", base + ".obj"],
                            cwd=out, capture_output=True, text=True, timeout=600, env=dict(os.environ, **extra))
        assert r2.returncode == 0, r2.stdout[-2000:] + r2.stderr[-2000:]
        png2 = np.asarray(PILImage.open(out / "RT_output.png").convert("RGBA"))
        assert np.array_equal(png, png2), extra
