"""Geometry updates on the flagship scene (C3: 1 M-triangle displaced sphere on a ground quad, 1920x1080, 2048x1024 sky): what an
in-place refit costs against rebuilding, and how much traversal speed the refitted tree gives up as the deformation grows.

    python tools/refit_bench.py [--frames 30] [--out profiles/r5_refit_bench.json]

Two animations of the sphere (the ground quad stays): a twist about y by an angle growing with height (up to --max-turns turns at
the top), and a rigid rotation about y (up to --max-turns turns). Per frame:
* the refit's kernel time (stats kernel_ms: extent pass + every level of both layouts + SAH) and the wall time of
  b200rt_scene_update_triangles from pageable numpy memory, from page-locked memory, and of the _device variant from a CUDA tensor;
* the refitted tree's sah_cost.
At --checkpoints frames also:
* the 16-spp, 8-bounce frame time (kernel_ms) on the refitted scene and on a scene freshly created from the same vertices, and
  whether the two frames are bit-identical;
* the rebuild alternatives at those vertices: the device builder's and the host builder's build time, and a whole
  b200rt_scene_create (host builder, upload, environment tables).
The card's name, power limit and maximum SM clock are read by the same process (nvidia-smi queries only).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import sycl_ray_tracing_b200 as rt  # noqa: E402
from sycl_ray_tracing_b200 import scenes  # noqa: E402

W, H, SPP, BOUNCES = 1920, 1080, 16, 8


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    cards = []
    for line in r.stdout.strip().splitlines() if r.returncode == 0 else []:
        i, name, power, clock = [s.strip() for s in line.split(",")]
        cards.append(dict(index=int(i), name=name, power_limit=power, max_sm_clock=clock))
    return dict(cards=cards, torch_device_count=torch.cuda.device_count(), torch_name=torch.cuda.get_device_name(0))


def rotate_y(v, ang):
    c, s = np.cos(ang), np.sin(ang)
    return np.stack([c * v[:, 0] + s * v[:, 2], v[:, 1], -s * v[:, 0] + c * v[:, 2]], 1)


def animate(mesh, kind, turns):
    v = mesh.reshape(-1, 3).astype(np.float64)
    if kind == "twist":
        lo, hi = v[:, 1].min(), v[:, 1].max()
        ang = 2 * np.pi * turns * (v[:, 1] - lo) / (hi - lo)
    else:
        ang = np.full(len(v), 2 * np.pi * turns)
    return rotate_y(v, ang).reshape(-1, 9).astype(np.float32)


def run_curve(c3, kind, frames, max_turns, checkpoints):
    cam = c3["camera"]
    mesh, ground = c3["tri9"][:-2], c3["tri9"][-2:]
    sc = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"])
    sc.render(cam, W, H, 2, BOUNCES)                                     # warm-up: modules and wavefront state
    pinned = rt.pinned_array(c3["tri9"].shape, np.float32)
    dev = torch.empty(c3["tri9"].shape, dtype=torch.float32, device="cuda")
    sc.update_triangles(c3["tri9"])                                      # the first update builds the level lists
    rows = []
    for f in range(frames):
        turns = max_turns * f / max(frames - 1, 1)
        tri = np.concatenate([animate(mesh, kind, turns), ground])
        row = dict(frame=f, turns=turns)
        t0 = time.perf_counter()
        st = sc.update_triangles(tri)
        row["pageable_wall_ms"] = (time.perf_counter() - t0) * 1e3
        row["pageable_total_ms"] = st["total_ms"]
        row["kernel_ms"] = st["kernel_ms"]
        row["gpu_launches"] = st["gpu_launches"]
        pinned[...] = tri
        t0 = time.perf_counter()
        st = sc.update_triangles(pinned)
        row["pinned_wall_ms"] = (time.perf_counter() - t0) * 1e3
        row["pinned_kernel_ms"] = st["kernel_ms"]
        dev.copy_(torch.from_numpy(tri))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st = sc.update_triangles_device(dev.data_ptr(), len(tri))
        row["device_wall_ms"] = (time.perf_counter() - t0) * 1e3
        row["device_kernel_ms"] = st["kernel_ms"]
        row["sah_cost"] = sc.bvh_info()["sah_cost"]
        if f in checkpoints:
            img, sr = sc.render(cam, W, H, SPP, BOUNCES)
            t0 = time.perf_counter()
            fresh = rt.Scene(tri, c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"])
            row["scene_create_wall_ms"] = (time.perf_counter() - t0) * 1e3
            row["fresh_sah_cost"] = fresh.bvh_info()["sah_cost"]
            fresh.render(cam, W, H, 2, BOUNCES)
            img_f, sf = fresh.render(cam, W, H, SPP, BOUNCES)
            row["frame_ms_refitted"] = sr["kernel_ms"]
            row["frame_ms_fresh"] = sf["kernel_ms"]
            row["frames_bit_identical"] = bool(np.array_equal(img.view(np.uint32), img_f.view(np.uint32)) and sr["rays"] == sf["rays"])
            row["device_build_s"] = rt.BVH(tri, on_device=True).info()["build_seconds"]
            row["host_build_s"] = rt.BVH(tri).info()["build_seconds"]
            del fresh
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows


def summary(rows):
    keys = ("kernel_ms", "pageable_wall_ms", "pinned_wall_ms", "device_wall_ms")
    return {k: dict(min=float(np.min([r[k] for r in rows[1:]])), median=float(np.median([r[k] for r in rows[1:]]))) for k in keys}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--max-turns", type=float, default=0.5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_refit_bench.json"))
    a = ap.parse_args()
    c3 = scenes.c3_scene()
    checkpoints = {0, a.frames // 6, a.frames // 3, a.frames // 2, (2 * a.frames) // 3, a.frames - 1}
    out = dict(gpu=gpu_info(), scene="C3: 1 000 002 triangles, 1920x1080, 2048x1024 sky", spp=SPP, max_bounces=BOUNCES,
               frames=a.frames, max_turns=a.max_turns, curves={})
    for kind in ("twist", "rigid"):
        rows = run_curve(c3, kind, a.frames, a.max_turns, checkpoints)
        out["curves"][kind] = dict(rows=rows, summary=summary(rows))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(dict(gpu=out["gpu"], twist=out["curves"]["twist"]["summary"], rigid=out["curves"]["rigid"]["summary"]), indent=1))


if __name__ == "__main__":
    main()
