"""Progressive accumulation on multi-device scenes, on the flagship frame (C3: 1 M triangles, 1920x1080, 64 spp, 8 bounces, 2048x1024
sky), and the cost of a float resolve against an RGBA8 resolve.

    python tools/accum_bench.py [--reps 3] [--resolve-reps 20] [--out profiles/r4_accum_bench.json]

Rank layouts: every visible GPU as one rank each (Scene(devices=N)); on a one-GPU box also 2 ranks sharing device 0, labelled
"shared": the ranks then compete for one GPU, so that row shows the host orchestration, not multi-GPU scaling. For each layout:
* b200rt_render(64 spp) on the multi-device scene: the stats' kernel_ms (slowest rank) and the host wall time of the call;
* the same 64 samples accumulated in chunks of 64, 16, 4 and 1 samples: the adds' kernel_ms (max over ranks) summed over the frame,
  and the host wall time of all adds; the final resolve is checked against the render's frame bit for bit;
* resolve against resolve_rgba8 at 1920x1080 and 3840x2160 (1 sample accumulated; into pageable numpy arrays, as Accumulator
  returns them): host wall time per call.
Every timing is repeated (--reps, --resolve-reps) after a warm-up of the same shape; min and median are reported. The card's name,
power limit and maximum SM clock are read by the same process (nvidia-smi queries only).
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

SPP, BOUNCES, W, H = 64, 8, 1920, 1080
CHUNKS = (64, 16, 4, 1)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    cards = []
    for line in r.stdout.strip().splitlines() if r.returncode == 0 else []:
        i, name, power, clock = [s.strip() for s in line.split(",")]
        cards.append(dict(index=int(i), name=name, power_limit=power, max_sm_clock=clock))
    return dict(cards=cards, torch_device_count=torch.cuda.device_count(), torch_name=torch.cuda.get_device_name(0))


def spread(values):
    v = np.asarray(values, np.float64)
    return dict(min=float(v.min()), median=float(np.median(v)), max=float(v.max()), reps=int(v.size))


def bench_layout(c3, devices, reps, resolve_reps):
    cam = c3["camera"]
    sc = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"], devices=devices)
    out = dict(devices=devices, ranks=len(devices), shared=len(set(devices)) < len(devices))

    sc.render(cam, W, H, 4, BOUNCES)                                      # warm-up: modules, wavefront buffers, gather buffer
    kernel, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        frame, st = sc.render(cam, W, H, SPP, BOUNCES)
        wall.append((time.perf_counter() - t0) * 1e3)
        kernel.append(st["kernel_ms"])
    out["render"] = dict(kernel_ms=spread(kernel), wall_ms=spread(wall), rays=st["rays"])

    out["chunks"] = {}
    for chunk in CHUNKS:
        warm = rt.Accumulator(sc, cam, W, H, SPP, BOUNCES)
        warm.add(chunk)
        del warm
        kernel, wall, equal = [], [], []
        for _ in range(reps):
            acc = rt.Accumulator(sc, cam, W, H, SPP, BOUNCES)
            k, rays = 0.0, 0
            t0 = time.perf_counter()
            for _ in range(SPP // chunk):
                s = acc.add(chunk)
                k += s["kernel_ms"]
                rays += s["rays"]
            wall.append((time.perf_counter() - t0) * 1e3)
            kernel.append(k)
            equal.append(bool(np.array_equal(acc.resolve().view(np.uint32), frame.view(np.uint32))) and rays == st["rays"])
            del acc
        out["chunks"][str(chunk)] = dict(adds=SPP // chunk, kernel_ms=spread(kernel), wall_ms=spread(wall), equal_to_render=all(equal),
                                         kernel_vs_render=float(np.median(kernel)) / out["render"]["kernel_ms"]["median"])

    out["resolve"] = {}
    for (w, h) in ((1920, 1080), (3840, 2160)):
        acc = rt.Accumulator(sc, cam, w, h, SPP, BOUNCES)
        acc.add(1)
        row = dict(width=w, height=h)
        for name, call, bytes_down in (("float", acc.resolve, w * h * 16), ("rgba8", acc.resolve_rgba8, w * h * 4)):
            call()
            times = []
            for _ in range(resolve_reps):
                t0 = time.perf_counter()
                call()
                times.append((time.perf_counter() - t0) * 1e3)
            row[name] = dict(wall_ms=spread(times), d2h_bytes=bytes_down)
        row["float_vs_rgba8"] = row["float"]["wall_ms"]["median"] / row["rgba8"]["wall_ms"]["median"]
        out["resolve"][f"{w}x{h}"] = row
        del acc
    del sc
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--resolve-reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_accum_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "accum_bench measures the GPU: no CUDA device"
    n = torch.cuda.device_count()
    layouts = [list(range(n))] + ([[0, 0]] if n == 1 else [])
    c3 = scenes.c3_scene()
    res = dict(gpu=gpu_info(), workload=dict(scene="C3", triangles=int(len(c3["tri9"])), width=W, height=H, spp=SPP, bounces=BOUNCES),
               layouts=[])
    for devices in layouts:
        r = bench_layout(c3, devices, args.reps, args.resolve_reps)
        res["layouts"].append(r)
        print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
