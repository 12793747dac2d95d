"""Cost of the denoiser's feature buffers and of the guided filter on the flagship frame (C3: 1 M triangles, 1920x1080, PBRT dragon
camera, 2048x1024 sky).

    python tools/aov_bench.py [--reps 50] [--out profiles/r3_aov_bench.json]

* AOV pass (b200rt_render_aovs_device) for k = 1, 2, 4 stratified rays per pixel axis, next to b200rt_trace_primary_device on the
  same frame: CUDA events around every call on the launching stream, median and mean over --reps calls after a warm-up of each shape.
* Denoise, 5 passes, 3 channels at 1080p, colour-only vs guided (albedo + normal from the k = 2 pass): kernel time per call from
  torch.profiler (the sum of the a-trous and blend kernels of one call), and the wall time of the whole host call (allocations and
  PCIe copies included).
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


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in r.stdout.strip().split(",")] if r.returncode == 0 else ("unknown", "unknown", "unknown")
    return dict(name=name, power_limit=power, max_sm_clock=clock, torch_name=torch.cuda.get_device_name(0))


def time_calls(fn, reps):
    fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return dict(median_ms=float(np.median(ms)), mean_ms=float(ms.mean()), min_ms=float(ms.min()), reps=reps)


def denoise_kernel_ms(call, reps):
    """kernel time of one call: the a-trous and blend kernels of `reps` calls under torch.profiler, summed, over reps"""
    from torch.profiler import ProfilerActivity, profile
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.key_averages():
        if "k_atrous" in e.key or "k_denoise_blend" in e.key:
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            per_kernel[e.key] = dict(us_per_call=t / reps, launches_per_call=e.count / reps)
    return sum(v["us_per_call"] for v in per_kernel.values()) / 1e3, per_kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_aov_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "aov_bench measures the GPU: no CUDA device"
    info = gpu_info()
    c3 = scenes.c3_scene()
    sc = rt.Scene(c3["tri9"], c3["mat_idx"], c3["mats10"], c3["emissive"], skysphere=c3["env"], device=0)
    cam, w, h = c3["camera"], 1920, 1080
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    albedo = torch.empty((h, w, 3), dtype=torch.float32, device=dev)
    normal = torch.empty_like(albedo)
    prim = torch.empty((h, w), dtype=torch.int32, device=dev)
    t = torch.empty((h, w), dtype=torch.float32, device=dev)
    res = dict(gpu=info, scene=dict(name="C3", triangles=int(len(c3["tri9"])), width=w, height=h))

    primary = lambda: sc.trace_primary_device(cam, w, h, prim.data_ptr(), t.data_ptr(), stream_ptr=stream)
    aov = {k: (lambda k=k: sc.render_aovs_device(cam, w, h, albedo.data_ptr(), normal.data_ptr(), samples_per_axis=k, stream_ptr=stream))
           for k in (1, 2, 4)}
    for fn in [primary] + list(aov.values()):          # warm every shape
        fn()
    torch.cuda.synchronize()
    p = time_calls(primary, args.reps)
    p["mrays_per_s"] = w * h / p["median_ms"] / 1e3
    res["trace_primary"] = p
    for k, fn in aov.items():
        r = time_calls(fn, args.reps)
        r["rays"] = w * h * k * k
        r["mrays_per_s"] = r["rays"] / r["median_ms"] / 1e3
        r["vs_trace_primary"] = r["median_ms"] / p["median_ms"]
        res[f"aov_k{k}"] = r

    # denoise inputs: a 1-spp C3 frame and its k = 2 feature buffers
    img, _ = sc.render(cam, w, h, 1, 8)
    img = np.ascontiguousarray(img[..., :3])
    a2, n2, _ = sc.render_aovs(cam, w, h, samples_per_axis=2)
    calls = dict(colour_only=lambda: rt.OIDN_denoise(img), guided=lambda: rt.OIDN_denoise(img, albedo=a2, normal=n2))
    for name, call in calls.items():
        kms, per_kernel = denoise_kernel_ms(call, args.reps)
        call()
        t0 = time.perf_counter()
        for _ in range(10):
            call()
        wall = (time.perf_counter() - t0) / 10 * 1e3
        res[f"denoise_{name}"] = dict(kernel_ms_per_call=kms, kernels=per_kernel, host_call_ms=wall, passes=5, channels=3)
    res["denoise_guided_vs_colour_kernel_ratio"] = res["denoise_guided"]["kernel_ms_per_call"] / res["denoise_colour_only"]["kernel_ms_per_call"]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
