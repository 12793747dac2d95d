#!/usr/bin/env python
"""bench.py — the path-tracing hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c3|c3k|c2|c1|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (default) = BASELINE.json config 3, the one the metric is quoted on: "Dragon" at 1920x1080, 64 spp, 8 bounces,
HDR skysphere with env-map importance sampling + BRDF importance sampling + MIS. The reference ships neither the Dragon
OBJ nor the HDR (.MISSING_LARGE_BLOBS), so the Dragon-class procedural stand-in of SURVEY.md Appendix A is used
(1 000 002 triangles, gold metal roughness 0.25, 2048x1024 sun+sky) — `data` says so. When data/OBJs/pbrt_dragon.obj and
data/Skyspheres/evening_road_01_puresky_2k.hdr exist (under $B200RT_ASSET_ROOT, this directory or /root/reference) they are
ingested by the library (b200rt_obj_load / b200rt_hdr_load) and used instead. `--workload c3k` is the same configuration on
the concave stand-in (displaced torus knot).

A step = one full frame: every rank renders its interleaved 16x16 tiles (wavefront integrator by default: wf_shade /
wf_trace kernel pairs over 4 tile groups on 4 streams), the tile buffers are gathered to rank 0 (NCCL) and un-tiled there. value = INTERSECT_SCENE-equivalent rays of the whole frame / step time
(CUDA events on the launching stream, max over ranks). Total work is fixed as N grows => "scaling": "strong".
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (width, height, spp, bounces, description)
    "c1": (512, 512, 16, 4, "cornell_pbr.obj 512x512 16spp 4 bounces, constant 1e-20 env (BASELINE config 1)"),
    "c2": (1920, 1080, 1, 1, "1M-triangle displaced sphere, 1920x1080 un-jittered primary rays (BASELINE config 2)"),
    "c3": (1920, 1080, 64, 8, "Dragon-class stand-in (1,000,002 tris, gold metal r=0.25), 1920x1080 64spp 8 bounces, "
                              "2048x1024 sun+sky env-map IS + BRDF IS + MIS (BASELINE config 3)"),
    "c3k": (1920, 1080, 64, 8, "concave Dragon-class stand-in (displaced (2,3) torus knot, 1,000,002 tris, gold metal r=0.25), 1920x1080 "
                               "64spp 8 bounces, 2048x1024 sun+sky env-map IS + BRDF IS + MIS (BASELINE config 3, SURVEY 8d's 'better' stand-in)"),
    "c5": (3840, 2160, 1024, 8, "20M-triangle procedural scene 3840x2160 1024spp 8 bounces (BASELINE config 5)"),
}


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    p.add_argument("--spp", type=int, default=0, help="override samples per pixel (0 = the workload's)")
    p.add_argument("--width", type=int, default=0)
    p.add_argument("--height", type=int, default=0)
    p.add_argument("--integrator", type=int, default=1, help="0 = megakernel, 1 = wavefront (default), 2 = persistent")
    p.add_argument("--warmup-spp", type=int, default=0, help="spp of the warm-up frames (0 = the workload's; c5 defaults to 8: a 1024-spp warm-up frame is minutes)")
    p.add_argument("--flags", type=int, default=0)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-sample", default="", help="WxHxSPP of the bounded CPU sample (default per workload)")
    p.add_argument("--lean", action="store_true", help="skip the optional legs (kernel-alone timing, RGBA8 end-to-end, dead-ray frame): for minutes-long frames (c5)")
    p.add_argument("--verify", action="store_true", help="N>1: rank 0 also renders the frame alone and asserts the gathered frame is bit-identical")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0): image.npy, the tone-mapped "
                        "RGBA frame, or prim.npy and t.npy for c2; over 60 MiB in all, the same seeded sample of pixels from each")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def load_workload(name, args):
    from sycl_ray_tracing_b200 import scenes
    import sycl_ray_tracing_b200 as rt
    w, h, spp, bounces, desc = WORKLOADS[name]
    if name == "c1":
        g = np.load(os.path.join(ROOT, "tests", "golden", "scenes.npz"))
        s = dict(tri9=g["cornell_tri9"], mat_idx=g["cornell_mat_idx"], mats10=g["cornell_mats10"], emissive=g["cornell_emissive"],
                 env=rt.constant_env(1.0e-20), camera=rt.Camera.CORNELL_BOX_CAMERA)
    elif name == "c2":
        s = scenes.c2_scene()
        s["env"] = rt.constant_env(1.0)
    elif name == "c3":
        real = scenes.find_real_dragon([os.environ.get("B200RT_ASSET_ROOT"), ROOT, "/root/reference"])
        if real:
            s = scenes.real_dragon_scene(*real)
            desc = f"PBRT Dragon ({len(s['tri9'])} tris, {os.path.basename(real[0])}) under {os.path.basename(real[1])}, 1920x1080 64spp 8 bounces (BASELINE config 3, real assets)"
        else:
            s = scenes.c3_scene()
    elif name == "c3k":
        s = scenes.c3_knot_scene()
    else:
        s = scenes.c5_scene()
    w = args.width or w
    h = args.height or h
    spp = args.spp or spp
    return s, w, h, spp, bounces, desc


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons of one GPU during the timed region (pynvml)."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz, self.ok = index, [], set(), False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if one exists for this workload."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)).get(workload)
        except Exception:
            return None
    return None


def cpu_sample_shape(name, args, w, h, spp):
    if args.cpu_sample:
        a = [int(v) for v in args.cpu_sample.lower().split("x")]
        return a[0], a[1], a[2]
    if name in ("c3", "c3k"):
        return 768, 432, 4          # 4/25 of the pixels, 1/16 of the spp: ~10-30 s of reference CPU work on 16 cores
    if name == "c5":
        return 192, 108, 1
    return w, h, spp                # c1 / c2 run in full on the CPU


def host_threads():
    """All host cores (torchrun exports OMP_NUM_THREADS=1 to its workers, so the count is passed explicitly)."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_cpu_sample(oracle_scene, cam17, name, sw, sh, sspp, bounces):
    """One pass of the reference CPU implementation over the bounded sample on all host cores; returns seconds."""
    if name == "c2":
        _, _, sec = oracle_scene.primary(cam17, sw, sh, mode=0, nthreads=host_threads())
        return sec
    _, sec = oracle_scene.render(cam17, sw, sh, sspp, bounces, nthreads=host_threads())
    return sec


def make_oracle_scene(s, need_env=True):
    from oracle.oracle import best_oracle
    o = best_oracle()
    sc = o.scene_from_arrays(s["tri9"], s["mat_idx"], s["mats10"], s["emissive"])
    if need_env:
        sc.set_env(s["env"])
    return o, sc


def port_ray_count(s, cam17, name, sw, sh, sspp, bounces):
    """INTERSECT_SCENE-equivalent query count of the sample (the reference cannot count; the port restatement can)."""
    if name == "c2":
        return sw * sh
    from oracle.oracle import PortOracle
    po = PortOracle()
    ps = po.scene_from_arrays(s["tri9"], s["mat_idx"], s["mats10"], s["emissive"])
    ps.set_env(s["env"])
    _, _, rays = po.render_counted(ps, cam17, sw, sh, sspp, bounces, nthreads=host_threads())
    return rays


def reference_arm(args, stdout_fd=1):
    """--impl reference: the reference's own CPU implementation (oracle/_ref when it was compiled, else the port) on all
    host cores, same workload config / metric / unit; each step is a bounded sample of the frame. Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    s, w, h, spp, bounces, desc = load_workload(args.workload, args)
    sw, sh, sspp = cpu_sample_shape(args.workload, args, w, h, spp)
    cam17 = s["camera"].as_array17()
    o, sc = make_oracle_scene(s)
    rays = port_ray_count(s, cam17, args.workload, sw, sh, sspp, bounces)
    for _ in range(args.warmup):
        run_cpu_sample(sc, cam17, args.workload, min(sw, 96), min(sh, 54), 1, bounces)      # warm caches / thread pool only
    secs = [run_cpu_sample(sc, cam17, args.workload, sw, sh, sspp, bounces) for _ in range(args.steps)]
    sec = sum(secs) / len(secs)
    value = rays / sec / 1e6
    sample = f"{sw}x{sh} px x {sspp} spp of the {w}x{h} x {spp} spp frame per step ({rays} rays)"
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "spp_per_s": sw * sh * sspp / sec,
        "config": {"workload": desc, "width": w, "height": h, "spp": spp, "max_bounces": bounces, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": host_threads(), "kind": o.kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(stdout_fd, line)


def ncu_counters(workload):
    """What actually bounds the dominant kernel, from the committed ncu capture of this round (profiles/r2_counters.json, written by
    tools/ncu_counters.py from the .ncu-rep of the shipping kernel): reported next to the nominal HBM fraction."""
    path = os.path.join(ROOT, "profiles", "r2_counters.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)).get(workload)
        except Exception:
            return None
    return None


DUMP_LIMIT_BYTES = 60 << 20          # 62.9 MB of data: the files stay under 64 MB with their headers


def dump_outputs(path, arrays):
    """Writes each (h, w, ...) array as path/<name>.npy: float32, integer arrays as float64 (exact). Over DUMP_LIMIT_BYTES in all,
    every array keeps the same pixels, a fixed seeded sample in row-major order, as (n_pixels, channels)."""
    os.makedirs(path, exist_ok=True)
    out = {k: np.asarray(a, np.float64 if np.issubdtype(a.dtype, np.integer) else np.float32) for k, a in arrays.items()}
    n_px = {a.shape[0] * a.shape[1] for a in out.values()}.pop()
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n_px, DUMP_LIMIT_BYTES // (total // n_px), replace=False))
        out = {k: a.reshape(n_px, -1)[keep] for k, a in out.items()}
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def emit_line(stdout_fd, line):
    """The one JSON line goes to the process's ORIGINAL stdout; everything else any library prints (NCCL's version banner, warnings)
    was sent to stderr by main()."""
    os.write(stdout_fd, (json.dumps(line) + "\n").encode())


def main():
    args = parse_args()
    # stdout carries exactly one JSON line: keep the real stdout aside and point fd 1 at stderr for the rest of the run
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        reference_arm(args, stdout_fd)
        return

    import torch
    import torch.distributed as dist
    import sycl_ray_tracing_b200 as rt
    from sycl_ray_tracing_b200 import distributed as D
    from sycl_ray_tracing_b200 import scenes

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # NCCL would print its version banner on stdout: stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=device)

    s, w, h, spp, bounces, desc = load_workload(args.workload, args)
    t_build = time.perf_counter()
    scene = rt.Scene(s["tri9"], s["mat_idx"], s["mats10"], s["emissive"], skysphere=s.get("env"), device=local_rank)
    build_s = time.perf_counter() - t_build
    cam = s["camera"]
    n_tri = len(s["tri9"])
    bytes_per_ray = scenes.algorithmic_bytes_per_ray(n_tri)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)      # > 126 MB L2
    warm_spp = args.warmup_spp or (8 if args.workload == "c5" and spp > 8 else spp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def cur_stream():
        return torch.cuda.current_stream(device).cuda_stream

    primary_only = args.workload == "c2"
    if primary_only:
        prim = torch.empty((h, w), dtype=torch.int32, device=device)
        tbuf = torch.empty((h, w), dtype=torch.float32, device=device)

        def step():
            scene.trace_primary_device(cam, w, h, prim.data_ptr(), tbuf.data_ptr(), stream_ptr=cur_stream(), rank=rank, world=world, flags=args.flags)
        warm_step = step
        rays_per_frame = w * h
        kernel_name = "k_primary"
        launches_per_step = 1
    else:
        g = D.make_cuda_gatherer(scene, cam, w, h, spp, bounces, rank, world, device, integrator=args.integrator, flags=args.flags)
        step = g.frame
        warm_step = step if warm_spp == spp else D.make_cuda_gatherer(scene, cam, w, h, warm_spp, bounces, rank, world, device,
                                                                     integrator=args.integrator, flags=args.flags).frame
        kernel_name = {0: "k_pathtrace_mega", 1: "wf_trace_coop", 2: "pt_persist"}[args.integrator]

    for _ in range(args.warmup):
        warm_step()
    barrier()

    verified = None
    if args.verify and not primary_only:
        img = step()
        if rank == 0:
            solo = D.make_cuda_gatherer(scene, cam, w, h, spp, bounces, 0, 1, device, integrator=args.integrator, flags=args.flags).frame()
            verified = bool(torch.equal(img.view(torch.int32), solo.view(torch.int32)))
            if not verified:
                raise SystemExit(f"bench.py --verify: the {world}-rank frame differs from the 1-rank frame")
        barrier()
        warm_step()            # rank 0's 1-rank frame re-sized the integrator's buffers: size them for this world again, outside the timed steps
        barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        flush.fill_(i & 0xff)                 # L2 flush between timed iterations (outside the event pair)
        ev[i][0].record()
        frame = step()
        ev[i][1].record()
    barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in (dict(prim=prim, t=tbuf) if primary_only else dict(image=frame)).items()})
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / args.steps
    print(f"bench.py rank {rank}: timed steps {['%.2f' % v for v in step_ms]} ms", file=sys.stderr, flush=True)

    # ---- roofline of the dominant kernel, measured live (CUDA events on the streams the kernels are launched on) ---------------------
    peak, peak_src = measured_peak()
    probe = torch.empty((D.tiles_for_rank(w, h, 0, world) * 256, 4), dtype=torch.float32, device=device)
    roofline = {"bound": "hbm", "kernel": kernel_name, "peak": peak, "unit": "GB/s", "peak_source": peak_src, "bytes_per_ray": bytes_per_ray,
                "bound_note": "nominal: algorithmic bytes of the reference's data shapes over the measured HBM copy peak (SURVEY 8d); the BVH is "
                              "L1/L2-resident, so DRAM is not what bounds the kernel: see 'ncu'"}
    if primary_only or args.integrator != 1:
        # one launch per step: the kernel's duration is the frame's render time
        kms = []
        kst = None
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(args.steps):
            flush.fill_(i & 0xff)
            k0.record()
            if primary_only:
                scene.trace_primary_device(cam, w, h, prim.data_ptr(), tbuf.data_ptr(), stream_ptr=cur_stream(), rank=rank, world=world, flags=args.flags)
            else:
                kst = scene.render_tiles_device(cam, w, h, spp, bounces, probe.data_ptr(), stream_ptr=cur_stream(), integrator=args.integrator,
                                                flags=args.flags, rank=rank, world=world, want_stats=(i == 0)) or kst
            k1.record()
            torch.cuda.synchronize()
            kms.append(k0.elapsed_time(k1))
        kernel_ms = torch.tensor([sum(kms) / len(kms)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(kernel_ms, op=dist.ReduceOp.MAX)
        kernel_ms = float(kernel_ms.item())
        if not primary_only:
            rank_rays, rank_launches = int(kst["rays"]), int(kst["gpu_launches"])
        rays_per_launch = w * h / world if primary_only else rank_rays
        achieved = rays_per_launch * bytes_per_ray / (kernel_ms * 1e-3) / 1e9
        roofline.update({"achieved": achieved, "frac": achieved / peak, "launches": 1, "avg_launch_ms": kernel_ms, "rays_per_launch": rays_per_launch})
    else:
        # Wavefront: the frame is ~3 400 launches on 3-4 overlapping streams. One more frame runs with every launch bracketed by CUDA
        # events on its own group stream (B200RT_FLAG_TIME_INLINE: nothing serialised, same schedule as a timed step). achieved =
        # algorithmic bytes of this rank's rays / the time during which at least one wf_trace_coop launch was running (the union of
        # the launch intervals, <= ms_per_step); sum_launch_ms adds up the overlapping launches and may exceed the step.
        flush.fill_(7)
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        kst = scene.render_tiles_device(cam, w, h, spp, bounces, probe.data_ptr(), stream_ptr=cur_stream(), integrator=args.integrator,
                                        flags=args.flags | rt.FLAG_TIME_INLINE, rank=rank, world=world, want_stats=True)
        t1e.record()
        torch.cuda.synchronize()
        frame_ms = t0e.elapsed_time(t1e)
        rank_rays, rank_launches = int(kst["rays"]), int(kst["gpu_launches"])
        union = max(kst["trace_union_ms"], 1e-9)
        achieved = kst["rays"] * bytes_per_ray / (union * 1e-3) / 1e9
        roofline.update({"achieved": achieved, "frac": achieved / peak, "launches": kst["trace_launches"],
                         "avg_launch_ms": kst["trace_ms"] / max(1, kst["trace_launches"]), "sum_launch_ms": kst["trace_ms"],
                         "union_launch_ms": kst["trace_union_ms"], "timed_frame_ms": frame_ms, "share_of_step": kst["trace_union_ms"] / frame_ms,
                         "rays_per_launch": kst["rays"] / max(1, kst["trace_launches"]),
                         "shade": {"kernel": "wf_shade", "launches": kst["shade_launches"], "sum_launch_ms": kst["shade_ms"],
                                   "avg_launch_ms": kst["shade_ms"] / max(1, kst["shade_launches"])},
                         "tail": {"kernel": "wf_tail", "launches": kst["tail_launches"], "sum_launch_ms": kst["tail_ms"]}})
        # the same kernel with the machine to itself (B200RT_FLAG_TIME_KERNELS: groups one after the other, full persistent grid): round 1's figure
        flush.fill_(9)
        ast = {"trace_launches": 0, "trace_ms": 0.0} if args.lean else scene.render_tiles_device(
            cam, w, h, spp, bounces, probe.data_ptr(), stream_ptr=cur_stream(), integrator=args.integrator,
            flags=args.flags | rt.FLAG_TIME_KERNELS, rank=rank, world=world, want_stats=True)
        if ast["trace_launches"] > 0 and ast["trace_ms"] > 0:
            a_ach = ast["rays"] * bytes_per_ray / (ast["trace_ms"] * 1e-3) / 1e9
            roofline["alone"] = {"launches": ast["trace_launches"], "avg_launch_ms": ast["trace_ms"] / ast["trace_launches"], "achieved": a_ach,
                                 "frac": a_ach / peak, "share_of_kernel_time": ast["trace_ms"] / (ast["trace_ms"] + ast["shade_ms"])}
    # rays of the whole frame (deterministic: counted by the device during the frame timed above) and this rank's launch count
    if not primary_only:
        rays_t = torch.tensor([rank_rays], dtype=torch.int64, device=device)
        if world > 1:
            dist.all_reduce(rays_t)
        rays_per_frame = int(rays_t.item())
        launches_per_step = rank_launches + (2 if rank == 0 else 0)       # + framebuffer fill and the accumulating un-tile on rank 0
    value = rays_per_frame / (ms_per_step * 1e-3) / 1e6
    tpr = profile_traffic(args.workload + "_trace_bytes_per_ray")
    roofline["traffic"] = (tpr * roofline["rays_per_launch"]) if (tpr and not primary_only and args.integrator == 1) else None
    roofline["ncu"] = ncu_counters(args.workload)

    # ---- end to end through the public host API: pinned host buffers in and out, copies inside the timed region ---------------------
    e2e = None
    if world == 1:
        fbimg = rt.Image(w, h, pinned=True)
        fb = fbimg.pixels
        prim_h = rt.pinned_array((h, w), np.int32) if primary_only else None
        t_h = rt.pinned_array((h, w), np.float32) if primary_only else None
        times = []
        stats = None
        if not primary_only:
            scene.render(cam, w, h, min(spp, 2), bounces, framebuffer=fb, integrator=args.integrator, flags=args.flags)       # allocations of this entry point
        else:
            scene.trace_primary_into(cam, w, h, prim_h, t_h, flags=args.flags)                                              # allocations of this entry point
        for i in range(max(1, min(args.steps, 3))):
            fb[...] = (0.0, 0.0, 0.0, 1.0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if primary_only:
                stats = scene.trace_primary_into(cam, w, h, prim_h, t_h, flags=args.flags)
            else:
                _, stats = scene.render(cam, w, h, spp, bounces, framebuffer=fb, integrator=args.integrator, flags=args.flags)
            times.append(time.perf_counter() - t0)
        e_sec = sum(times) / len(times)
        e2e = {"value": rays_per_frame / e_sec / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(stats["h2d_bytes"]),
               "d2h_bytes_per_step": int(stats["d2h_bytes"]), "api": "b200rt_trace_primary" if primary_only else "b200rt_render",
               "host_buffers": "page-locked (b200rt_host_alloc)"}
        if not primary_only and not args.lean:
            # the same frame leaving the GPU as the PNG's RGBA8 bytes (b200rt_render_rgba8: 4 B/pixel down instead of 16)
            out8 = rt.pinned_array((h, w, 4), np.uint8)
            scene.render_rgba8(cam, w, h, min(spp, 2), bounces, framebuffer=fb, out=out8, integrator=args.integrator, flags=args.flags)   # allocations
            t0 = time.perf_counter()
            _, st8 = scene.render_rgba8(cam, w, h, spp, bounces, framebuffer=fb, out=out8, integrator=args.integrator, flags=args.flags)
            e8 = time.perf_counter() - t0
            e2e["rgba8"] = {"value": rays_per_frame / e8 / 1e6, "h2d_bytes_per_step": int(st8["h2d_bytes"]), "d2h_bytes_per_step": int(st8["d2h_bytes"]),
                            "api": "b200rt_render_rgba8"}
    else:
        pinned = torch.empty((h, w, 4), dtype=torch.float32).pin_memory() if rank == 0 else None
        fb_host = torch.zeros((h, w, 4), dtype=torch.float32).pin_memory() if rank == 0 else None
        if rank == 0:
            fb_host[..., 3] = 1.0
        cam_host = torch.from_numpy(cam.as_array17()).pin_memory()
        cam_dev = torch.empty(17, dtype=torch.float32, device=device)
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(1, min(args.steps, 3))
        for i in range(n_e2e):
            cam_dev.copy_(cam_host, non_blocking=True)          # the frame's inputs: camera on every rank, the incoming framebuffer on rank 0
            img = g.frame(fb_in_host=fb_host)
            if rank == 0:
                pinned.copy_(img, non_blocking=True)
            torch.cuda.synchronize()
        barrier()
        e_sec = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=device)
        dist.all_reduce(e_sec, op=dist.ReduceOp.MAX)
        e2e = {"value": rays_per_frame / float(e_sec.item()) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": 68 + w * h * 16,
               "d2h_bytes_per_step": w * h * 16, "api": "distributed.FrameGatherer.frame (pinned framebuffer up, gathered frame down, rank 0)"}

    # same frame with the rays that provably cannot change the image skipped (B200RT_FLAG_SKIP_DEAD_RAYS): reported next to
    # the headline, which keeps the reference's full ray set
    dead = None
    if not primary_only and not args.lean:
        g2 = D.make_cuda_gatherer(scene, cam, w, h, spp, bounces, rank, world, device, integrator=args.integrator,
                                  flags=args.flags | rt.binding.FLAG_SKIP_DEAD_RAYS)
        g2.frame()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g2.frame(); b.record()
        barrier()
        dms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(dms, op=dist.ReduceOp.MAX)
        dead = {"ms_per_step": float(dms.item()), "spp_per_s": (w * h * spp) / (float(dms.item()) * 1e-3)}
        del g2

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            sw, sh, sspp = cpu_sample_shape(args.workload, args, w, h, spp)
            o, osc = make_oracle_scene(s)
            cam17 = cam.as_array17()
            # ray count of the sample from the GPU's own counter (identical paths => identical query count)
            if primary_only:
                srays = sw * sh
            else:
                _, sst = scene.render(cam, sw, sh, sspp, bounces, flags=args.flags & ~rt.FLAG_SKIP_DEAD_RAYS)
                srays = sst["rays"]
            sec = run_cpu_sample(osc, cam17, args.workload, sw, sh, sspp, bounces)
            cpu_baseline = {"value": srays / sec / 1e6, "unit": "Mrays/s", "cores": host_threads(), "kind": o.kind,
                            "sample": f"{sw}x{sh} px x {sspp} spp of the {w}x{h} x {spp} spp frame ({srays} rays, {sec:.2f} s)",
                            "spp_per_s": sw * sh * sspp / sec}
        except Exception as e:          # the baseline is reported context, never a reason to lose the GPU numbers
            cpu_baseline = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        info = scene.bvh_info()
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "step_ms_rank0": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": ("the reference's own assets, ingested by the library" if "real assets" in desc else
                     "synthetic (procedural stand-ins: the reference ships neither the Dragon OBJ nor the HDR skysphere)")
                    if args.workload != "c1" else "bundled cornell_pbr.obj (parsed by the reference, committed fixture)",
            "spp_per_s": (w * h * spp) / (ms_per_step * 1e-3),
            "rays_per_frame": rays_per_frame, "rays_per_sample": rays_per_frame / (w * h * spp),
            "config": {"workload": desc, "width": w, "height": h, "spp": spp, "max_bounces": bounces, "triangles": n_tri,
                       "integrator": {0: "megakernel", 1: "wavefront", 2: "persistent"}[args.integrator], "flags": args.flags,
                       "partition": f"interleaved 16x16 tiles over {world} rank(s), scene replicated, NCCL gather of mean-radiance tiles to rank 0, "
                                    "framebuffer += / tone map there",
                       "l2": "256 MiB buffer written between timed iterations (L2 flush)",
                       "warmup_spp": warm_spp,
                       "bvh": {k: info[k] for k in ("n_inner_nodes", "n_leaves", "max_depth", "has_diag_slabs", "n_wide_nodes", "wide_max_depth", "build_seconds")},
                       "scene_build_s": build_s, "scene_device_bytes": scene.device_bytes()},
            "skip_dead_rays": dead, "verified_equal_to_1_rank": verified,
            "clocks": sampler.result(),
            "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }
        emit_line(stdout_fd, line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
