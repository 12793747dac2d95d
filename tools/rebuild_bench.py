"""In-place BVH rebuilds (b200rt_scene_rebuild_bvh[_device]) against the alternatives, and the frame time they win back from a refitted
tree.

    python tools/rebuild_bench.py [--reps 5] [--out profiles/r6_rebuild_bench.json] [--no-c5]

* C3 (1 M-triangle displaced sphere on a ground quad) per call, --reps times each: the rebuild from pageable numpy memory, from
  page-locked memory and (_device) from a CUDA tensor, with its stats (kernel_ms, gpu_launches, h2d / d2h bytes); against the
  refit (b200rt_scene_update_triangles), b200rt_bvh_build_device's build_seconds and a whole b200rt_scene_create (host builder,
  upload, environment tables).
* The refit benchmark's two animations (tools/refit_bench.py: a twist about y growing with height, a rigid rotation about y, up to
  half a turn): at each checkpoint the 16-spp, 8-bounce 1920x1080 frame (kernel_ms) on the refitted scene, on the rebuilt scene, on a
  fresh host-built scene and on a fresh scene over b200rt_bvh_build_device's tree, and whether the frames are bit-identical.
* The C5 mesh (20 M triangles): the rebuild (_device and pageable) against b200rt_bvh_build_device's build_seconds.
The card's name, power limit and maximum SM clock are read by the same process (nvidia-smi queries only).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import sycl_ray_tracing_b200 as rt  # noqa: E402
from refit_bench import BOUNCES, H, SPP, W, animate, gpu_info  # noqa: E402
from sycl_ray_tracing_b200 import scenes  # noqa: E402

STAT_KEYS = ("kernel_ms", "total_ms", "gpu_launches", "h2d_bytes", "d2h_bytes")


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st = fn()
    return (time.perf_counter() - t0) * 1e3, st


def med(rows, k):
    return float(np.median([r[k] for r in rows]))


def per_call(c, reps, label):
    """Every way to get a good tree for new vertices of a resident scene, at the same vertices."""
    tri = c["tri9"]
    sc = rt.Scene(tri, c["mat_idx"], c["mats10"], c["emissive"], skysphere=c.get("env"))
    pinned = rt.pinned_array(tri.shape, np.float32)
    pinned[...] = tri
    dev = torch.from_numpy(tri).cuda()
    sc.rebuild_bvh(tri)                                                    # warm-up: builder modules, the refit and staging buffers
    sc.update_triangles(tri)
    out = {}
    for name, fn in (("rebuild_pageable", lambda: sc.rebuild_bvh(tri)), ("rebuild_pinned", lambda: sc.rebuild_bvh(pinned)),
                     ("rebuild_device", lambda: sc.rebuild_bvh_device(dev.data_ptr(), len(tri))),
                     ("refit_pageable", lambda: sc.update_triangles(tri)),
                     ("refit_device", lambda: sc.update_triangles_device(dev.data_ptr(), len(tri)))):
        rows = []
        for _ in range(reps):
            wall, st = timed(fn)
            rows.append(dict(wall_ms=wall, **{k: st[k] for k in STAT_KEYS}))
        out[name] = dict(rows=rows, median_wall_ms=med(rows, "wall_ms"), median_kernel_ms=med(rows, "kernel_ms"))
        print(label, name, json.dumps(out[name]["rows"][-1]), flush=True)
    info = sc.bvh_info()
    out["tree"] = dict(n_wide_nodes=info["n_wide_nodes"], n_inner_nodes=info["n_inner_nodes"], n_triangles=info["n_triangles"],
                       bytes=80 * info["n_wide_nodes"] + 64 * info["n_inner_nodes"] + 48 * info["n_triangles"],
                       vertex_bytes=int(tri.nbytes))
    builds = [rt.BVH(tri, on_device=True).info()["build_seconds"] * 1e3 for _ in range(reps)]
    out["device_build_ms"] = dict(rows=builds, median=float(np.median(builds)))
    print(label, "device build", out["device_build_ms"], flush=True)
    return sc, out


def scene_create_ms(c, reps):
    rows = []
    for _ in range(reps):
        wall, s = timed(lambda: rt.Scene(c["tri9"], c["mat_idx"], c["mats10"], c["emissive"], skysphere=c["env"]))
        rows.append(wall)
        del s
    return dict(rows=rows, median=float(np.median(rows)))


def frame(sc, cam):
    sc.render(cam, W, H, 2, BOUNCES)
    img, st = sc.render(cam, W, H, SPP, BOUNCES)
    return img, st


def curve(c3, kind, checkpoints):
    cam = c3["camera"]
    mesh, ground = c3["tri9"][:-2], c3["tri9"][-2:]
    args = (c3["mat_idx"], c3["mats10"], c3["emissive"])
    refitted = rt.Scene(c3["tri9"], *args, skysphere=c3["env"])
    rebuilt = rt.Scene(c3["tri9"], *args, skysphere=c3["env"])
    rows = []
    for turns in checkpoints:
        tri = np.concatenate([animate(mesh, kind, turns), ground])
        refitted.update_triangles(tri)
        st_rb = rebuilt.rebuild_bvh(tri)
        fresh = rt.Scene(tri, *args, skysphere=c3["env"])
        fresh_dev = rt.Scene(tri, *args, skysphere=c3["env"], bvh=rt.BVH(tri, on_device=True))
        res = {name: frame(s, cam) for name, s in (("refitted", refitted), ("rebuilt", rebuilt), ("fresh_host_built", fresh),
                                                   ("fresh_device_built", fresh_dev))}
        ref_img, ref_st = res["fresh_host_built"]
        row = dict(turns=turns, rebuild_kernel_ms=st_rb["kernel_ms"], rebuild_total_ms=st_rb["total_ms"],
                   sah_refitted=refitted.bvh_info()["sah_cost"], sah_rebuilt=rebuilt.bvh_info()["sah_cost"],
                   sah_fresh_host_built=fresh.bvh_info()["sah_cost"])
        for name, (img, st) in res.items():
            row[f"frame_ms_{name}"] = st["kernel_ms"]
            row[f"bit_identical_{name}"] = bool(np.array_equal(img.view(np.uint32), ref_img.view(np.uint32)) and st["rays"] == ref_st["rays"])
        rows.append(row)
        print(kind, json.dumps(row), flush=True)
        del fresh, fresh_dev
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_rebuild_bench.json"))
    ap.add_argument("--no-c5", action="store_true")
    a = ap.parse_args()
    out = dict(gpu=gpu_info(), spp=SPP, max_bounces=BOUNCES, frame=f"{W}x{H}")
    c3 = scenes.c3_scene()
    sc, out["c3_per_call"] = per_call(c3, a.reps, "c3")
    del sc
    out["c3_per_call"]["scene_create_ms"] = scene_create_ms(c3, a.reps)
    print("c3 scene create", out["c3_per_call"]["scene_create_ms"], flush=True)
    checkpoints = [0.0, 0.125, 0.25, 0.375, 0.5]
    out["curves"] = {kind: curve(c3, kind, checkpoints) for kind in ("twist", "rigid")}
    if not a.no_c5:
        c5 = scenes.c5_scene(sky_w=64, sky_h=32)
        c5 = dict(tri9=c5["tri9"], mat_idx=c5["mat_idx"], mats10=c5["mats10"], emissive=c5["emissive"])
        sc, out["c5_per_call"] = per_call(c5, max(2, a.reps // 2), "c5")
        del sc
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
