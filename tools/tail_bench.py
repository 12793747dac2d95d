"""Development tool: the wavefront integrator's barrier-free tail (csrc/persist.cu wf_tail) against the pass-synchronous frame,
whole frames and one rank of 8 emulated on one GPU, over the tail's knobs and the tile-group count — all inside one process (the
knobs are environment variables the library reads per frame). One JSON line per configuration.

    SPP=64 python tools/tail_bench.py [config-set ...]          # sets: base tail groups
"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import sycl_ray_tracing_b200 as rt
from sycl_ray_tracing_b200 import scenes

spp = int(os.environ.get("SPP", "64"))
reps = int(os.environ.get("REPS", "2"))
workload = os.environ.get("WORKLOAD", "c3")
sets = sys.argv[1:] or ["base"]
w, h = (3840, 2160) if workload == "c5" else (1920, 1080)
s = {"c5": scenes.c5_scene, "c3k": scenes.c3_knot_scene if hasattr(scenes, "c3_knot_scene") else scenes.c3_scene}.get(workload, scenes.c3_scene)()
sc = rt.Scene(s["tri9"], s["mat_idx"], s["mats10"], s["emissive"], skysphere=s["env"])
fb = rt.Image(w, h, pinned=True).pixels
KNOBS = ("B200RT_WF_GROUPS", "B200RT_WF_TAIL_PCT", "B200RT_WF_TAIL_CAP", "B200RT_WF_TAIL_MIN")

configs = []
def add(name, world, flags=0, **env):
    configs.append((name, world, flags, {("B200RT_" + k): str(v) for k, v in env.items()}))

for world in (1, 8):
    if "base" in sets:
        add("passes only", world, rt.FLAG_WF_PASSES_ONLY)
        add("default (passes + per-warp tail)", world)
    if "tail" in sets:
        add("default (passes + per-warp tail)", world)
        for pct, cap in ((10, 30000), (20, 30000), (20, 100000), (40, 100000)):
            add(f"tail pct {pct} cap {cap}", world, WF_TAIL_PCT=pct, WF_TAIL_CAP=cap)
        add("all tail from the start (groups <= 10M)", world, WF_TAIL_MIN=10000000)
    if "groups" in sets:
        for g in (1, 2, 3, 4, 6):
            add(f"groups {g}", world, WF_GROUPS=g)

first = {}
for name, world, flags, env in configs:
    for k in KNOBS:
        os.environ.pop(k, None)
    os.environ.update(env)
    sc.render(s["camera"], w, h, 1, 8, framebuffer=fb, rank=0, world=world, flags=flags)
    best = None
    for rep in range(reps):
        fb[...] = (0, 0, 0, 1)
        _, st = sc.render(s["camera"], w, h, spp, 8, framebuffer=fb, rank=0, world=world, flags=flags)
        best = st if best is None or st["kernel_ms"] < best["kernel_ms"] else best
    key = (world,)
    img = fb.copy()
    if key not in first:
        first[key] = (img, best["rays"])
    same = bool(np.array_equal(img.view(np.uint32), first[key][0].view(np.uint32))) and best["rays"] == first[key][1]
    print(json.dumps(dict(workload=workload, config=name, world=world, spp=spp, kernel_ms=round(best["kernel_ms"], 2), mrays_s=round(best["rays"] / best["kernel_ms"] / 1e3, 1),
                          launches=best["gpu_launches"], rays=best["rays"], equal_to_first=same, env=env)), flush=True)
