"""Cost of the first-hit AOVs on C3 (1920x1080, 1.31 M triangles): device time of rbrt_gpu_render_aov_device (all seven planes) for
S = 1, 4, 16 and 64 samples, in CUDA events around the kernel (rbrt_stats.ms_device), the median of REPS calls after one warm-up call
each; Mrays/s; BVH node visits and triangle tests per camera ray from the kernel's counters; and, for scale, the device time of one
64-spp frame of the same camera (rbrt_gpu_render, median of 3).  The calls repeat on the same scene, so the tree and the triangle
records (about 100 MB) are mostly in the 126 MB L2 after the first one, as they are in an animation loop.
Writes one JSON line to stdout (and to OUT if given): python scripts/aov_time.py [OUT] [REPS]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
import rbrt_b200 as R
from rbrt_b200 import _abi

OUT = sys.argv[1] if len(sys.argv) > 1 else None
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 10


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, spp = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    lib = _abi.lib()
    n = W * H
    planes = {k: torch.empty(n * c, dtype=torch.float32, device="cuda")
              for k, c in (("depth", 1), ("normal", 3), ("albedo", 3), ("coverage", 1), ("hit_kind", 1), ("elem_idx", 1), ("tri_idx", 1))}
    out = _abi.AovOutC(**{k: t.data_ptr() for k, t in planes.items()})
    stream = torch.cuda.current_stream()
    res = {"gpu": gpu, "workload": desc, "width": W, "height": H, "reps": REPS, "aov": {}}
    for s in (1, 4, 16, 64):
        ms, st = [], _abi.StatsC()
        for r in range(REPS + 1):
            _abi.check(lib.rbrt_gpu_render_aov_device(scene.handle(), cam.to_c(), s, 7, out, stream.cuda_stream, st))
            if r:
                ms.append(st.ms_device)
        med = statistics.median(ms)
        rays = n * s
        res["aov"][s] = {"ms_device": round(med, 4), "ms_min": round(min(ms), 4), "ms_max": round(max(ms), 4),
                         "mrays_per_s": round(rays / med / 1e3, 1), "node_visits_per_ray": round(st.node_visits / rays, 3),
                         "tri_tests_per_ray": round(st.tri_tests / rays, 3), "nan_rays": st.nan_rays}
        print("S =", s, res["aov"][s], file=sys.stderr)
    frame = []
    for r in range(4):
        st = {}
        R.render_scene(cam, spp, scene, stats=st, seed=7)
        if r:
            frame.append(st["ms_device"])
    res["frame_64spp_ms_device"] = round(statistics.median(frame), 3)
    res["aov16_share_of_frame"] = round(res["aov"][16]["ms_device"] / res["frame_64spp_ms_device"], 4)
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
