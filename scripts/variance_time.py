"""Cost of the per-pixel variance and of the variance-guided filter on C3 (1920x1080, 64 spp).

Render: rbrt_gpu_render_hdr_variance_device at K = 2 and 4 against the plain frame, rbrt_gpu_render_frames_device into an HDR plane with
RBRT_OPT_SPLIT_BATCHES (the device work of rbrt_gpu_render_hdr for this frame, which sets that flag itself from 2^26 paths).  Each call is
enqueued without stats on one stream and timed with CUDA events around it; the three are alternated, REPS rounds after one warm-up round,
and the median, min and max are reported.  The images are checked against each other (the sharded means within 1e-5 relative of the
plain frame).  Filter: device time of rbrt_gpu_denoise_variance_device for L = 1..5 levels and the default, from its stats (CUDA events
around its kernels), the median of REPS calls after one warm-up call each; inputs the K = 4 frame, its variance and AOVs at S = 4 of the
same camera and seed.  The card's name, power limit and SM clock are read in the same run.
Writes one JSON line to stdout (and to OUT if given): python scripts/variance_time.py [OUT] [REPS]"""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import rbrt_b200 as R
from rbrt_b200 import _abi

OUT = sys.argv[1] if len(sys.argv) > 1 else None
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 10
SEED = 7


def stat(ms):
    return {"ms_device": round(statistics.median(ms), 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3)}


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, spp = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    lib = _abi.lib()
    stream = torch.cuda.current_stream()
    plain = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
    hdr = {K: torch.empty((H, W, 3), dtype=torch.float32, device="cuda") for K in (2, 4)}
    var = {K: torch.empty((H, W, 3), dtype=torch.float32, device="cuda") for K in (2, 4)}
    seeds = (C.c_uint64 * 1)(SEED)
    d_hdr = (C.c_void_p * 1)(plain.data_ptr())
    split = R.render.make_opts(seed=SEED, split=True)
    opts = R.render.make_opts(seed=SEED)

    def run(which):
        if which == "plain":
            _abi.check(lib.rbrt_gpu_render_frames_device(scene.handle(), cam.to_c(), seeds, 1, spp, split, None, d_hdr, stream.cuda_stream, None))
        else:
            _abi.check(lib.rbrt_gpu_render_hdr_variance_device(scene.handle(), cam.to_c(), spp, which, opts, hdr[which].data_ptr(),
                                                               var[which].data_ptr(), stream.cuda_stream, None))

    times = {"plain": [], 2: [], 4: []}
    for r in range(REPS + 1):
        for which in ("plain", 2, 4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run(which)
            e1.record(stream)
            e1.synchronize()
            if r:
                times[which].append(e0.elapsed_time(e1))
    ref = plain.cpu().numpy().astype(np.float64)
    rel = {K: float((np.abs(hdr[K].cpu().numpy() - ref) / np.maximum(np.abs(ref), 1e-30)).max()) for K in (2, 4)}
    res = {"gpu": gpu, "workload": desc, "width": W, "height": H, "spp": spp, "reps": REPS, "seed": SEED,
           "plain_frame": stat(times["plain"]),
           "render_hdr_variance": {str(K): dict(stat(times[K]), splits=K, max_rel_diff_vs_plain=rel[K],
                                                ratio_to_plain=round(statistics.median(times[K]) / statistics.median(times["plain"]), 4))
                                   for K in (2, 4)}}
    print("render", res["plain_frame"], res["render_hdr_variance"], file=sys.stderr)
    aov = R.render_aovs_device(cam, 4, scene, seed=SEED, passes=("depth", "normal", "albedo"), stream=stream)
    g = _abi.AovOutC(depth=aov["depth"].data_ptr(), normal=aov["normal"].data_ptr(), albedo=aov["albedo"].data_ptr())
    out = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
    rgb = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
    res["filter"] = {}
    for L in (1, 2, 3, 4, 5, 0):
        ms, st = [], _abi.StatsC()
        for r in range(REPS + 1):
            _abi.check(lib.rbrt_gpu_denoise_variance_device(W, H, hdr[4].data_ptr(), var[4].data_ptr(), g, _abi.DenoiseOptsC(levels=L),
                                                            out.data_ptr(), rgb.data_ptr(), stream.cuda_stream, st))
            if r:
                ms.append(st.ms_device)
        key = "default" if L == 0 else str(L)
        res["filter"][key] = {"levels": L or 5, "ms_device": round(statistics.median(ms), 4), "ms_min": round(min(ms), 4),
                              "ms_max": round(max(ms), 4), "launches": st.launches}
        print("L =", key, res["filter"][key], file=sys.stderr)
    levels = [res["filter"][str(L)]["ms_device"] for L in (1, 2, 3, 4, 5)]
    res["filter_ms_per_level"] = round((levels[4] - levels[0]) / 4, 4)
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
