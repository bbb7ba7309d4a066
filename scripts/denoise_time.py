"""Cost of the guided denoiser on C3 (1920x1080): device time of rbrt_gpu_denoise_device for L = 1..5 levels and for the default, from
CUDA events around the call's kernels (rbrt_stats.ms_device), the median of REPS calls after one warm-up call each.  Inputs: a 64-spp
render_scene_hdr frame and render_aovs_device guides at S = 4 of the same camera and seed.  For scale, the device time of that 64-spp
frame (median of 3 after a warm-up).  The packed planes of a level (2 x 33 MB) fit the 126 MB L2, as they do in a render loop.
Writes one JSON line to stdout (and to OUT if given): python scripts/denoise_time.py [OUT] [REPS]"""
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
DEFAULT_LEVELS = 4


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, spp = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    frame = []
    for r in range(4):
        st = {}
        hdr = R.render_scene_hdr(cam, spp, scene, stats=st, seed=7)
        if r:
            frame.append(st["ms_device"])
    stream = torch.cuda.current_stream()
    aov = R.render_aovs_device(cam, 4, scene, seed=7, passes=("depth", "normal", "albedo"), stream=stream)
    d_hdr = torch.from_numpy(hdr).cuda()
    out = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
    rgb = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
    g = _abi.AovOutC(depth=aov["depth"].data_ptr(), normal=aov["normal"].data_ptr(), albedo=aov["albedo"].data_ptr())
    lib = _abi.lib()
    res = {"gpu": gpu, "workload": desc, "width": W, "height": H, "reps": REPS, "guides_spp": 4, "outputs": "hdr_out and rgb_out",
           "denoise": {}}
    for L in (1, 2, 3, 4, 5, 0):
        ms, st = [], _abi.StatsC()
        for r in range(REPS + 1):
            _abi.check(lib.rbrt_gpu_denoise_device(W, H, d_hdr.data_ptr(), g, _abi.DenoiseOptsC(levels=L), out.data_ptr(), rgb.data_ptr(),
                                                   stream.cuda_stream, st))
            if r:
                ms.append(st.ms_device)
        key = "default" if L == 0 else str(L)
        res["denoise"][key] = {"levels": L or DEFAULT_LEVELS, "ms_device": round(statistics.median(ms), 4), "ms_min": round(min(ms), 4),
                               "ms_max": round(max(ms), 4), "launches": st.launches}
        print("L =", key, res["denoise"][key], file=sys.stderr)
    levels = [res["denoise"][str(L)]["ms_device"] for L in (1, 2, 3, 4, 5)]
    res["ms_per_level"] = round((levels[4] - levels[0]) / 4, 4)
    res["frame_64spp_ms_device"] = round(statistics.median(frame), 3)
    res["default_share_of_frame"] = round(res["denoise"]["default"]["ms_device"] / res["frame_64spp_ms_device"], 4)
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
