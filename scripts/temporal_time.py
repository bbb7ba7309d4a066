"""Cost of the temporal accumulation on C3 (1920x1080): device time of rbrt_gpu_temporal_accumulate_device from CUDA events around its
kernel (rbrt_stats.ms_device), the median of REPS calls after one warm-up call.  Inputs: two frames of a sideways camera move (0.04 to the
right), each a 16-spp render_hdr_variance_device frame (K = 4) with render_aovs_device guides at S = 4 of the same camera and seed; the
first is accumulated as the history of the second.  Timed for the moving camera (reprojection, bilinear taps), for a static camera (each
pixel from itself), and with var_out for both.  The planes a call reads and writes (about 150 MB) exceed the 126 MB L2 only slightly; they
are not flushed between calls, as in a render loop that accumulates right after rendering.
Writes one JSON line to stdout (and to OUT if given): python scripts/temporal_time.py [OUT] [REPS]"""
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
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, _ = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    p = camkw["position"]
    cams = [R.Camera.new(R.Vec3(p.x + 0.04 * f, p.y, p.z), camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"]) for f in (0, 1)]
    stream = torch.cuda.current_stream()
    frames = []
    for f, cam in enumerate(cams):
        hdr, var = R.render_hdr_variance_device(cam, 16, scene, splits=4, seed=7 + f, stream=stream)
        aovs = R.render_aovs_device(cam, 4, scene, seed=7 + f, passes=("depth", "normal", "ids"), stream=stream)
        frames.append((hdr, var, aovs))
    h0 = R.temporal_accumulate_device(cams[0], frames[0][0], frames[0][2], var=frames[0][1], stream=stream)
    hist = {"hdr": h0[0], "var": h0[1], "length": h0[2], "aovs": frames[0][2]}
    torch.cuda.synchronize()
    lib = _abi.lib()
    g = lambda a: _abi.AovOutC(depth=a["depth"].data_ptr(), normal=a["normal"].data_ptr(), hit_kind=a["hit_kind"].data_ptr(),
                               elem_idx=a["elem_idx"].data_ptr())
    out = [torch.empty((H, W, 3), dtype=torch.float32, device="cuda"), torch.empty((H, W, 3), dtype=torch.float32, device="cuda"),
           torch.empty((H, W), dtype=torch.float32, device="cuda")]
    hdr, var, aovs = frames[1]
    res = {"gpu": gpu, "workload": desc, "width": W, "height": H, "reps": REPS, "frame_spp": 16, "splits": 4, "guides_spp": 4,
           "temporal": {}}
    for label, prev in (("moving", cams[0]), ("static", cams[1])):
        h = _abi.TemporalHistoryC(cam=prev.to_c(), hdr=hist["hdr"].data_ptr(), var=hist["var"].data_ptr(), length=hist["length"].data_ptr(),
                                  guides=g(hist["aovs"]))
        for with_var in (False, True):
            ms, st = [], _abi.StatsC()
            for r in range(REPS + 1):
                _abi.check(lib.rbrt_gpu_temporal_accumulate_device(W, H, cams[1].to_c(), hdr.data_ptr(), var.data_ptr(), g(aovs), h, None,
                                                                   out[0].data_ptr(), out[1].data_ptr() if with_var else None,
                                                                   out[2].data_ptr(), stream.cuda_stream, st))
                if r:
                    ms.append(st.ms_device)
            kept = float((out[2] > 1).float().mean())
            key = label + ("_with_var" if with_var else "")
            res["temporal"][key] = {"ms_device": round(statistics.median(ms), 4), "ms_min": round(min(ms), 4), "ms_max": round(max(ms), 4),
                                    "launches": st.launches, "history_kept": round(kept, 4)}
            print(key, res["temporal"][key], file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
