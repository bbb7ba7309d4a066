"""Cost of the per-object motion vectors on C3 (1920x1080), each the median of REPS calls after one warm-up call:
  snapshot        rbrt_gpu_scene_snapshot, CUDA events around the call on the stream (1.31 M triangle records scattered, 63 MB);
  motion_static   rbrt_gpu_render_motion_device after a snapshot of the unchanged scene (rbrt_stats.ms_device);
  motion_refit    the same after a refit of the whole mesh (scripts/update_time.py's travelling wave, step 1) since the snapshot: every
                  mesh hit forms P' from its triangle's snapshot record;
  temporal_motion rbrt_gpu_temporal_accumulate_motion_device with that motion pass (rbrt_stats.ms_device), next to the camera-only call
                  on the same planes (temporal_camera).
The history and the frame are 16-spp render_hdr_variance_device frames (K = 4) of the static camera with render_aovs_device guides at
S = 4.  The planes are not flushed from L2 between calls, as in a frame loop.  The card's name and power limit are read in the same run.
Writes one JSON line to stdout (and to OUT if given): python scripts/motion_time.py [OUT] [REPS]"""
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


def deform(base, k):
    ph = 0.05 * k
    return (base + 0.6 * torch.sin(0.15 * base.roll(1, dims=-1) + ph)).contiguous()


def stat(ms):
    return {"ms": round(statistics.median(ms), 4), "ms_min": round(min(ms), 4), "ms_max": round(max(ms), 4)}


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, _ = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    stream = torch.cuda.current_stream()
    lib = _abi.lib()
    h = scene.handle()
    res = {"gpu": gpu, "workload": desc, "width": W, "height": H, "reps": REPS}

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for r in range(REPS + 1):
        e0.record(stream)
        _abi.check(lib.rbrt_gpu_scene_snapshot(h, stream.cuda_stream))
        e1.record(stream)
        e1.synchronize()
        if r:
            ms.append(e0.elapsed_time(e1))
    res["snapshot"] = stat(ms)

    m = torch.empty((H, W, 2), dtype=torch.float32, device="cuda")
    pd = torch.empty((H, W), dtype=torch.float32, device="cuda")
    out = _abi.MotionOutC(m.data_ptr(), pd.data_ptr())

    def motion(label):
        ms, st = [], _abi.StatsC()
        for r in range(REPS + 1):
            _abi.check(lib.rbrt_gpu_render_motion_device(h, cam.to_c(), cam.to_c(), out, stream.cuda_stream, st))
            if r:
                ms.append(st.ms_device)
        fin = torch.isfinite(m).all(-1)
        res[label] = {**stat(ms), "launches": st.launches, "rays": st.rays, "hit": round(float(fin.float().mean()), 4),
                      "moving": round(float((fin & (m != 0).any(-1)).float().mean()), 4)}

    motion("motion_static")
    base = torch.from_numpy(meshes[0][0].reshape(-1, 3, 3).copy()).cuda()
    scene.update_mesh_device(0, deform(base, 1), stream=stream)
    motion("motion_refit")

    hdr0, var0 = R.render_hdr_variance_device(cam, 16, scene, splits=4, seed=7, stream=stream)
    aov0 = R.render_aovs_device(cam, 4, scene, seed=7, passes=("depth", "normal", "ids"), stream=stream)
    t0 = R.temporal_accumulate_device(cam, hdr0, aov0, var=var0, stream=stream)
    hdr, var = R.render_hdr_variance_device(cam, 16, scene, splits=4, seed=8, stream=stream)
    aovs = R.render_aovs_device(cam, 4, scene, seed=8, passes=("depth", "normal", "ids"), stream=stream)
    torch.cuda.synchronize()
    g = lambda a: _abi.AovOutC(depth=a["depth"].data_ptr(), normal=a["normal"].data_ptr(), hit_kind=a["hit_kind"].data_ptr(),
                               elem_idx=a["elem_idx"].data_ptr())
    hist = _abi.TemporalHistoryC(cam=cam.to_c(), hdr=t0[0].data_ptr(), var=t0[1].data_ptr(), length=t0[2].data_ptr(), guides=g(aov0))
    o = [torch.empty((H, W, 3), dtype=torch.float32, device="cuda"), torch.empty((H, W, 3), dtype=torch.float32, device="cuda"),
         torch.empty((H, W), dtype=torch.float32, device="cuda")]
    for label in ("temporal_camera", "temporal_motion"):
        ms, st = [], _abi.StatsC()
        for r in range(REPS + 1):
            args = (W, H, cam.to_c(), hdr.data_ptr(), var.data_ptr(), g(aovs), hist)
            tail = (None, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), stream.cuda_stream, st)
            if label == "temporal_motion":
                _abi.check(lib.rbrt_gpu_temporal_accumulate_motion_device(*args, out, *tail))
            else:
                _abi.check(lib.rbrt_gpu_temporal_accumulate_device(*args, *tail))
            if r:
                ms.append(st.ms_device)
        res[label] = {**stat(ms), "history_kept": round(float((o[2] > 1).float().mean()), 4)}
    for k, v in res.items():
        if isinstance(v, dict):
            print(k, v, file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
