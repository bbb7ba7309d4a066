"""Ray queries on device memory against the parity hook on C3 (1920x1080, 1.31 M triangles + 4 spheres), on the same rays:
  - camera rays: rbrt_gpu_primary_rays (seed 7, sample 0);
  - bounce-like rays: origins on the camera rays' first hits, directions uniform on the sphere (numpy seed 11), incoherent.
For each set:
  - the closest-hit query (k_query, warp-voted traversal, shared-memory stack; rbrt_gpu_query_closest_device, all seven planes, no stats)
    against k_trace_rays (one lane per ray, local-memory stack; rbrt_gpu_trace_rays' stats.ms_device, which counts visits as it runs),
    alternating in one process: device time from CUDA events around each call, the median of REPS after a warm-up of each;
  - the occlusion query with max_dist = the first hit's dist and = +inf, against the closest query;
  - node visits and triangle tests per ray from each kernel's counters (one extra call with stats).
The rays and the planes stay on the device; the calls repeat on the same scene, so the tree and triangle records (about 100 MB) are mostly
in the 126 MB L2 after the first call.  The card's name, power limit and SM clocks are read in the same run.
Writes one JSON line to stdout (and to OUT if given): python scripts/query_time.py [OUT] [REPS]"""
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


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()[0]


def timed(fn, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    R.gpu_init(0)
    desc, W, H, _ = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    lib = _abi.lib()
    h = scene.handle()
    stream = torch.cuda.current_stream()
    gpu_before = smi()

    cam_rays = R.primary_rays(cam, 7, 0)
    first = scene.hit(cam_rays)
    hit = first["kind"] != _abi.HIT_NONE
    rng = np.random.default_rng(11)
    d = rng.normal(size=(int(hit.sum()), 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    bounce = np.concatenate([first["point"][hit], d], 1).astype(np.float32)
    bounce_first = scene.hit(bounce)

    res = {"workload": desc, "reps": REPS, "sets": {}}
    for name, rays, hits in (("camera", cam_rays, first), ("bounce", bounce, bounce_first)):
        n = len(rays)
        t_rays = torch.from_numpy(rays).cuda()
        planes = {k: torch.empty(n * (3 if k in ("point", "normal") else 1), dtype=torch.float32, device="cuda")
                  for k in ("t", "dist", "kind", "elem_idx", "tri_idx", "point", "normal")}
        out = _abi.QueryOutC(**{k: p.data_ptr() for k, p in planes.items()})
        md_hit = torch.from_numpy(np.where(hits["kind"] != _abi.HIT_NONE, hits["dist"], np.float32(np.inf)).astype(np.float32)).cuda()
        occ = torch.empty(n, dtype=torch.uint8, device="cuda")
        host_hits = np.zeros(n, dtype=_abi.HIT_DTYPE)

        def closest():
            _abi.check(lib.rbrt_gpu_query_closest_device(h, t_rays.data_ptr(), n, out, stream.cuda_stream, None))

        def occluded(md):
            return lambda: _abi.check(lib.rbrt_gpu_query_occluded_device(h, t_rays.data_ptr(), n, md, occ.data_ptr(), stream.cuda_stream, None))

        def trace_rays():
            st = _abi.StatsC()
            _abi.check(lib.rbrt_gpu_trace_rays(h, rays.ctypes.data, n, _abi.TRACE_BVH, host_hits.ctypes.data, st))
            return st.ms_device

        arms = {"query_closest": lambda: timed(closest, stream), "trace_rays_k_trace_rays": trace_rays,
                "query_occluded_at_hit_dist": lambda: timed(occluded(md_hit.data_ptr()), stream),
                "query_occluded_inf": lambda: timed(occluded(None), stream)}
        ms = {k: [] for k in arms}
        for r in range(REPS + 1):                                         # alternating; the first round is the warm-up
            for k, f in arms.items():
                v = f()
                if r:
                    ms[k].append(v)
        counts = {}
        for k, call in (("query_closest", lambda st: lib.rbrt_gpu_query_closest_device(h, t_rays.data_ptr(), n, out, stream.cuda_stream, st)),
                        ("query_occluded_at_hit_dist", lambda st: lib.rbrt_gpu_query_occluded_device(h, t_rays.data_ptr(), n, md_hit.data_ptr(),
                                                                                                    occ.data_ptr(), stream.cuda_stream, st)),
                        ("query_occluded_inf", lambda st: lib.rbrt_gpu_query_occluded_device(h, t_rays.data_ptr(), n, None, occ.data_ptr(),
                                                                                            stream.cuda_stream, st)),
                        ("trace_rays_k_trace_rays", lambda st: lib.rbrt_gpu_trace_rays(h, rays.ctypes.data, n, _abi.TRACE_BVH, host_hits.ctypes.data, st))):
            st = _abi.StatsC()
            _abi.check(call(st))
            counts[k] = (st.node_visits / n, st.tri_tests / n, st.ms_device)
        entry = {"rays": n, "hit_share": round(float((hits["kind"] != _abi.HIT_NONE).mean()), 4)}
        for k in arms:
            med = statistics.median(ms[k])
            entry[k] = {"ms_device": round(med, 4), "ms_min": round(min(ms[k]), 4), "ms_max": round(max(ms[k]), 4),
                        "grays_per_s": round(n / med / 1e6, 3), "node_visits_per_ray": round(counts[k][0], 3),
                        "tri_tests_per_ray": round(counts[k][1], 3), "ms_device_with_counters": round(counts[k][2], 4)}
        entry["closest_speedup_vs_trace_rays"] = round(entry["trace_rays_k_trace_rays"]["ms_device"] / entry["query_closest"]["ms_device"], 3)
        # the planes of the timed calls are the parity hook's records
        got = planes["dist"].cpu().numpy()
        entry["closest_dist_bit_identical"] = bool(np.array_equal(got.view(np.uint32), host_hits["dist"].view(np.uint32)))
        res["sets"][name] = entry
        print(name, json.dumps(entry), file=sys.stderr)
    res["gpu_before"], res["gpu_after"] = gpu_before, smi()
    res["gpu_fields"] = "name, power.limit, clocks.sm, clocks.max.sm"
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
