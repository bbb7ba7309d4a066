"""Nearest-surface queries (rbrt_gpu_query_nearest_device) on C3 (1.31 M triangles + 4 spheres), 2^21 points per set:
  - near: points on the sphere mesh's triangles offset along their normals by up to 1 % of the radius (40), either side;
  - box:  points uniform in the scene's box (the mesh's exact box, which holds the four spheres' nearest parts);
each without a bound (max_dist NULL) and with max_dist = 1 % of the radius (0.4) for every point.
For each set: device time from CUDA events around the call (all seven planes, no stats), the median of REPS after a warm-up, points per
second, and node visits and triangle tests per point (one extra call with stats).  As a yardstick, the brute force of tests/point_ref.py
in torch on the same GPU (every point against every candidate, one elementwise kernel per f32 operation) is timed on the first SUB points
of the near set.  The card's name, power limit and SM clocks are read in the same run.
Writes one JSON line to stdout (and to OUT if given): python scripts/point_time.py [OUT] [REPS]"""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import rbrt_b200 as R
from rbrt_b200 import _abi
from tests import point_ref as P

OUT = sys.argv[1] if len(sys.argv) > 1 else None
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 10
N = 1 << 21
SUB = 256


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
    desc = bench.WORKLOADS["c3"][0]
    spheres, meshes, _ = bench.build_workload("c3")
    scene = bench.make_scene(spheres, meshes)
    lib = _abi.lib()
    h = scene.handle()
    stream = torch.cuda.current_stream()
    gpu_before = smi()

    tris = np.asarray(scene.triangle_meshes[0].triangles, np.float32)
    rng = np.random.default_rng(5)
    k = rng.integers(0, len(tris), N)
    a, b = rng.random(N), rng.random(N)
    flip = a + b > 1
    a[flip], b[flip] = 1 - a[flip], 1 - b[flip]
    t = tris[k].astype(np.float64)
    on = t[:, 0] + a[:, None] * (t[:, 1] - t[:, 0]) + b[:, None] * (t[:, 2] - t[:, 0])
    nrm = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    radius = 40.0
    near = (on + nrm * rng.uniform(-0.01, 0.01, N)[:, None] * radius).astype(np.float32)
    lo, hi = tris.reshape(-1, 3).min(0), tris.reshape(-1, 3).max(0)
    box = (lo + rng.random((N, 3)) * (hi - lo)).astype(np.float32)

    res = {"workload": desc, "points": N, "reps": REPS, "sets": {}}
    planes = {"dist": (N,), "kind": (N,), "elem_idx": (N,), "tri_idx": (N,), "point": (N, 3), "normal": (N, 3), "uv": (N, 2)}
    bufs = {k: torch.empty(s, dtype=torch.float32, device="cuda") for k, s in planes.items()}
    out = _abi.NearestOutC(**{k: v.data_ptr() for k, v in bufs.items()})
    md = torch.full((N,), 0.01 * radius, dtype=torch.float32, device="cuda")
    for name, pts in (("near", near), ("box", box)):
        tp = torch.from_numpy(pts).cuda()
        for bound in ("none", "max_dist_0.4"):
            mdp = md.data_ptr() if bound != "none" else None

            def call():
                _abi.check(lib.rbrt_gpu_query_nearest_device(h, tp.data_ptr(), N, mdp, out, stream.cuda_stream, None))
            call()
            torch.cuda.synchronize()
            ms = statistics.median(timed(call, stream) for _ in range(REPS))
            st = _abi.StatsC()
            _abi.check(lib.rbrt_gpu_query_nearest_device(h, tp.data_ptr(), N, mdp, out, stream.cuda_stream, st))
            hits = int((bufs["kind"].view(torch.int32) != _abi.HIT_NONE).sum().item())
            res["sets"][f"{name}/{bound}"] = {"ms_device": round(ms, 4), "points_per_s": round(N / (ms * 1e-3)),
                                              "node_visits_per_point": round(st.node_visits / N, 2), "tri_tests_per_point": round(st.tri_tests / N, 2),
                                              "found": hits}
    # the brute-force yardstick on SUB near points
    cand = P.candidates(scene)
    P.nearest(cand, near[:8], X=P.TORCH)                                    # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bf = P.nearest(cand, near[:SUB], X=P.TORCH)
    torch.cuda.synchronize()
    bf_ms = (time.perf_counter() - t0) * 1e3
    tp = torch.from_numpy(near).cuda()
    _abi.check(lib.rbrt_gpu_query_nearest_device(h, tp.data_ptr(), N, None, out, stream.cuda_stream, None))
    same = bool(np.array_equal(bufs["dist"][:SUB].cpu().numpy().view(np.uint32), bf["dist"].view(np.uint32)))
    res["torch_brute_force"] = {"points": SUB, "candidates": len(cand["rec"]), "ms": round(bf_ms, 1), "points_per_s": round(SUB / (bf_ms * 1e-3), 1),
                                "dist_bit_identical_to_the_kernel": same}
    res["gpu"] = smi()
    res["gpu_before"] = gpu_before
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
