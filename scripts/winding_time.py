"""Winding numbers (rbrt_gpu_query_winding_device) on C3 (1.31 M triangles + 4 spheres), 2^21 points per set:
  - near: points on the sphere mesh's triangles offset along their normals by up to 1 % of the radius (40), either side;
  - box:  points uniform in the mesh's exact box;
at beta = 2 (the default).  For each set: device time from CUDA events around the call (both planes, no stats), the median of REPS after
a warm-up, points per second, and node visits and triangle terms per point (one extra call with stats).  beta = +inf (the exact sum over
all 1.31 M triangles per point) is timed on the first SUB near points only.  The moments: the first call after an update recomputes them,
so the time of k_wind_moments is the device time of such a call minus that of a call on fresh moments (SUB points each), and the moment
block's bytes are the device memory the first call of the scene allocated (torch.cuda.mem_get_info before and after).  The card's name,
power limit and SM clocks are read in the same run.
Writes one JSON line to stdout (and to OUT if given): python scripts/winding_time.py [OUT] [REPS]"""
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
N = 1 << 21
SUB = 1024


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
    scene.info()                                                            # the build has finished
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

    w = torch.empty(N, dtype=torch.float32, device="cuda")
    ins = torch.empty(N, dtype=torch.uint8, device="cuda")
    out = _abi.WindingOutC(winding=w.data_ptr(), inside=ins.data_ptr())
    tn = torch.from_numpy(near).cuda()

    def call(tp, n, beta, st=None):
        _abi.check(lib.rbrt_gpu_query_winding_device(h, tp.data_ptr(), n, _abi.WindingOptsC(beta), out, stream.cuda_stream, st))

    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    call(tn, SUB, 2.0)                                                      # allocates the moment block and computes the moments
    torch.cuda.synchronize()
    block_bytes = free0 - torch.cuda.mem_get_info()[0]
    res = {"workload": desc, "points": N, "reps": REPS, "beta": 2.0, "sets": {}, "moment_block_bytes_allocated": block_bytes}
    for name, pts in (("near", near), ("box", box)):
        tp = torch.from_numpy(pts).cuda()
        call(tp, N, 2.0)
        torch.cuda.synchronize()
        ms = statistics.median(timed(lambda: call(tp, N, 2.0), stream) for _ in range(REPS))
        st = _abi.StatsC()
        call(tp, N, 2.0, st)
        res["sets"][name] = {"ms_device": round(ms, 4), "points_per_s": round(N / (ms * 1e-3)), "node_visits_per_point": round(st.node_visits / N, 2),
                             "tri_terms_per_point": round(st.tri_tests / N, 2), "inside": int(ins.sum().item())}
    # beta = +inf on SUB near points
    call(tn, SUB, float("inf"))
    torch.cuda.synchronize()
    ms = statistics.median(timed(lambda: call(tn, SUB, float("inf")), stream) for _ in range(3))
    st = _abi.StatsC()
    call(tn, SUB, float("inf"), st)
    res["exact_sub"] = {"points": SUB, "ms_device": round(ms, 3), "points_per_s": round(SUB / (ms * 1e-3), 1),
                        "tri_terms_per_point": round(st.tri_tests / SUB, 1)}
    # k_wind_moments: a call behind a refit (same vertices) against a call on fresh moments
    verts = torch.from_numpy(tris.copy()).cuda()
    fresh, stale = [], []
    for _ in range(REPS):
        fresh.append(timed(lambda: call(tn, SUB, 2.0), stream))
        scene.update_mesh_device(0, verts)
        torch.cuda.synchronize()
        stale.append(timed(lambda: call(tn, SUB, 2.0), stream))
    res["moments"] = {"triangles": int(scene.info()["num_triangles_tested"]), "ms_call_with_recompute": round(statistics.median(stale), 4),
                      "ms_call_on_fresh_moments": round(statistics.median(fresh), 4),
                      "ms_k_wind_moments": round(statistics.median(stale) - statistics.median(fresh), 4)}
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
