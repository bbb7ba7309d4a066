"""Animation on C3 (1920x1080, 64 spp, 2 groups in flight): per step a seeded deformation of the 1.31 M-triangle mesh, then one frame.
Four ways of getting the new geometry into the library:
  recreate      a new scene per step (upload + full LBVH build + a new block), from page-locked host memory;
  refit_host    rbrt_gpu_scene_update_mesh from page-locked host memory (H2D + refit);
  refit_device  rbrt_gpu_scene_update_mesh_device from a CUDA tensor (refit only);
  rebuild       rbrt_gpu_scene_update_mesh(..., RBRT_UPDATE_REBUILD) from page-locked host memory.
Reports ms per step (host clock over the timed steps, the last frame on the host), the time of one update alone on an otherwise idle
GPU (host clock around the call and a device synchronise; for the device path also CUDA events on its stream), node visits per
traversed ray after 1, 10 and 100 refit steps against a fresh build of the same geometry, and whether every path's last image equals
the recreate path's.  Writes one JSON line to stdout (and to OUT if given): python scripts/update_time.py [STEPS] [OUT]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import rbrt_b200 as R
from rbrt_b200 import _abi

STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
OUT = sys.argv[2] if len(sys.argv) > 2 else None
WARM = 2


def deform(base, k):
    """Step k of the animation, computed on the device: every vertex displaced by a travelling wave (seeded by k, deterministic)."""
    ph = 0.05 * k
    return (base + 0.6 * torch.sin(0.15 * base.roll(1, dims=-1) + ph)).contiguous()


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R.gpu_init(0)
    desc, W, H, spp = bench.WORKLOADS["c3"]
    spheres, meshes, camkw = bench.build_workload("c3")
    (tris0, mat), = meshes
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    base = torch.from_numpy(tris0).cuda()
    n = len(tris0)
    steps = range(WARM + STEPS)
    dev = [deform(base, k) for k in steps]                                # the device path's inputs
    host = [d.cpu().pin_memory() for d in dev]                            # the host paths' inputs (page-locked)
    torch.cuda.synchronize()
    lib = _abi.lib()
    res = {"gpu": gpu, "workload": desc, "steps": STEPS, "triangles": n, "modes": {}}
    last = {}
    for mode in ("recreate", "refit_host", "refit_device", "rebuild"):
        scene = bench.make_scene(spheres, [(host[0].numpy(), mat)])
        pipe = R.FramePipeline(W, H, depth=2, host_output=True)
        out = []
        t0 = None
        for k in steps:
            if k == WARM:
                out += pipe.drain()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            if mode == "recreate":
                scene = bench.make_scene(spheres, [(host[k].numpy(), mat)])
            elif mode == "refit_device":
                scene.update_mesh_device(0, dev[k])
            else:
                _abi.check(lib.rbrt_gpu_scene_update_mesh(scene.handle(), 0, host[k].data_ptr(), n, None,
                                                          _abi.UPDATE_REBUILD if mode == "rebuild" else _abi.UPDATE_REFIT))
            out += pipe.submit(cam, spp, scene, seed=k)
        out += pipe.drain()
        ms_step = (time.perf_counter() - t0) * 1e3 / STEPS
        last[mode] = out[-1][0].pixels
        # one update alone, on an otherwise idle GPU
        k = len(dev) - 1
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        ev = None
        if mode == "recreate":
            s2 = bench.make_scene(spheres, [(host[k].numpy(), mat)])
            s2.handle()
        elif mode == "refit_device":
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            scene.update_mesh_device(0, dev[k])
            e1.record()
            ev = e1
        else:
            _abi.check(lib.rbrt_gpu_scene_update_mesh(scene.handle(), 0, host[k].data_ptr(), n, None,
                                                      _abi.UPDATE_REBUILD if mode == "rebuild" else _abi.UPDATE_REFIT))
        torch.cuda.synchronize()
        ms_alone = (time.perf_counter() - t1) * 1e3
        r = {"ms_per_step": round(ms_step, 3), "ms_update_alone": round(ms_alone, 3)}
        if ev is not None:
            r["ms_update_alone_events"] = round(e0.elapsed_time(e1), 3)
        res["modes"][mode] = r
        print(mode, r, file=sys.stderr)
    res["last_image_equal_to_recreate"] = {m: bool(np.array_equal(last[m], last["recreate"])) for m in last}
    # tree quality: node visits per traversed ray after 1, 10, 100 refit steps of the animation, against a fresh build
    scene = bench.make_scene(spheres, [(tris0, mat)])
    scene.handle()
    q = {}
    for k in range(1, 101):
        d = deform(base, k)
        scene.update_mesh_device(0, d)
        if k in (1, 10, 100):
            st, sf = {}, {}
            R.render_scene(cam, 4, scene, stats=st, seed=1, count_visits=True)
            fresh = bench.make_scene(spheres, [(d.cpu().numpy(), mat)])
            R.render_scene(cam, 4, fresh, stats=sf, seed=1, count_visits=True)
            q[k] = {"refit": round(st["node_visits"] / st["traversed_rays"], 3), "fresh": round(sf["node_visits"] / sf["traversed_rays"], 3),
                    "same_rays": st["rays"] == sf["rays"]}
            fresh.close()
            print("visits per traversed ray after", k, q[k], file=sys.stderr)
    res["visits_per_traversed_ray"] = q
    line = json.dumps(res)
    print(line)
    if OUT:
        os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
        with open(OUT, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
