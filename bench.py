#!/usr/bin/env python
"""bench.py — the headline benchmark of BASELINE.json: Mrays/s (and samples/s) of the path-tracing hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c1|c4] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is ONE render of the whole frame of the workload (all pixels x all samples, up to 51 ray segments per
path) — the reference's `render_scene(cam, spp, scene)` (lib.rs:75-124).  Rays = closest-hit queries
(`Scene::hit` calls, primary + bounces), counted on the device.

  value      whole-job Mrays/s with the scene (SoA buffers + LBVH) already resident in HBM; the timed region is
             K x collective render_scene (shard render -> per-GPU finalise (1/spp, sqrt, x256, saturating u8) -> gather on rank 0,
             all inside librbrt_gpu.so), with --frames-in-flight groups (default 2) of --frames-per-batch frames (default 4, THE SAME
             at every N) in flight on their own streams (rbrt_b200.FramePipeline): the sparse, latency-bound last bounces of one
             group overlap the dense first bounces of the next.  Every timed arm runs exactly K steps after its warm-up.
             `single_frame` is one frame at a time, `frames_per_batch_1` the pipelined figure with one frame per batch.  The last
             pipelined image is checked against the single-frame one; --dump-outputs DIR writes it as DIR/image.npy (float32,
             H x W x 3, values 0..255; above 64 MB a fixed seeded pixel sample, image_sample.npy + image_sample_index.npy).
  e2e        the same metric through the reference-facing call with HOST buffers: every step uploads the
             triangle soup from pinned host memory (rbrt_gpu_scene_create: H2D + LBVH build on rank 0, NCCL broadcast of the
             scene block to the other ranks), renders and copies the RGB8 image back to the host.
  roofline   the trace kernel (BVH traversal + intersection tests): algorithmic bytes per step from an
             instrumented counting pass (64 B per node visit, 48 B per triangle test, 64 B of queue / path-record traffic per
             traversed ray) / the summed CUDA-event durations of that kernel's launches, against the measured HBM copy
             bandwidth (MEASURED_PEAKS.json); `traffic` / `dram_frac` / `ncu` from the committed ncu capture for this N.
  image_check at EVERY N: the collective render vs the CPU oracle on a pixel lattice (bit-identical expected).
  cpu_baseline / --impl reference
             the CPU oracle (C++/AVX restatement of the reference; the Rust reference cannot be built here) on all
             host threads, on a bounded stratified pixel sample of the same workload.  That arm never loads librbrt_gpu.so.

Multi-GPU: one process per GPU (torchrun); torch.distributed only carries the NCCL unique id to the library
(rbrt_b200.dist.init_comm); sharding by interleaved 8x4-pixel tiles (fixed total work => "strong" scaling), gather and scene
broadcast run inside librbrt_gpu.so (csrc/multi.cu).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (description, width, height, spp)
    "c1": ("C1: spheres-only scene of scenes/example_scene.yaml (mesh removed), 256x192, 8 spp", 256, 192, 8),
    "c2": ("C2: scenes/example_scene.yaml with an 81920-triangle displaced icosphere (.obj) for bunny.obj, 1024x768, 50 spp", 1024, 768, 50),
    "c3": ("C3: 1310720-triangle displaced icosphere (radius 40) + 4 spheres, 1920x1080, 64 spp, tile-sharded", 1920, 1080, 64),
    "c4": ("C4: dielectric/metal-heavy scene (36 glass/metal spheres + 20480-triangle glass mesh), depth 50, 1024x768, 256 spp", 1024, 768, 256),
    "c5": ("C5: 5242880-triangle displaced icosphere (radius 100) + 4 spheres, 3840x2160, 1024 spp, sample-range sharded + NCCL reduce", 3840, 2160, 1024),
}
SAMPLE_SHARDED = {"c5"}
SEED = 0x5EED
_STDOUT = sys.stdout


def build_workload(name, pinned=False):
    """Returns (spheres [(center, radius, material)], [(triangles [N,3,3] f32, material)], camera kwargs)."""
    import rbrt_b200 as R
    from rbrt_b200 import synth
    from rbrt_b200.vec3 import Vec3

    _, W, H, spp = WORKLOADS[name]
    excam = synth.EXAMPLE_CAMERA
    cam_ex = dict(position=Vec3(*excam["camera_position"]), look_at=Vec3(*excam["camera_look_at"]), up=Vec3(*excam["camera_up"]),
                  focal_len_mm=excam["camera_focal_length_mm"])
    if name == "c1":
        bp = synth.spheres_only_blueprint()
        sc = R.create_scene_from_scene_blueprint(bp)
        return [(s.center, s.radius, s.material) for s in sc.elements], [], cam_ex
    if name == "c2":
        obj = os.path.join(synth.cache_dir(), "standin6.obj")
        if not os.path.exists(obj):
            synth.write_bunny_standin(obj, 6)
        sc = R.create_scene_from_scene_blueprint(synth.example_scene_blueprint(obj))
        return ([(s.center, s.radius, s.material) for s in sc.elements],
                [(m.triangles, m.material) for m in sc.triangle_meshes], cam_ex)
    if name == "c3":
        cam, spheres, tris, mat = synth.big_mesh_config(8, 40.0)
        return spheres, [(tris, mat)], cam
    if name == "c5":
        cam, spheres, tris, mat = synth.big_mesh_config(9, 100.0)
        return spheres, [(tris, mat)], cam
    if name == "c4":
        spheres, tris, mat = synth.stress_config()
        return spheres, [(tris, mat)], cam_ex
    raise SystemExit(f"unknown workload {name}")


def make_scene(spheres, meshes, pinned_cache=None, broadcast=False):
    import rbrt_b200 as R
    sc = R.Scene(broadcast=broadcast)
    sc.elements += [R.Sphere(c, r, m) for c, r, m in spheres]
    for i, (tris, mat) in enumerate(meshes):
        if pinned_cache is not None:
            tris = pinned_cache[i]
        sc.triangle_meshes.append(R.TriangleMesh.from_triangles(tris, mat))
    return sc


def pin_meshes(meshes):
    """Copies of the triangle arrays in page-locked host memory (the e2e leg uploads from these)."""
    import torch
    out, keep = [], []
    for tris, _ in meshes:
        t = torch.empty(tris.shape, dtype=torch.float32, pin_memory=True)
        t.numpy()[...] = tris
        keep.append(t)
        out.append(t.numpy())
    return out, keep


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, image):
    """The RGB8 image of the last timed step as out_dir/image.npy (float32 [H, W, 3], values 0..255, exact).  An image above
    DUMP_BYTES as float32 is written as a fixed sample of 2^21 pixels drawn with SEED: image_sample.npy (float32 [n, 3]) and
    image_sample_index.npy (float64 [n], the flat pixel index y * W + x, ascending)."""
    os.makedirs(out_dir, exist_ok=True)
    px = image.astype(np.float32)
    if px.nbytes <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "image.npy"), px)
        return
    px = px.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(SEED).choice(len(px), 1 << 21, replace=False))
    np.save(os.path.join(out_dir, "image_sample.npy"), px[idx])
    np.save(os.path.join(out_dir, "image_sample_index.npy"), idx.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU (B200_PROFILING.md).  nvidia-smi needs a few hundred ms before its first
    sample, longer than a whole timed region of this benchmark, so the sampler is started BEFORE the warm-up steps and the
    samples are filtered by their timestamps: those inside [mark_begin, mark_end] (the timed region, padded by one sampling
    period) are used; if the region was too short to catch any, the samples of the warm-up steps (same load) are used and
    `window` says so."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 20

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t_begin, self.t_end, self.t_start = index, None, [], None, None, time.time()

    def __enter__(self):
        if os.environ.get("RBRT_BENCH_NO_CLOCKS"):            # debugging aid: measure without the nvidia-smi side process
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.PERIOD_MS)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def __exit__(self, *a):
        if self.proc:
            time.sleep(2.5 * self.PERIOD_MS / 1e3)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        import datetime
        rows = []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                vals = (float(f[1]), float(f[2]), float(f[3]))
            except ValueError:
                continue
            ts = None
            for fmt in ("%Y/%m/%d %H:%M:%S.%f", "%Y-%m-%d %H:%M:%S.%f", "%Y/%m/%d %H:%M:%S"):
                try:
                    ts = datetime.datetime.strptime(f[0], fmt).timestamp()
                    break
                except ValueError:
                    pass
            rows.append((ts if ts is not None else (self.t_begin or 0.0), *vals, f[4:8]))
        pad = self.PERIOD_MS / 1e3
        inside = [r for r in rows if self.t_begin is not None and self.t_begin - pad <= r[0] <= (self.t_end or time.time()) + pad]
        window = "timed region"
        if not inside:
            inside = [r for r in rows if r[0] <= (self.t_end or time.time()) + pad]
            window = "warm-up + timed region (timed region shorter than the sampling period)"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": max(r[2] for r in inside), "reasons": sorted(reasons),
                "samples": len(inside), "power_w_max": max(r[3] for r in inside), "window": window}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(st, n_spheres, n_meshes):
    """Trace kernel (stage B: LBVH traversal of the rays that entered a mesh AABB), DESIGN.md section 4:
    bytes/step = 64 V + 48 T + 64 C   (V node visits x 64-B node, T triangle tests x 48-B record, C traversed rays x
    64 B of queue / path-record traffic: 4 B queue index + the 32-byte path record read; the 32-byte pending-hit record (or
    16 B of radiance on a miss) + 4 B material-queue index written — up to 72 B, still charged as the 64 B of the earlier
    40 + 16-byte record so that the figure stays comparable and conservative).  The sphere and mesh-AABB tests of SURVEY.md section 8(d)
    (16 S + 24 M per ray) run in the producing kernels (k_generate / k_shade) and are not charged to this kernel."""
    return 64 * st["node_visits"] + 48 * st["tri_tests"] + 64 * st["traversed_rays"]      # counts of k_trace only (tail kernel subtracted by the caller)


def algorithmic_flops(st, n_spheres, n_meshes):
    """SURVEY.md section 8(d) restated for the 4-wide node: four slab tests of 12 flops (6 FMA) + 12 min/max each = 96 per node
    visit; 46 per Moeller-Trumbore test (triangle.rs:189-234)."""
    return 96 * st["node_visits"] + 46 * st["tri_tests"]


# ------------------------------------------------------------------------------------------- CPU legs
def oracle_scene(spheres, meshes):
    from oracle import oracle_ffi as O
    import rbrt_b200 as R
    els = [R.Sphere(c, r, m) for c, r, m in spheres]
    ms = [R.TriangleMesh.from_triangles(t, m) for t, m in meshes]
    return O, O.OracleScene(els, ms, 8)


def oracle_camera(O, camkw, H, W):
    """Camera::new (cam.rs:22-62) computed by the ORACLE (the reference arm never touches the product library)."""
    return O.camera_new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])


def choose_stride(O, osc, cam_c, spp_full, target_s):
    """Pick a pixel lattice (stride, stride) and a sample count so that one oracle pass takes about target_s."""
    from rbrt_b200 import _abi
    W, H = cam_c.img_width_pix, cam_c.img_height_pix
    stride = max(1, int(max(W, H) // 24))
    st, _ = O.render_subset(osc, cam_c, 1, stride, stride, _abi.RenderOptsC(seed=SEED))
    per_path = max(st["ms_total"], 1e-3) / 1e3 / max(st["paths"], 1)
    paths = max(1.0, target_s / per_path)
    full_px = W * H
    if paths >= full_px * spp_full:
        return 1, spp_full
    if paths >= full_px:
        return 1, max(1, int(paths // full_px))
    s = int(np.ceil(np.sqrt(full_px / paths)))
    return max(1, s), 1


def cpu_leg(O, osc, cam_c, stride, spp, want_image=False):
    from rbrt_b200 import _abi
    st, acc = O.render_subset(osc, cam_c, spp, stride, stride, _abi.RenderOptsC(seed=SEED), want_image=want_image)
    return (st, acc) if want_image else st


def product_lib_loaded():
    try:
        return "librbrt_gpu" in open("/proc/self/maps").read()
    except OSError:
        return None


def run_reference(args):
    """--impl reference: the oracle on all host threads, each step a bounded stratified sample of the workload.  The product
    library (librbrt_gpu.so) is never loaded in this arm: camera and vertex transform come from the oracle's own twins."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle_ffi as O
    import rbrt_b200.mesh as M

    def oracle_transform(ptr, n_vertices, scale, rot_c, tr_c):
        O.check(O.lib().rbrt_ref_transform_vertices(ptr, n_vertices, scale, rot_c, tr_c))
    M._transform_in_place = oracle_transform
    M._load_obj_soup = M.load_obj_soup_python                             # the product's loader is in librbrt_gpu.so
    desc, W, H, spp = WORKLOADS[args.workload]
    spheres, meshes, camkw = build_workload(args.workload)
    O, osc = oracle_scene(spheres, meshes)
    cam_c = oracle_camera(O, camkw, H, W)
    cores = O.lib().rbrt_ref_hardware_threads()
    budget = 150.0 / max(1, args.steps + args.warmup)
    stride, s_spp = choose_stride(O, osc, cam_c, spp, min(8.0, budget))
    for _ in range(args.warmup):
        cpu_leg(O, osc, cam_c, stride, s_spp)
    t0 = time.perf_counter()
    rays = paths = 0
    for _ in range(args.steps):
        st = cpu_leg(O, osc, cam_c, stride, s_spp)
        rays += st["rays"]; paths += st["paths"]
    dt = time.perf_counter() - t0
    val = rays / dt / 1e6
    sample = f"pixel lattice stride {stride}x{stride} of the {W}x{H} frame, {s_spp} of {spp} spp: {paths // max(1, args.steps)} paths/step"
    line = {"impl": "reference", "metric": "Mrays/s", "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "samples_per_s": paths / dt,
            "config": workload_config(args.workload, spheres, meshes, args.gpus),
            "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": int(cores), "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "product_lib_loaded": product_lib_loaded(),
            "note": "CPU oracle (C++/AVX restatement; rustc/cargo absent so the Rust reference cannot be built); full-frame time is "
                    "extrapolated only in DESIGN.md, this value is measured rays / measured seconds on the sample"}
    print(json.dumps(line), file=_STDOUT, flush=True)
    return 0


def workload_config(name, spheres, meshes, n_gpus):
    desc, W, H, spp = WORKLOADS[name]
    return {"workload": desc, "width": W, "height": H, "spp": spp, "max_depth": 50, "spheres": len(spheres),
            "triangles": int(sum(len(t) for t, _ in meshes)), "seed": SEED,
            "sharding": "none" if n_gpus == 1 else (f"sample ranges over {n_gpus} ranks + one NCCL reduce (sum) of the f32 accumulators, inside librbrt_gpu.so" if name in SAMPLE_SHARDED
                                                    else f"interleaved 8x4-pixel tiles over {n_gpus} ranks, every rank finalises its own pixels, NCCL gather of 3 B/pixel on rank 0, inside librbrt_gpu.so"),
            "l2_policy": "no explicit flush: per step the wavefront streams >400 MB of ray/hit queues and the scene (nodes+triangles+normals) "
                         "is larger than or comparable to L2; inputs larger than L2"}


def ncu_evidence(workload, world):
    """What ncu measured for the dominant kernel, from the COMMITTED summary profiles/r2_ncu_summary.json (written by
    scripts/ncu_summary.py from the raw CSVs next to it; the file names the exact ncu command).  Keyed by workload and by the tile-shard
    denominator N (one GPU rendering 1/N of the frame = what one rank of N renders).  None when no capture exists for this (workload, N)."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_summary.json")
    if not os.path.exists(p):
        return None
    try:
        d = json.load(open(p))
        e = d.get(workload, {}).get(str(world))
        if e is not None:
            e = dict(e, source="profiles/r2_ncu_summary.json", command=d.get("command"))
        return e
    except (ValueError, OSError):
        return None


# ------------------------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import ctypes as C

    import torch
    import torch.distributed as dist

    import rbrt_b200 as R
    from rbrt_b200 import _abi
    from rbrt_b200 import dist as D
    from rbrt_b200.render import make_opts

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run --nproc-per-node N (one process per GPU)")
        args.gpus = world
    torch.cuda.set_device(local)
    R.gpu_init(local)
    comm = {"active": 0, "transport": 0, "nccl_version": 0}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        comm = D.init_comm(dist)                               # the library's own NCCL communicator (torch only carries the unique id)
        assert comm["active"] and comm["world"] == world and comm["rank"] == rank
    lib = _abi.lib()
    desc, W, H, spp = WORKLOADS[args.workload]
    spheres, meshes, camkw = build_workload(args.workload)
    cam = R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])
    cam_c = cam.to_c()
    scene = make_scene(spheres, meshes)                        # under the communicator: rank 0 uploads + builds, the block is broadcast
    info = scene.info()
    stream = torch.cuda.current_stream()
    rgb = torch.empty(H * W * 3, dtype=torch.uint8, device="cuda")
    shard_mode = _abi.SHARD_SAMPLES if args.workload in SAMPLE_SHARDED else _abi.SHARD_TILES
    mode_kw = dict(shard_mode=shard_mode) if world > 1 else {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cams1 = (_abi.CameraC * 1)(cam_c)
    seeds1 = (C.c_uint64 * 1)(SEED)
    rgb1 = (C.c_void_p * 1)(rgb.data_ptr())

    def step_single(flags_kw, st, n_spp=spp, out=rgb1, hdr=None):
        """ONE collective render_scene: shard render -> per-GPU finalise -> gather on rank 0 (rbrt_gpu_render_frames_device);
        with st it waits for the frame."""
        _abi.check(lib.rbrt_gpu_render_frames_device(scene.handle(), cams1, seeds1, 1, n_spp, make_opts(seed=SEED, **mode_kw, **flags_kw),
                                                     out, hdr, stream.cuda_stream, st))

    # ---- counting pass (untimed): node visits / triangle tests per step, identical every step (fixed seed)
    cst = _abi.StatsC()
    step_single(dict(count_visits=True), cst)
    barrier()
    counts = cst.as_dict()

    # ---- single-frame pass: one frame at a time (host waits for each), every trace launch bracketed by CUDA events.
    #      Gives the per-frame counters (identical every frame: fixed seed), the un-overlapped kernel times the roofline
    #      is computed from, and the reference image the pipelined frames are checked against.
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats = []
    for _ in range(max(args.warmup, 3)):
        step_single(dict(time_kernels=True), _abi.StatsC())
    barrier()
    n_single = args.steps
    single_ms = []
    for _ in range(n_single):
        st = _abi.StatsC()
        e0.record(stream)
        step_single(dict(time_kernels=True), st)
        e1.record(stream)
        barrier()
        single_ms.append(e0.elapsed_time(e1))
        stats.append(st.as_dict())
    ms_single_one_lane = statistics.median(single_ms)
    rgb_ref = rgb.clone() if rank == 0 else None
    # the lone frame as rbrt_gpu_render issues it: its sample batches on two lanes (RBRT_OPT_SPLIT_BATCHES), so that the sparse end of
    # one batch runs under the dense start of the next
    use_split = (W * H * spp) // world >= (1 << 26)          # rbrt_gpu_render's own rule: two lanes from 2^26 paths per GPU
    single_ms = []
    for k in range(3 + n_single):
        e0.record(stream)
        step_single(dict(split=use_split), _abi.StatsC())
        e1.record(stream)
        barrier()
        if k >= 3:
            single_ms.append(e0.elapsed_time(e1))
    ms_single = statistics.median(single_ms)
    if rank == 0 and not os.environ.get("RBRT_DEBUG_NO_GATHER"):
        assert torch.equal(rgb, rgb_ref), "two-lane frame differs from the one-lane frame"
    frame = stats[-1]
    assert all(s_["rays"] == frame["rays"] and s_["paths"] == frame["paths"] for s_ in stats), "frames of one seed differ"

    # ---- resident arm (timed region): `steps` frames through the FramePipeline, `frames_in_flight` groups in flight on their own
    #      streams and wavefront pools, `frames_per_batch` frames per group — THE SAME at every N (a rank's launches on 8 GPUs
    #      then have about the size they have on one GPU with one frame).  The region is bracketed by barrier + synchronize.
    # 4 frames per batch at every N — unless ONE frame of the workload already fills a wavefront pool (2^27 paths: C4, C5), where
    # batching frames only cuts each frame's samples into more, smaller batches (measured on C4: 59.1 ms with 4, 52.0 with 1)
    fpb = args.frames_per_batch or (1 if (args.workload in SAMPLE_SHARDED or W * H * spp > (1 << 27)) else 4)

    def timed_pipeline(fpb_):
        pipe = R.FramePipeline(W, H, depth=args.frames_in_flight, host_output=False, shard_mode=shard_mode, frames_per_batch=fpb_)
        for _ in range(max(args.warmup, 3) * fpb_):
            pipe.submit(cam_c, spp, scene, seed=SEED)
        pipe.drain()
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            pipe.submit(cam_c, spp, scene, seed=SEED)
        pipe.flush()                                          # a last, partially filled group of frames
        pipe.wait_on(stream)
        e1.record(stream)
        last = pipe.drain()[-1][0]
        barrier()
        return e0.elapsed_time(e1), last

    with ClockSampler(local) as clk:
        time.sleep(0.3)                                       # let nvidia-smi deliver its first samples
        clk.mark_begin()
        ms, last = timed_pipeline(fpb)
        clk.mark_end()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last.cpu().numpy().reshape(H, W, 3))
    check_images = not os.environ.get("RBRT_DEBUG_NO_GATHER")   # (a timing experiment of csrc/multi.cu that leaves rank 0's image incomplete)
    if rank == 0 and check_images:
        assert torch.equal(last, rgb_ref), "pipelined frame differs from the single-frame render"
    ms_fpb1 = None
    if fpb != 1:                                              # the same measurement with ONE frame per batch, for the record
        ms_fpb1, last1 = timed_pipeline(1)
        if rank == 0 and check_images:
            assert torch.equal(last1, rgb_ref), "pipelined frame (1 per batch) differs from the single-frame render"
    t = torch.tensor([ms, ms_single, ms_fpb1 or 0.0, ms_single_one_lane], dtype=torch.float64, device="cuda")
    agg = torch.tensor([frame["rays"] * args.steps, frame["paths"] * args.steps, (frame["launches"]) * args.steps,
                        counts["node_visits"] - counts["tail_node_visits"], counts["tri_tests"] - counts["tail_tri_tests"], counts["rays"],
                        counts["traversed_rays"] - counts["tail_traversed_rays"]], dtype=torch.float64, device="cuda")
    trace_ms = torch.tensor([sum(s_["ms_trace"] for s_ in stats) / n_single * args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
        dist.all_reduce(trace_ms, op=dist.ReduceOp.MAX)
    ms, ms_single, ms_fpb1, ms_single_one_lane = (float(x) for x in t.tolist())
    rays, paths, launches, V, T, Rc, Cc = (float(x) for x in agg.tolist())
    trace_ms = float(trace_ms.item())
    clocks = clk.summary()

    # ---- e2e arm: host buffers in, host image out, every step (scene upload + LBVH build [+ broadcast] inside the timed region)
    pinned, keep = pin_meshes(meshes)
    h2d = sum(t_.nbytes for t_ in pinned) + 36 * len(spheres) + 20 * (len(spheres) + len(meshes)) + 64
    d2h = H * W * 3

    pipe_e = R.FramePipeline(W, H, depth=args.frames_in_flight, host_output=True, shard_mode=shard_mode)
    e2e_last = [None]

    def retire(fin):
        if fin is not None:
            img, old_scene = fin
            old_scene.close()
            e2e_last[0] = img

    e2e_broadcast = [False]

    def step_e2e():
        t_a = time.perf_counter()
        sc = make_scene(spheres, meshes, pinned, broadcast=e2e_broadcast[0])
        sc.handle()                                           # rbrt_gpu_scene_create: H2D of the triangle soup + LBVH build, enqueued (every rank its own; or rank 0 + NCCL broadcast)
        t_b = time.perf_counter()
        # render -> finalise -> [gather] -> RGB8 image to pinned host memory, enqueued on the frame's stream; the image of
        # the frame submitted `frames_in_flight` steps ago is collected (host buffer ready) and its scene destroyed
        for fin in pipe_e.submit(cam_c, spp, sc, tag=sc, seed=SEED):
            retire(fin)
        t_c = time.perf_counter()
        return (t_b - t_a) * 1e3, (t_c - t_b) * 1e3

    def timed_e2e():
        for _ in range(max(2, args.frames_in_flight + 1)):
            step_e2e()
        for fin in pipe_e.drain():
            retire(fin)
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(args.steps):
            ms_create, ms_render = step_e2e()
        for fin in pipe_e.drain():                            # every image of the timed steps is on the host when the clock stops
            retire(fin)
        e1.record(stream)
        barrier()
        ms_ = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)   # host-side work (malloc, sync copies) counts too
        print(f"[e2e rank {rank}] broadcast={e2e_broadcast[0]} last step: scene_create {ms_create:.1f} ms, submit (+ wait for the frame {args.frames_in_flight} steps back) "
              f"{ms_render:.1f} ms; {args.steps} steps", file=sys.stderr)
        return ms_

    e_ms = timed_e2e()
    e_ms_bcast = None
    if world > 1:                                             # for the record: rank 0 alone uploads + builds, NCCL broadcast of the scene block
        e2e_broadcast[0] = True
        e_ms_bcast = timed_e2e()
        e2e_broadcast[0] = False
    if rank == 0 and check_images:
        assert np.array_equal(e2e_last[0].pixels.reshape(-1), rgb_ref.cpu().numpy()), "e2e image differs from the single-frame render"
    e_rays = frame["rays"] * args.steps
    te = torch.tensor([e_ms, e_ms_bcast or 0.0], dtype=torch.float64, device="cuda")
    re = torch.tensor([float(e_rays)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(re, op=dist.ReduceOp.SUM)
    e_ms_max, e_ms_bcast_max = (float(x) for x in te.tolist())
    e_val = float(re.item()) / (e_ms_max / 1e3) / 1e6

    # ---- image check at EVERY N: rank 0 renders a pixel lattice of the same frame with the CPU oracle; all ranks render that
    #      frame collectively at the same seed and sample count; the lattice pixels must agree bit for bit.  At N = 1 the oracle
    #      pass is the cpu_baseline sample (~20 s); at N > 1 it is a few seconds.
    plan = [0, 0]
    O = osc = None
    if rank == 0 and not args.no_cpu:
        O, osc = oracle_scene(spheres, meshes)
        plan = list(choose_stride(O, osc, cam_c, spp, 22.0 if world == 1 else 3.0))
    if world > 1:
        pl = torch.tensor(plan, dtype=torch.int64, device="cuda")
        dist.broadcast(pl, src=0)
        plan = [int(x) for x in pl.tolist()]
    stride, s_spp = plan
    image_check = cpu_baseline = None
    if stride:
        hdr = torch.empty(H * W * 3, dtype=torch.float32, device="cuda")
        hdr1 = (C.c_void_p * 1)(hdr.data_ptr())
        if rank == 0:
            cpu_st, acc_cpu = cpu_leg(O, osc, cam_c, stride, s_spp, want_image=True)
            if world == 1 and cpu_st["ms_total"] < 10e3 and stride > 1 and s_spp == 1:   # the probe under-estimated the cost per path: one denser pass (~18 s)
                stride2 = max(1, int(stride * (cpu_st["ms_total"] / 18e3) ** 0.5))
                if stride2 < stride:
                    stride = stride2
                    cpu_st, acc_cpu = cpu_leg(O, osc, cam_c, stride, s_spp, want_image=True)
        step_single({}, _abi.StatsC(), n_spp=s_spp, out=None, hdr=hdr1)
        barrier()
        if rank == 0:
            hdr_gpu = hdr.cpu().numpy().reshape(H, W, 3)[::stride, ::stride]
            acc_ref = np.asarray(acc_cpu, np.float32).reshape(H, W, 4)[::stride, ::stride, :3]
            hdr_ref = acc_ref * np.float32(1.0 / s_spp)                                  # lib.rs:101
            to_u8 = lambda h_: np.clip(np.nan_to_num(np.sqrt(np.maximum(h_, 0)) * 256.0), 0, 255).astype(np.uint8).astype(np.float64)
            image_check = {"pixels": int(acc_ref.shape[0] * acc_ref.shape[1]), "spp": int(s_spp), "n_gpus": world,
                           "bit_identical": bool(np.array_equal(np.ascontiguousarray(hdr_gpu).view(np.uint32), np.ascontiguousarray(hdr_ref).view(np.uint32))),
                           "hdr_rmse": float(np.sqrt(np.mean((hdr_gpu.astype(np.float64) - hdr_ref) ** 2))),
                           "u8_rmse": float(np.sqrt(np.mean((to_u8(hdr_gpu) - to_u8(hdr_ref)) ** 2))),
                           "note": "the N-GPU collective render vs the CPU oracle on a pixel lattice, same seed and spp (equal Philox streams => RMSE 0 "
                                   "expected); the criterion for independent seeds, RMSE(gpu, cpu_a) <= 1.10 RMSE(cpu_b, cpu_a), is in tests/"}
            if world == 1:
                cores = int(O.lib().rbrt_ref_hardware_threads())
                cpu_baseline = {"value": cpu_st["rays"] / (cpu_st["ms_total"] / 1e3) / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                                "sample": f"pixel lattice stride {stride}x{stride} of the {W}x{H} frame, {s_spp} of {spp} spp: {cpu_st['paths']} paths, "
                                          f"{cpu_st['rays']} rays in {cpu_st['ms_total'] / 1e3:.1f} s"}

    if rank != 0:
        if world > 1:
            lib.rbrt_gpu_comm_destroy()
            dist.destroy_process_group()
        return 0

    peak, peak_src = peaks()
    ns, nm = len(spheres), len(meshes)
    cstep = {"rays": Rc, "node_visits": V, "tri_tests": T, "traversed_rays": Cc}
    bytes_step = algorithmic_bytes(cstep, ns, nm)
    flops_step = algorithmic_flops(cstep, ns, nm)
    trace_ms_step = trace_ms / args.steps          # max over ranks of the per-rank sum; ranks run concurrently
    achieved = bytes_step / max(world, 1) / (trace_ms_step / 1e3) / 1e9 if trace_ms_step > 0 else None
    ev = ncu_evidence(args.workload, world)
    traffic = ev.get("dram_bytes_per_step") if ev else None
    line = {
        "metric": "Mrays/s", "value": rays / (ms / 1e3) / 1e6, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args.workload, spheres, meshes, world), frames_in_flight=args.frames_in_flight, frames_per_batch=fpb),
        "timed_region": {"steps": args.steps, "ms": ms,
                         "note": "one region of K steps (barrier + synchronize on both sides, CUDA events, max over ranks)"},
        "single_frame": {"ms_per_step": ms_single, "value": rays / args.steps / (ms_single / 1e3) / 1e6, "unit": "Mrays/s",
                         "ms_per_step_one_lane": ms_single_one_lane, "two_lanes": bool(use_split),
                         "note": "one frame at a time, host waits for each (latency of a lone render_scene call, gather on rank 0 included), the frame's "
                                 "sample batches on two lanes when it has >= 2^26 paths per GPU, as rbrt_gpu_render issues it (RBRT_OPT_SPLIT_BATCHES; one lane: ms_per_step_one_lane); `value` "
                                 "keeps `frames_in_flight` groups of `frames_per_batch` frames in flight on separate streams"},
        "frames_per_batch_1": ({"ms_per_step": ms_fpb1 / args.steps, "value": rays / (ms_fpb1 / 1e3) / 1e6, "unit": "Mrays/s"} if ms_fpb1 else None),
        "samples_per_s": paths / (ms / 1e3), "rays_per_step": rays / args.steps, "rays_per_sample": rays / max(paths, 1),
        "clocks": clocks,
        "e2e": {"value": e_val, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": args.steps,
                "ms_per_step": e_ms_max / args.steps,
                "ms_per_step_scene_broadcast": (e_ms_bcast_max / args.steps) if e_ms_bcast else None,
                "includes": "scene upload from pinned host memory + LBVH build (every rank its own replica, the library's default with one process per GPU; "
                            "ms_per_step_scene_broadcast: rank 0 alone + ncclBroadcast of the 168 MB block) + render + RGB8 image to pinned host memory, per step; "
                            "frames_in_flight frames overlap (FramePipeline), all images on the host when the clock stops"},
        "gpu_launches": int(launches),
        "multi_gpu": {"inside_library": True, "transport": {0: "none", 1: "nccl", 2: "peer"}.get(comm["transport"], "?"), "nccl_version": comm["nccl_version"]},
        "roofline": {"bound": "hbm", "limiter": "issue / ALU pipe under partial lane occupancy, NOT memory (see `ncu`): the kernel's requested bytes are served by L1/L2",
                     "kernel": "k_trace (stage B: persistent LBVH traversal with dynamic fetch + Moeller-Trumbore tests)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                     "dram_frac": (traffic / (trace_ms_step / 1e3) / 1e9 / peak) if (traffic and trace_ms_step > 0) else None,
                     "ncu": ev,
                     "peak_source": peak_src, "algorithmic_bytes_per_traversed_ray": bytes_step / max(Cc, 1),
                     "traversed_rays_per_step": Cc, "traversed_share_of_rays": Cc / max(Rc, 1),
                     "node_visits_per_traversed_ray": V / max(Cc, 1), "tri_tests_per_traversed_ray": T / max(Cc, 1),
                     "trace_ms_per_step": trace_ms_step, "trace_share_of_step": trace_ms_step / ms_single_one_lane,
                     "fp32_achieved_tflops": flops_step / max(world, 1) / (trace_ms_step / 1e3) / 1e12 if trace_ms_step > 0 else None,
                     "fp32_peak_tflops": 37.2, "fp32_frac": (flops_step / max(world, 1) / (trace_ms_step / 1e3) / 1e12 / 37.2) if trace_ms_step > 0 else None,
                     "fp32_note": "secondary bound of SURVEY.md 8(d): 148 SMs x 128 lanes x 1.965 GHz = 37.2 T lane-ops/s without FMA contraction (parity forbids it)",
                     "note": "achieved = per-GPU ALGORITHMIC bytes of all trace launches of a step / their summed CUDA-event time (events on the launching stream, "
                             "this run's single-frame pass); `frac` is that REQUESTED bandwidth against the HBM copy peak as the contract defines it. `traffic` = "
                             "dram__bytes_read+write of the same launches from the committed ncu capture for THIS N (`ncu`), `dram_frac` = traffic / trace time / peak: "
                             "what HBM actually sees"},
        "scene": {"bvh_nodes": info["num_bvh_nodes"], "device_bytes": info["device_bytes"], "ms_upload": info["ms_upload"], "ms_build": info["ms_build"]},
    }
    if image_check:
        line["image_check"] = image_check
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    print(json.dumps(line), file=_STDOUT, flush=True)
    if world > 1:
        lib.rbrt_gpu_comm_destroy()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU oracle legs (cpu_baseline, image_check): profiling runs")
    ap.add_argument("--frames-per-batch", type=int, default=0, choices=[0, 1, 2, 3, 4],
                    help="frames rendered together in the same wavefront batches in the timed region (0 = 4 at EVERY N; sample-sharded workloads 1)")
    ap.add_argument("--frames-in-flight", type=int, default=2, choices=[1, 2, 3, 4],
                    help="groups of frames kept in flight on separate streams in the timed region (1 = one group at a time)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the image of the last timed step as DIR/<name>.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU arm computed; the reference arm has no such output")
    # exactly ONE line goes to stdout (the JSON); the host mirror's progress prints (lib.rs:80,114, mesh.rs:115) go to stderr
    # (NCCL and the host mirror also write to fd 1 from C: redirect the descriptor itself, keep a private duplicate for the JSON)
    global _STDOUT
    sys.stdout.flush()
    _STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
