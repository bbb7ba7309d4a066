"""Per-pixel variance from sample-range shards (rbrt_gpu_render_hdr_variance*) and the variance-guided filter (rbrt_gpu_denoise_variance*;
csrc/variance.cu, csrc/api.cu) on the GPU.

hdr_out is compared bit for bit with the PEER sample-sharded render, var_out with tests/variance_ref.py applied to the accumulators of
explicit shard renders, and the filter with the numpy restatement of its definition (NaN equal to NaN whatever its payload).  The
calibration test checks the variance against the spread of independent renders, and the quality test measures both filters on real
renders against 4096-spp references."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi, png

from . import scenes as S
from . import variance_ref as V
from .test_cli_cpp import write_scene
from .test_denoise_host import adversarial, scene_like
from .test_gpu_denoise import BOUNDS as PLAIN_BOUNDS
from .test_gpu_denoise import boundary, rmse
from .test_gpu_update import fresh, twist
from .test_variance_host import variance_like

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VAR = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_variance.so")


@pytest.fixture(scope="module", autouse=True)
def variance_module():
    if not os.path.exists(VAR):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return VAR


def workload(name, W=256, H=192):
    import bench
    spheres, meshes, camkw = bench.build_workload(name)
    scene = bench.make_scene(spheres, meshes)
    return scene, R.Camera.new(camkw["position"], camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])


def shard_accumulators(scene, cam, S_, K, seed):
    """The K per-pixel sums of explicit rbrt_gpu_render_accum_device shard renders: [K, H, W, 4] float32."""
    import torch
    W, H = cam.img_width_pix, cam.img_height_pix
    out = []
    for k in range(K):
        buf = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
        _abi.check(_abi.lib().rbrt_gpu_render_accum_device(
            scene.handle(), cam.to_c(), S_, R.render.make_opts(seed=seed, shard_mode=_abi.SHARD_SAMPLES, shard_rank=k, shard_count=K),
            buf.data_ptr(), None, None))
        torch.cuda.synchronize()
        out.append(buf.cpu().numpy())
    return np.stack(out)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def to_t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check_filter(planes, v, what, **opts):
    """R.denoise_variance of (c, a, n, z) and v against the numpy reference; returns the outputs."""
    c, a, n, z = planes
    out, img = R.denoise_variance(c, v, {"depth": z, "normal": n, "albedo": a}, **opts)
    want, want_rgb = V.denoise_variance(c, v, a, n, z, **opts)
    assert V.same_bits(out, want), f"{what}: hdr_out differs in {int((~np.isclose(out, want, equal_nan=True)).sum())} values"
    assert np.array_equal(img.pixels, want_rgb), what
    return out, img.pixels


# ============================================================================== 1. the moments
@pytest.mark.parametrize("K", [2, 4])
def test_hdr_equals_the_peer_sample_sharded_render(gpu, K):
    """hdr_out is the PEER sample-sharded rbrt_gpu_render_hdr on K ranks (one GPU emulating them) bit for bit, also when the variance
    call runs under that communicator (on replica 0, not collective)."""
    lib = _abi.lib()
    devs = (C.c_int * K)(*([0] * K))
    _abi.check(lib.rbrt_gpu_init_multi(devs, K, _abi.TRANSPORT_PEER))
    try:
        scene, cam = workload("c2", 96, 64)
        peer = R.render_scene_hdr(cam, 8 * K, scene, seed=3, shard_mode=_abi.SHARD_SAMPLES)
        hdr_comm, var_comm = R.render_scene_hdr_variance(cam, 8 * K, scene, splits=K, seed=3)
        scene.close()
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)
    scene, cam = workload("c2", 96, 64)
    hdr, var = R.render_scene_hdr_variance(cam, 8 * K, scene, splits=K, seed=3)
    assert np.array_equal(bits(hdr), bits(peer))
    assert np.array_equal(bits(hdr_comm), bits(peer)) and np.array_equal(bits(var_comm), bits(var))


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_hdr_is_within_1e5_of_the_unsharded_render(gpu, name):
    scene, cam = workload(name)
    for K, S_ in ((2, 64), (4, 64), (16, 64), (3, 12)):
        hdr, _ = R.render_scene_hdr_variance(cam, S_, scene, splits=K, seed=11)
        plain = R.render_scene_hdr(cam, S_, scene, seed=11)
        assert np.isfinite(plain).all()
        assert (np.abs(hdr.astype(np.float64) - plain) <= 1e-5 * np.abs(plain.astype(np.float64))).all(), (name, K)


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_variance_equals_numpy_on_explicit_shard_renders(gpu, name):
    scene, cam = workload(name)
    for K in (2, 3, 4, 16):
        S_ = 4 * K
        acc = shard_accumulators(scene, cam, S_, K, seed=11)
        want_h, want_v = V.moments(acc, S_)
        st = {}
        hdr, var = R.render_scene_hdr_variance(cam, S_, scene, splits=K, seed=11, stats=st)
        assert V.same_bits(hdr, want_h), (name, K)
        assert V.same_bits(var, want_v), (name, K, int((bits(var) != bits(want_v)).sum()))
        assert (var >= 0).all() and (var > 0).mean() > 0.2
        n = 256 * 192
        assert st["paths"] == n * S_ and st["rays"] >= n * S_ and st["ms_device"] > 0 and st["launches"] > K
        dh, dv = R.render_hdr_variance_device(cam, S_, scene, splits=K, seed=11)
        import torch
        torch.cuda.synchronize()
        assert np.array_equal(bits(dh.cpu().numpy()), bits(hdr)) and np.array_equal(bits(dv.cpu().numpy()), bits(var))


def test_variance_is_calibrated_across_seeds(gpu):
    """Σ over pixels of the mean var_out of 32 seeds against Σ of the across-seed variance of hdr_out: a wrong K(K-1) is off by a
    factor of at least 1.3 (K = 4)."""
    scene, cam = workload("c1", 128, 96)
    hs, vs = [], []
    for seed in range(32):
        h, v = R.render_scene_hdr_variance(cam, 16, scene, splits=4, seed=1000 + seed)
        hs.append(h.astype(np.float64))
        vs.append(v.astype(np.float64))
    hs, vs = np.stack(hs), np.stack(vs)
    ok = np.isfinite(hs).all(0) & np.isfinite(vs).all(0)
    empirical = hs.var(0, ddof=1)[ok].sum()
    predicted = vs.mean(0)[ok].sum()
    assert empirical > 0
    assert 0.9 <= predicted / empirical <= 1.1, predicted / empirical


# ============================================================================== 2. the filter, bit for bit
@pytest.mark.parametrize("levels", range(1, 9))
def test_filter_random_planes_every_level(gpu, levels):
    check_filter(adversarial(37, 53, levels), variance_like(37, 53, levels), f"adversarial L={levels}", levels=levels)
    check_filter(scene_like(40, 64, levels), variance_like(40, 64, levels, specials=False), f"scene-like L={levels}", levels=levels)
    check_filter(scene_like(40, 64, 50 + levels), variance_like(40, 64, 50 + levels, specials=False), f"scene-like L={levels}, sigmas",
                 levels=levels, sigma_depth=0.3, sigma_luminance=0.5)


@pytest.mark.parametrize("shape", [(1, 1), (1, 40), (40, 1), (5, 7), (17, 33)])
def test_filter_image_shapes(gpu, shape):
    H, W = shape
    for L in (0, 3, 8):
        check_filter(adversarial(H, W, H * 100 + W), variance_like(H, W, H * 100 + W), f"{W}x{H} L={L}", levels=L)


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_filter_real_renders(gpu, name):
    scene, cam = workload(name)
    hdr, var = R.render_scene_hdr_variance(cam, 16, scene, splits=4, seed=11)
    aov = R.render_aovs(cam, 4, scene, seed=11)
    planes = (hdr, aov["albedo"], aov["normal"], aov["depth"])
    out, _ = check_filter(planes, var, name)
    assert not V.same_bits(out, hdr)
    check_filter(planes, var, f"{name}, L=2 and sigmas", levels=2, sigma_depth=0.05, sigma_luminance=1.0)


# ============================================================================== 3. host and device variants, streams, updates
def test_filter_device_variant_equals_the_host_variant_on_a_side_stream(gpu):
    import torch
    c, a, n, z = scene_like(120, 200, 3)
    v = variance_like(120, 200, 3, specials=False)
    host, img = R.denoise_variance(c, v, {"depth": z, "normal": n, "albedo": a})
    s = torch.cuda.Stream()
    g = {"depth": to_t(z), "normal": to_t(n), "albedo": to_t(a)}
    tc, tv = to_t(c), to_t(v)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(2e9))                                       # about a second of work ahead of the call on its stream
        t0 = time.perf_counter()
        out, rgb = R.denoise_variance_device(tc, tv, g, stream=s)
        dt = time.perf_counter() - t0
        busy = not s.query()
    s.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    assert np.array_equal(bits(out.cpu().numpy()), bits(host))
    assert np.array_equal(rgb.cpu().numpy(), img.pixels)


def test_render_on_side_streams_two_calls_in_flight(gpu):
    """Two device calls enqueued on two streams behind queued work, each returning before its stream runs, each equal to the host call
    (different wavefront pools: frames in flight at the same time use different pools)."""
    import torch
    scene, cam = workload("c2", 128, 96)
    want = [R.render_scene_hdr_variance(cam, 16, scene, splits=4, seed=s) for s in (5, 6)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs, busy = [], []
    for i, (s, seed) in enumerate(zip(streams, (5, 6))):
        with torch.cuda.stream(s):
            torch.cuda._sleep(int(1e9))
            t0 = time.perf_counter()
            outs.append(R.render_hdr_variance_device(cam, 16, scene, splits=4, seed=seed, stream=s, pool=i))
            busy.append((not s.query(), time.perf_counter() - t0))
    for s in streams:
        s.synchronize()
    assert all(b for b, _ in busy) and all(dt < 0.5 for _, dt in busy), busy
    for (h, v), (wh, wv) in zip(outs, want):
        assert np.array_equal(bits(h.cpu().numpy()), bits(wh)) and np.array_equal(bits(v.cpu().numpy()), bits(wv))
    assert not np.array_equal(want[0][1], want[1][1])


def test_two_filter_calls_in_flight_on_two_streams(gpu):
    import torch
    ins = [(scene_like(300, 400, k), variance_like(300, 400, k, specials=False)) for k in (1, 2)]
    dev = [(to_t(c), to_t(v), {"depth": to_t(z), "normal": to_t(n), "albedo": to_t(a)}) for (c, a, n, z), v in ins]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = []
    for s, (tc, tv, g) in zip(streams, dev):
        with torch.cuda.stream(s):
            torch.cuda._sleep(int(3e8))
            outs.append(R.denoise_variance_device(tc, tv, g, levels=6, stream=s)[0])
    for s in streams:
        s.synchronize()
    want = [R.denoise_variance(c, v, {"depth": z, "normal": n, "albedo": a}, levels=6)[0] for (c, a, n, z), v in ins]
    for o, w in zip(outs, want):
        assert np.array_equal(bits(o.cpu().numpy()), bits(w))


def test_ordering_against_a_scene_update(gpu):
    import torch
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(48, 36)
    old = R.render_scene_hdr_variance(cam, 8, fresh(scene), splits=2, seed=4)
    new = twist(scene.triangle_meshes[0].triangles, 0.8)
    ref_scene = fresh(scene)
    ref_scene.triangle_meshes[0] = R.TriangleMesh.from_triangles(new, ref_scene.triangle_meshes[0].material)
    want_new = R.render_scene_hdr_variance(cam, 8, ref_scene, splits=2, seed=4)
    assert not np.array_equal(old[0], want_new[0]), "the deformation must change the image"
    R.render_scene_hdr_variance(cam, 2, scene, splits=2)                  # built and in use before the update
    t_new = torch.from_numpy(new.copy()).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(5e8))                                       # the first call waits in the stream while the update is enqueued
        a = R.render_hdr_variance_device(cam, 8, scene, splits=2, seed=4, stream=s)
        scene.update_mesh_device(0, t_new, stream=s)
        b = R.render_hdr_variance_device(cam, 8, scene, splits=2, seed=4, stream=s)
    s.synchronize()
    for got, want, what in ((a, old, "before"), (b, want_new, "after")):
        assert np.array_equal(bits(got[0].cpu().numpy()), bits(want[0])), what
        assert np.array_equal(bits(got[1].cpu().numpy()), bits(want[1])), what


def test_stats_of_the_filter(gpu):
    c, a, n, z = scene_like(64, 96, 4)
    v = variance_like(64, 96, 4, specials=False)
    st = {}
    R.denoise_variance(c, v, {"depth": z, "normal": n, "albedo": a}, levels=3, stats=st)
    assert st["launches"] == 4 and st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"]
    st = {}
    R.denoise_variance(c, v, {"depth": z, "normal": n, "albedo": a}, stats=st)
    assert st["launches"] == 1 + V.DEFAULT_LEVELS


# ============================================================================== 4. refusals, communicator, missing module
def test_refusals_on_the_device(gpu):
    import torch
    from .test_gpu_bvh_build import REFUSED, deep_camera, deep_scene
    lib = _abi.lib()
    scene, cam = workload("c1", 16, 12)
    out = torch.full((12, 16, 3), 7.0, device="cuda")
    host_out = np.full((12, 16, 3), 7.0, np.float32)
    O = R.render.make_opts
    for args, msg in [((8, 4, O(), out.data_ptr(), host_out.ctypes.data), b"device memory"),
                      ((8, 1, O(), out.data_ptr(), None), b"splits"),
                      ((8, 3, O(), out.data_ptr(), None), b"multiple"),
                      ((8, 4, O(shard_mode=_abi.SHARD_SAMPLES, shard_count=2), out.data_ptr(), None), b"shard_count"),
                      ((8, 4, O(max_depth=1025), out.data_ptr(), None), b"max_depth")]:
        assert lib.rbrt_gpu_render_hdr_variance_device(scene.handle(), cam.to_c(), *args, None, None) == _abi.E_INVALID, msg
        assert msg in lib.rbrt_last_error(), (msg, lib.rbrt_last_error())
    torch.cuda.synchronize()
    assert (out == 7.0).all() and (host_out == 7.0).all()
    deep = deep_scene(REFUSED)
    with pytest.raises(_abi.RbrtGpuError, match="BVH deeper than the traversal stack allows") as e:
        R.render_scene_hdr_variance(deep_camera(8, 6), 4, deep, splits=2, seed=1)
    assert e.value.code == _abi.E_INVALID
    c, a, n, z = scene_like(8, 8, 5)
    v = variance_like(8, 8, 5, specials=False)
    t = {k: to_t(x) for k, x in (("c", c), ("v", v), ("a", a), ("n", n), ("z", z))}
    o = torch.full((8, 8, 3), 7.0, device="cuda")
    g = _abi.AovOutC(depth=t["z"].data_ptr(), normal=t["n"].data_ptr(), albedo=t["a"].data_ptr())
    assert lib.rbrt_gpu_denoise_variance_device(8, 8, t["c"].data_ptr(), v.ctypes.data, g, None, o.data_ptr(), None, None, None) == _abi.E_INVALID
    assert b"device memory" in lib.rbrt_last_error()
    torch.cuda.synchronize()
    assert (o == 7.0).all()
    _abi.check(lib.rbrt_gpu_denoise_variance_device(8, 8, t["c"].data_ptr(), t["v"].data_ptr(), g, None, o.data_ptr(), None, None, None))
    torch.cuda.synchronize()
    assert V.same_bits(o.cpu().numpy(), V.denoise_variance(c, v, a, n, z)[0])


def test_filter_under_an_emulated_communicator(gpu):
    planes = scene_like(48, 64, 6)
    v = variance_like(48, 64, 6, specials=False)
    lib = _abi.lib()
    devs = (C.c_int * 2)(0, 0)
    _abi.check(lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER))
    try:
        check_filter(planes, v, "under a one-GPU two-rank communicator")
    finally:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


def test_missing_module_is_refused_with_a_message(gpu):
    """Without librbrt_gpu_variance.so both calls fail with a message naming the module; render, AOV and denoise calls still work."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); cam = S.example_camera(16, 12)\n"
            "hdr = R.render_scene_hdr(cam, 2, sc); aov = R.render_aovs(cam, 2, sc)\n"
            "for f in (lambda: R.render_scene_hdr_variance(cam, 4, sc, splits=2), lambda: R.denoise_variance(hdr, np.zeros_like(hdr), aov)):\n"
            "    try:\n        f()\n        print('NO ERROR')\n"
            "    except _abi.RbrtGpuError as e:\n        print('CODE', e.code, str(e))\n"
            "print('RENDER', hdr.shape, 'AOV', aov['depth'].shape, 'DENOISE', R.denoise(hdr, aov)[0].shape)\n") % ROOT
    env = dict(os.environ, RBRT_GPU_VARIANCE_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_variance.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count(f"CODE {_abi.E_CUDA}") == 2 and r.stdout.count("variance module is missing") == 2, r.stdout
    assert "RENDER (12, 16, 3) AOV (12, 16) DENOISE (12, 16, 3)" in r.stdout, r.stdout


# ============================================================================== 5. CLI
def test_cli_denoise_splits_equals_the_python_composition(gpu, tmp_path):
    cli = os.path.join(ROOT, "rbrt_b200", "rbrt")
    y, _ = write_scene(tmp_path)
    bp = R.load_blueprints_from_yaml_file(y)
    cb = bp.camera_blueprint
    cam = R.Camera.new(cb.camera_position, cb.camera_look_at, cb.camera_up, 30, 44, cb.camera_focal_length_mm)
    scene = R.create_scene_from_scene_blueprint(bp)
    base = [cli, "-c", y, "--height", "30", "-w", "44", "--seed", "5", "--denoise"]
    for spp, k, extra, s_aov in [(16, 4, [], 4), (8, 4, [], 2), (16, 2, ["--aov-samples", "8"], 8)]:
        target = str(tmp_path / f"dv{spp}_{k}_{s_aov}.png")
        r = subprocess.run(base + ["-s", str(spp), "--denoise-splits", str(k), "-t", target] + extra, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        hdr, var = R.render_scene_hdr_variance(cam, spp, scene, splits=k, seed=5)
        aov = R.render_aovs(cam, s_aov, scene, seed=5)
        _, img = R.denoise_variance(hdr, var, aov)
        want = tmp_path / f"want{spp}_{k}_{s_aov}.png"
        img.save(str(want))
        assert png.decode_png(open(target, "rb").read()).tobytes() == png.decode_png(open(want, "rb").read()).tobytes(), (spp, k, s_aov)
    plain = str(tmp_path / "plain.png")                                   # without --denoise-splits: the plain filter, as before
    r = subprocess.run(base + ["-s", "8", "-t", plain], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    _, img = R.denoise(R.render_scene_hdr(cam, 8, scene, seed=5), R.render_aovs(cam, 4, scene, seed=5))
    assert png.decode_png(open(plain, "rb").read()).tobytes() == img.pixels.tobytes()


# ============================================================================== 6. quality against 4096-spp references
# Denoised / noisy RMSE of the variance-guided filter with its defaults, K = 4, guides at S = 4, as measured on these renders (DESIGN.md
# section 14) with a margin of 0.02.  The target of 0.5 at 4 spp is not met (0.53 / 0.58 / 0.61).
BOUNDS = {("c1", 4): 0.56, ("c2", 4): 0.61, ("c4", 4): 0.64, ("c1", 16): 0.62, ("c2", 16): 0.72, ("c4", 16): 0.71,
          ("c1", 64): 0.72, ("c2", 64): 0.88, ("c4", 64): 0.82}


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_quality_against_a_4096_spp_reference(gpu, name):
    """The harness of tests/test_gpu_denoise.py (same cameras, reference seed 12345, noisy seed 11), K = 4; rbrt_gpu_denoise runs on the
    same frames."""
    scene, cam = workload(name)
    ref = R.render_scene_hdr(cam, 4096, scene, seed=12345)
    aov = R.render_aovs(cam, 4, scene, seed=11)
    edge = boundary(aov["hit_kind"], aov["elem_idx"])
    assert 500 < edge.sum() < 0.5 * edge.size
    for spp in (4, 16, 64):
        noisy, var = R.render_scene_hdr_variance(cam, spp, scene, splits=4, seed=11)
        out, _ = R.denoise_variance(noisy, var, aov)
        plain, _ = R.denoise(noisy, aov)
        ratio = rmse(out, ref) / rmse(noisy, ref)
        plain_ratio = rmse(plain, ref) / rmse(noisy, ref)
        print(f"{name} {spp} spp: variance-guided {ratio:.4f}, plain {plain_ratio:.4f}, boundary {rmse(out[edge], ref[edge]) / rmse(noisy[edge], ref[edge]):.4f}")
        assert ratio <= BOUNDS[name, spp], (name, spp, ratio)
        assert plain_ratio <= PLAIN_BOUNDS[name, spp], (name, spp, plain_ratio)
        assert ratio <= 1.0 if spp == 64 else ratio < 1.0, (name, spp, ratio)
        if spp <= 16:                                                     # no worse than rbrt_gpu_denoise on the same frame
            assert ratio <= plain_ratio, (name, spp, ratio, plain_ratio)
        if spp <= 16:
            assert rmse(out[edge], ref[edge]) <= rmse(noisy[edge], ref[edge]), (name, spp, "boundary pixels")
