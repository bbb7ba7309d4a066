"""Temporal accumulation (rbrt_gpu_temporal_accumulate*; csrc/temporal.cu, csrc/api.cu) on the GPU.

The kernel is compared bit for bit with tests/temporal_ref.py (NaN equal to NaN whatever its payload) on the synthetic planes of
tests/test_temporal_host.py and on real renders over camera sweeps.  A static camera with α_min = 0 is checked against the running mean
(RMSE) and its variance against the spread of independent sequences; a moved sphere checks that disoccluded pixels restart; and the
quality test measures temporal, spatial and temporal-then-spatial filtering against 4096-spp references."""
import os
import subprocess
import sys

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import temporal_ref as T
from .test_gpu_denoise import rmse
from .test_temporal_host import CASE_NAMES, cases, frame, history

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TMP = os.path.join(ROOT, "rbrt_b200", "librbrt_gpu_temporal.so")


@pytest.fixture(scope="module", autouse=True)
def temporal_module():
    """The session fixture only builds librbrt_gpu.so when it is missing; the module is built here when it is."""
    if not os.path.exists(TMP):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return TMP


def workload(name, W=256, H=192, dx=0.0):
    import bench
    spheres, meshes, camkw = bench.build_workload(name)
    scene = bench.make_scene(spheres, meshes)
    return scene, sweep_camera(camkw, W, H, dx)


def sweep_camera(camkw, W, H, dx):
    p = camkw["position"]
    return R.Camera.new(R.Vec3(p.x + dx, p.y, p.z), camkw["look_at"], camkw["up"], H, W, camkw["focal_len_mm"])


def camkw_of(name):
    import bench
    return bench.build_workload(name)[2]


def same_all(a, b):
    return all((x is None and y is None) or T.same_bits(x, y) for x, y in zip(a, b))


def check(cam, hdr, var, aovs, hist, what, **opts):
    got = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist, **opts)
    want = T.accumulate(cam, hdr, var, aovs, hist, **opts)
    for g, w, k in zip(got, want, ("hdr_out", "var_out", "len_out")):
        assert (g is None and w is None) or T.same_bits(g, w), f"{what}: {k} differs"
    return got


def to_t(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def u32(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(np.uint32)


# ============================================================================== 1. the kernel against numpy
@pytest.mark.parametrize("name", CASE_NAMES)
@pytest.mark.parametrize("shape", [(48, 32), (1, 1), (1, 40), (40, 1), (7, 5), (33, 17)])
def test_synthetic_planes(gpu, name, shape):
    (case,) = [c for c in cases(*shape) if c[0] == name]
    _, cam, prev, opts = case
    for specials in (False, True):
        hdr, var, aovs = frame(cam, 3, specials)
        hist = history(prev, 4, specials) if prev is not None else None
        for v in (var, None):
            check(cam, hdr, v, aovs, hist, f"{name} {shape} specials={specials} var={v is not None}", **opts)


def render_frame(scene, cam, seed, spp=4, splits=4, aov_spp=4):
    hdr, var = R.render_scene_hdr_variance(cam, spp, scene, splits=splits, seed=seed)
    return hdr, var, R.render_aovs(cam, aov_spp, scene, seed=seed)


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_real_renders_over_a_camera_sweep(gpu, name):
    """8 frames of a sideways camera sweep with a rotation in the middle, chained through the host call; every frame equals numpy."""
    scene, _ = workload(name)
    kw = camkw_of(name)
    hist, kept = None, 0
    for f in range(8):
        cam = sweep_camera(kw, 256, 192, 0.04 * f)
        if f == 4:
            cam = R.Camera.new(cam.position, R.Vec3(0.03, -0.1, -1.0), kw["up"], 192, 256, kw["focal_len_mm"])
        hdr, var, aovs = render_frame(scene, cam, 11 + f)
        out = check(cam, hdr, var, aovs, hist, f"{name} frame {f}", alpha_min=0.0 if f == 6 else 0.1)
        kept += int((out[2] > 1).sum())
        hist = {"cam": cam, "hdr": out[0], "var": out[1], "length": out[2], "aovs": aovs}
    assert kept > 0.15 * 7 * 256 * 192, kept


# ============================================================================== 2. host and device variants, streams
def test_device_variant_equals_the_host_variant_on_a_side_stream(gpu):
    import torch
    _, cam, prev, opts = [c for c in cases(64, 48) if c[0] == "translation"][0]
    hdr, var, aovs = frame(cam, 5, True)
    hist = history(prev, 6, True)
    host = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist)
    d_aovs = {k: to_t(v) for k, v in aovs.items()}
    d_hist = {"cam": prev, "hdr": to_t(hist["hdr"]), "var": to_t(hist["var"]), "length": to_t(hist["length"]),
              "aovs": {k: to_t(v) for k, v in hist["aovs"].items()}}
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        dev = R.temporal_accumulate_device(cam, to_t(hdr), d_aovs, var=to_t(var), history=d_hist, stream=side)
    side.synchronize()
    for h, d in zip(host, dev):
        assert np.array_equal(h.view(np.uint32), u32(d))
    # the accumulator: two steps ping-pong its own tensors and equal the host calls
    acc = R.TemporalAccumulator(64, 48, stream=side)
    h0, v0, aov0 = frame(prev, 7)
    a1 = acc.step(prev, to_t(h0), to_t(v0), {k: to_t(v) for k, v in aov0.items()})
    a2 = acc.step(cam, to_t(hdr), to_t(var), d_aovs)
    side.synchronize()
    w1 = R.temporal_accumulate(prev, h0, aov0, var=v0)
    w2 = R.temporal_accumulate(cam, hdr, aovs, var=var, history={"cam": prev, "hdr": w1[0], "var": w1[1], "length": w1[2], "aovs": aov0})
    for w, a in zip(w1 + w2, a1 + a2):
        assert np.array_equal(w.view(np.uint32), u32(a))
    assert a1[0].data_ptr() != a2[0].data_ptr()
    acc.reset()
    a3 = acc.step(cam, to_t(hdr), to_t(var), d_aovs)
    assert (u32(a3[2]) == np.float32(1).view(np.uint32)).sum() + (u32(a3[2]) == 0).sum() == 64 * 48


def test_stats_report_one_launch_and_a_device_time(gpu):
    _, cam, prev, _ = [c for c in cases(64, 48) if c[0] == "rotation"][0]
    hdr, var, aovs = frame(cam, 5)
    st = {}
    R.temporal_accumulate(cam, hdr, aovs, var=var, history=history(prev, 6), stats=st)
    assert st["launches"] == 1 and st["ms_device"] > 0 and st["ms_total"] >= st["ms_device"]


def test_var_without_var_out_reads_no_history_variance(gpu):
    """var given for the validity rule but var_out not requested: the history's var is not read (here NULL), and hdr_out and len_out
    equal the call that propagates the variance."""
    _, cam, prev, _ = [c for c in cases(64, 48) if c[0] == "translation"][0]
    hdr, var, aovs = frame(cam, 8, True)
    hist = history(prev, 9, True)
    ha = hist["aovs"]
    g = lambda a: _abi.AovOutC(depth=a["depth"].ctypes.data, normal=a["normal"].ctypes.data, hit_kind=a["hit_kind"].ctypes.data,
                               elem_idx=a["elem_idx"].ctypes.data)
    h = _abi.TemporalHistoryC(cam=prev.to_c(), hdr=hist["hdr"].ctypes.data, var=None, length=hist["length"].ctypes.data, guides=g(ha))
    out, length = np.zeros((48, 64, 3), np.float32), np.zeros((48, 64), np.float32)
    _abi.check(_abi.lib().rbrt_gpu_temporal_accumulate(64, 48, cam.to_c(), hdr.ctypes.data, var.ctypes.data, g(aovs), h, None,
                                                       out.ctypes.data, None, length.ctypes.data, None))
    want = T.accumulate(cam, hdr, var, aovs, hist)
    assert T.same_bits(out, want[0]) and T.same_bits(length, want[2])


# ============================================================================== 3. refusals, missing module
def test_refusals_write_nothing(gpu):
    import torch
    lib = _abi.lib()
    W, H = 8, 6
    _, cam, prev, _ = [c for c in cases(W, H) if c[0] == "translation"][0]
    hdr, var, aovs = frame(cam, 5)
    hist = history(prev, 6)
    t = {k: to_t(v) for k, v in aovs.items()}
    g = _abi.AovOutC(depth=t["depth"].data_ptr(), normal=t["normal"].data_ptr(), hit_kind=t["hit_kind"].data_ptr(), elem_idx=t["elem_idx"].data_ptr())
    th = {k: to_t(hist[k]) for k in ("hdr", "var", "length")}
    ta = {k: to_t(v) for k, v in hist["aovs"].items()}
    hc = _abi.TemporalHistoryC(cam=prev.to_c(), hdr=th["hdr"].data_ptr(), var=th["var"].data_ptr(), length=th["length"].data_ptr(),
                               guides=_abi.AovOutC(depth=ta["depth"].data_ptr(), normal=ta["normal"].data_ptr(),
                                                   hit_kind=ta["hit_kind"].data_ptr(), elem_idx=ta["elem_idx"].data_ptr()))
    d_hdr, d_var = to_t(hdr), to_t(var)
    outs = [torch.full((H, W, 3), 7.0, device="cuda"), torch.full((H, W, 3), 7.0, device="cuda"), torch.full((H, W), 7.0, device="cuda")]
    o = [x.data_ptr() for x in outs]
    host_out = np.full((H, W, 3), 7.0, np.float32)
    ok_opts = _abi.TemporalOptsC(0.1, 0.02, 0.9)

    def call(cam_=cam, h=d_hdr.data_ptr(), v=d_var.data_ptr(), gg=g, hh=hc, op=ok_opts, oo=None, w=W, hgt=H):
        return lib.rbrt_gpu_temporal_accumulate_device(w, hgt, cam_.to_c(), h, v, gg, hh, op, *(oo or o), None, None)

    refused = [
        call(h=None), call(gg=None), call(oo=[None, None, None]), call(v=None), call(w=0), call(hgt=0), call(w=W + 1),
        call(cam_=R.Camera.new(cam.position, cam.look_at, cam.up, H, W + 2, cam.focal_len_mm)),
        call(hh=_abi.TemporalHistoryC(cam=prev.to_c(), hdr=hc.hdr, var=hc.var, length=None, guides=hc.guides)),
        call(hh=_abi.TemporalHistoryC(cam=prev.to_c(), hdr=hc.hdr, var=None, length=hc.length, guides=hc.guides)),
        call(op=_abi.TemporalOptsC(float("nan"), 0.02, 0.9)), call(op=_abi.TemporalOptsC(-0.1, 0.02, 0.9)),
        call(op=_abi.TemporalOptsC(1.01, 0.02, 0.9)), call(op=_abi.TemporalOptsC(0.1, float("inf"), 0.9)),
        call(op=_abi.TemporalOptsC(0.1, 0.02, -0.5)),
        call(oo=[d_hdr.data_ptr(), o[1], o[2]]),                          # in place
        call(oo=[o[0], th["var"].data_ptr(), o[2]]),                      # over the history
        call(oo=[o[0], o[1], t["depth"].data_ptr()]),                     # over a guide
        call(oo=[o[0], o[0] + 8, o[2]]),                                  # two outputs overlap
        call(h=hdr.ctypes.data),                                          # unregistered host memory as an input, as an output
        call(oo=[host_out.ctypes.data, o[1], o[2]]),
        call(gg=_abi.AovOutC(depth=aovs["depth"].ctypes.data, normal=g.normal, hit_kind=g.hit_kind, elem_idx=g.elem_idx)),
        call(hh=_abi.TemporalHistoryC(cam=prev.to_c(), hdr=hc.hdr, var=hc.var, length=hist["length"].ctypes.data, guides=hc.guides)),
    ]
    assert all(rc == _abi.E_INVALID for rc in refused), refused
    torch.cuda.synchronize()
    assert all(bool((x == 7.0).all()) for x in outs) and (host_out == 7.0).all()
    if torch.cuda.device_count() > 1:                                     # another device's memory
        other = torch.zeros((H, W, 3), device="cuda:1")
        assert call(h=other.data_ptr()) == _abi.E_INVALID and call(oo=[other.data_ptr(), o[1], o[2]]) == _abi.E_INVALID
        assert (other == 0).all()
    _abi.check(call())                                                    # the same call, valid
    torch.cuda.synchronize()
    want = T.accumulate(cam, hdr, var, aovs, hist)
    assert all(T.same_bits(x.cpu().numpy(), w) for x, w in zip(outs, want))


def test_missing_module_is_refused_with_a_message(gpu):
    """Without librbrt_gpu_temporal.so the call fails with a message naming the module; a render in the same process still works."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, rbrt_b200 as R\nfrom tests import scenes as S\nfrom rbrt_b200 import _abi\n"
            "R.gpu_init(0); sc = S.small_mesh_scene(3); cam = S.example_camera(16, 12)\n"
            "hdr = R.render_scene_hdr(cam, 2, sc); aov = R.render_aovs(cam, 2, sc)\n"
            "for k in range(2):\n"
            "    try:\n        R.temporal_accumulate(cam, hdr, aov)\n        print('NO ERROR')\n"
            "    except _abi.RbrtGpuError as e:\n        print('CODE', e.code, str(e))\n"
            "img = R.render_scene(cam, 2, sc)\n"
            "print('RENDER', img.pixels.shape, bool(np.array_equal(R.render_scene_hdr(cam, 2, sc), hdr)))\n") % ROOT
    env = dict(os.environ, RBRT_GPU_TEMPORAL_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_temporal.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count(f"CODE {_abi.E_CUDA}") == 2 and r.stdout.count("temporal module is missing") == 2, r.stdout
    assert "RENDER (12, 16, 3) True" in r.stdout, r.stdout


STATIC_OWN_GUIDES_BOUND = 1.42                # measured 1.40 on C1 (DESIGN.md section 15)

# ============================================================================== 4. static camera: the running mean and its variance
def test_static_camera_is_the_running_mean(gpu):
    """α_min = 0, N = 8 frames of S = 4 spp with seeds 21..28 through the accumulator: bit for bit the numpy recurrence.  With the
    guides of one seed for every frame (a static camera's guides do not change) each valid pixel is the running mean, and the RMSE
    against a 4096-spp reference is within 10 % of one 32-spp render's.  With each frame's own guides, edge pixels whose sample-0 id
    changes between seeds restart; that RMSE is pinned (DESIGN.md section 15)."""
    import torch
    scene, cam = workload("c1")
    N, S_ = 8, 4
    ref = R.render_scene_hdr(cam, 4096, scene, seed=12345)
    one = R.render_scene_hdr(cam, N * S_, scene, seed=21)
    fixed = R.render_aovs_device(cam, 4, scene, seed=21, passes=("depth", "normal", "ids"))
    ratios = {}
    for label in ("fixed guides", "own guides"):
        acc = R.TemporalAccumulator(256, 192, alpha_min=0.0)
        hist = None
        for f in range(N):
            hdr, var = R.render_hdr_variance_device(cam, S_, scene, splits=4, seed=21 + f)
            aovs = fixed if label == "fixed guides" else R.render_aovs_device(cam, 4, scene, seed=21 + f, passes=("depth", "normal", "ids"))
            got = acc.step(cam, hdr, var, aovs)
            torch.cuda.synchronize()
            np_in = [hdr.cpu().numpy(), var.cpu().numpy(), {k: v.cpu().numpy() for k, v in aovs.items()}]
            want = T.accumulate(cam, np_in[0], np_in[1], np_in[2], hist, alpha_min=0.0)
            assert all(T.same_bits(g.cpu().numpy(), w) for g, w in zip(got, want)), (label, f)
            hist = {"cam": cam, "hdr": want[0], "var": want[1], "length": want[2], "aovs": np_in[2]}
        valid = np.isfinite(hist["aovs"]["depth"])
        ratios[label] = rmse(want[0], ref) / rmse(one, ref)
        print(f"static camera, {label}: accumulated / {N * S_}-spp RMSE {ratios[label]:.4f}, full history "
              f"{float((want[2] == N).mean()):.3f} of the pixels ({float(valid.mean()):.3f} valid)")
        if label == "fixed guides":
            assert (want[2][valid] == N).all()
    assert ratios["fixed guides"] <= 1.1
    assert ratios["own guides"] <= STATIC_OWN_GUIDES_BOUND


def test_variance_is_calibrated_across_seeds(gpu):
    """Static camera, α_min = 0, 4 frames of 16 spp (K = 4) per sequence, 32 independent sequences: the summed mean var_out is within
    [0.9, 1.1] of the summed across-sequence variance of hdr_out."""
    scene, cam = workload("c1", 128, 96)
    hs, vs = [], []
    for j in range(32):
        hist = None
        for f in range(4):
            hdr, var, aovs = render_frame(scene, cam, 1000 + 4 * j + f, spp=16)
            out = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist, alpha_min=0.0)
            hist = {"cam": cam, "hdr": out[0], "var": out[1], "length": out[2], "aovs": aovs}
        hs.append(out[0].astype(np.float64))
        vs.append(out[1].astype(np.float64))
    hs, vs = np.stack(hs), np.stack(vs)
    ok = np.isfinite(hs).all(0) & np.isfinite(vs).all(0)
    empirical = hs.var(0, ddof=1)[ok].sum()
    predicted = vs.mean(0)[ok].sum()
    print(f"calibration: predicted / empirical = {predicted / empirical:.4f}")
    assert empirical > 0
    assert 0.9 <= predicted / empirical <= 1.1, predicted / empirical


def test_disoccluded_pixels_restart(gpu):
    """A sphere moved with update_elements between two frames of a static camera: every valid pixel whose sample-0 id changed has no
    history (len_out = 1, hdr_out = hdr bit for bit)."""
    scene, cam = workload("c1")
    hdr0, var0, aov0 = render_frame(scene, cam, 5)
    out0 = R.temporal_accumulate(cam, hdr0, aov0, var=var0)
    els = list(scene.elements)
    big = max(range(len(els)), key=lambda k: els[k].radius if isinstance(els[k], R.Sphere) and els[k].radius < 50 else -1)
    c = els[big].center
    els[big] = R.Sphere(R.Vec3(c.x + 0.6 * els[big].radius, c.y, c.z), els[big].radius, els[big].material)
    scene.update_elements(els)
    hdr1, var1, aov1 = render_frame(scene, cam, 6)
    out1 = R.temporal_accumulate(cam, hdr1, aov1, var=var1, history={"cam": cam, "hdr": out0[0], "var": out0[1], "length": out0[2],
                                                                      "aovs": aov0})
    changed = ((aov1["hit_kind"] != aov0["hit_kind"]) | (aov1["elem_idx"] != aov0["elem_idx"])) & (out1[2] > 0)
    print(f"disocclusion: {int(changed.sum())} pixels changed id")
    assert changed.sum() > 100
    assert (out1[2][changed] == 1).all()
    assert np.array_equal(out1[0][changed].view(np.uint32), hdr1[changed].view(np.uint32))
    assert (out1[2] == 2).mean() > 0.25                                   # the rest keeps its history


# ============================================================================== 5. quality over a camera sweep
# RMSE / noisy RMSE, the largest over frames 3..7, pinned with a margin of 0.02 (DESIGN.md section 15).
BOUNDS = {("c1", "spatial"): 0.56, ("c1", "temporal"): 0.53, ("c1", "both"): 0.46,
          ("c2", "spatial"): 0.62, ("c2", "temporal"): 0.55, ("c2", "both"): 0.49,
          ("c4", "spatial"): 0.64, ("c4", "temporal"): 0.56, ("c4", "both"): 0.50}


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_quality_over_a_camera_sweep(gpu, name):
    """8 frames of a sideways sweep (0.04 per frame), 4 spp with K = 4 and seeds 11 + f, guides at 4 spp of the same seed, 4096-spp
    references with seed 12345: variance-guided spatial filter alone, temporal alone, and temporal followed by the spatial filter on its
    var_out."""
    scene, _ = workload(name)
    kw = camkw_of(name)
    hist = None
    worst = {"spatial": 0.0, "temporal": 0.0, "both": 0.0}
    for f in range(8):
        cam = sweep_camera(kw, 256, 192, 0.04 * f)
        hdr, var, aovs = render_frame(scene, cam, 11 + f)
        t = R.temporal_accumulate(cam, hdr, aovs, var=var, history=hist)
        hist = {"cam": cam, "hdr": t[0], "var": t[1], "length": t[2], "aovs": aovs}
        if f < 3:
            continue
        ref = R.render_scene_hdr(cam, 4096, scene, seed=12345)
        base = rmse(hdr, ref)
        r = {"spatial": rmse(R.denoise_variance(hdr, var, aovs)[0], ref) / base, "temporal": rmse(t[0], ref) / base,
             "both": rmse(R.denoise_variance(t[0], t[1], aovs)[0], ref) / base}
        print(f"{name} frame {f}: spatial {r['spatial']:.4f} temporal {r['temporal']:.4f} temporal+spatial {r['both']:.4f} "
              f"history {float((t[2] > 1).mean()):.3f}")
        for k in r:
            worst[k] = max(worst[k], r[k])
        assert r["both"] < r["spatial"], (name, f, r)
    for k, v in worst.items():
        assert v <= BOUNDS[name, k], (name, k, v)
