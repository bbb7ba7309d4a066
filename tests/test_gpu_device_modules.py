"""The host side of the device modules (csrc/api.cu) on the GPU: the module loader on the refit path, the staging block that the
host-pointer AOV and denoise calls share, and the timing events that every call with stats shares.

Each module's kernels are tested in its own file (test_gpu_update.py, test_gpu_aov.py, test_gpu_query.py, test_gpu_denoise.py,
test_gpu_variance.py); here the calls of different modules run one after another in one process, so that state one of them leaves
behind would show in the next."""
import os
import subprocess
import sys

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import scenes as S
from .test_denoise_host import scene_like
from .test_variance_host import variance_like

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODULES = [os.path.join(ROOT, "rbrt_b200", f"librbrt_gpu_{m}.so") for m in ("update", "aov", "query", "denoise", "variance")]


@pytest.fixture(scope="module", autouse=True)
def device_modules():
    """The session fixture only builds librbrt_gpu.so when it is missing; the modules are built here when one is."""
    if not all(os.path.exists(m) for m in MODULES):
        subprocess.run(["make", "-C", os.path.join(ROOT, "rbrt_b200", "csrc")], check=True)
    return MODULES


def u32(x):
    """A numpy array or CUDA tensor as a numpy array of its bit patterns (uint8 data stays uint8)."""
    import torch
    if isinstance(x, torch.Tensor):
        torch.cuda.synchronize()
        x = x.cpu().numpy()
    x = np.ascontiguousarray(x)
    return x if x.dtype == np.uint8 else x.view(np.uint32)


def assert_same(host, dev, what):
    assert set(host) == set(dev), what
    for k in host:
        assert np.array_equal(u32(host[k]), u32(dev[k]).reshape(u32(host[k]).shape)), f"{what}: {k}"


def test_missing_refit_module_is_refused_and_a_rebuild_still_works(gpu):
    """Without librbrt_gpu_update.so a refit fails with a message naming the module.  A rebuild does not need the module: in the same
    process it succeeds, and the render of the rebuilt mesh is the oracle's."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, rbrt_b200 as R\nfrom oracle import oracle_ffi\nfrom rbrt_b200 import _abi\n"
            "from tests.test_gpu_update import hdr, mesh_scene, oracle_hdr, twist\n"
            "R.gpu_init(0); sc = mesh_scene(); before = hdr(sc); new = twist(sc.triangle_meshes[0].triangles)\n"
            "for k in range(2):\n"
            "    try:\n        sc.update_mesh(0, new)\n        print('NO ERROR')\n"
            "    except _abi.RbrtGpuError as e:\n        print('CODE', e.code, str(e))\n"
            "sc.update_mesh(0, new, rebuild=True); after = hdr(sc)\n"
            "print('CHANGED', not np.array_equal(after.view(np.uint32), before.view(np.uint32)))\n"
            "print('ORACLE', np.array_equal(after.view(np.uint32), oracle_hdr(oracle_ffi, sc).view(np.uint32)))\n") % ROOT
    env = dict(os.environ, RBRT_GPU_UPDATE_LIB=os.path.join(ROOT, "no-such-dir", "librbrt_gpu_update.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count(f"CODE {_abi.E_CUDA}") == 2 and r.stdout.count("refit module is missing") == 2, r.stdout
    assert "CHANGED True" in r.stdout and "ORACLE True" in r.stdout, r.stdout


def test_host_variants_share_the_staging_block(gpu):
    """Host-pointer AOV and denoise calls of different sizes, in an order that grows the shared block, reuses it after the other
    feature and frees it: each equals the device-pointer variant of the same call bit for bit."""
    import torch
    scene = S.small_mesh_scene(3)

    def aov(W, H):
        cam = S.example_camera(W, H)
        assert_same(R.render_aovs(cam, 2, scene, seed=5), R.render_aovs_device(cam, 2, scene, seed=5), f"AOV {W}x{H}")

    def denoise(W, H, with_var):
        c, a, n, z = scene_like(H, W, W)
        guides = {"depth": z, "normal": n, "albedo": a}
        t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
        tguides = {k: t(v) for k, v in guides.items()}
        if with_var:
            v = variance_like(H, W, W)
            host = R.denoise_variance(c, v, guides)
            dev = R.denoise_variance_device(t(c), t(v), tguides)
        else:
            host = R.denoise(c, guides)
            dev = R.denoise_device(t(c), tguides)
        assert_same({"hdr": host[0], "rgb": host[1].pixels}, {"hdr": dev[0], "rgb": dev[1]}, f"denoise {W}x{H} var={with_var}")

    aov(1920, 1080)                                                       # grows the block
    denoise(64, 48, False)                                                # reuses it after the AOV call
    aov(64, 48)
    denoise(1920, 1080, True)                                             # grows it again
    _abi.check(_abi.lib().rbrt_gpu_release_cache())                       # frees it
    aov(64, 48)
    denoise(64, 48, False)


def test_calls_with_stats_share_the_timing_events(gpu):
    """Query, AOV, denoise and variance calls with stats, alternated on the default stream for three rounds: each reports a device time,
    and its counters do not change from round to round."""
    import torch
    scene = S.small_mesh_scene(3)
    cam = S.example_camera(64, 48)
    rays = torch.from_numpy(np.ascontiguousarray(S.random_rays(5000, (5.0, 1.4, -12.5), 4.0, 2), np.float32)).cuda()
    c, a, n, z = scene_like(48, 64, 3)
    guides = {"depth": z, "normal": n, "albedo": a}
    v = variance_like(48, 64, 3)
    calls = {"query": lambda st: scene.intersect_device(rays, stats=st),
             "aov": lambda st: R.render_aovs(cam, 2, scene, seed=5, stats=st),
             "denoise": lambda st: R.denoise(c, guides, stats=st),
             "variance": lambda st: R.render_scene_hdr_variance(cam, 8, scene, splits=2, seed=5, stats=st),
             "denoise_variance": lambda st: R.denoise_variance(c, v, guides, stats=st)}
    first = {}
    for rnd in range(3):
        for name, f in calls.items():
            st = {}
            f(st)
            assert st["ms_device"] > 0, (rnd, name, st)
            counters = {k: st[k] for k in ("rays", "node_visits", "tri_tests", "launches")}
            assert counters == first.setdefault(name, counters), (rnd, name, counters, first[name])
    assert first["query"]["node_visits"] > 0 and first["aov"]["node_visits"] > 0 and first["variance"]["rays"] > 0
