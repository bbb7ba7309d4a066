"""Multi-GPU INSIDE the C-ABI (csrc/multi.cu) on ONE GPU: rbrt_gpu_init_multi with the same device listed N times runs N
ranks of the collective render — scene replication, interleaved tile shards or sample ranges, per-rank finalise, gather /
sum on rank 0 — through the PEER transport.  The image must equal the one-GPU render bit for bit (tile shards: every pixel
is summed and finalised by exactly one rank) or within f32 re-association (sample shards).
The NCCL transport needs N distinct GPUs: scripts/multi_gpu_check.py runs the same checks there (profiles/)."""
import ctypes as C

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi

from . import scenes as S

pytestmark = pytest.mark.gpu


@pytest.fixture
def comm():
    lib = _abi.lib()
    made = []

    def start(n):
        devs = (C.c_int * n)(*([0] * n))
        _abi.check(lib.rbrt_gpu_init_multi(devs, n, _abi.TRANSPORT_AUTO))
        made.append(n)
        info = _abi.CommInfoC()
        _abi.check(lib.rbrt_gpu_comm_info(info))
        return info.as_dict()

    yield start
    _abi.check(lib.rbrt_gpu_comm_destroy())


def build(fn):
    return fn()


def sample_shard_mean(scene, cam, spp, world, seed):
    """What the PEER sample-sharded render computes: ((a_0 + a_1) + ... + a_{world-1}) * (1/spp) in f32 (k_sum_peers, then k_finalize),
    a_r the sums of an explicit sample shard r of `world` rendered on one GPU."""
    import torch
    W, H = cam.img_width_pix, cam.img_height_pix
    total = None
    for r in range(world):
        buf = torch.empty(H * W * 4, dtype=torch.float32, device="cuda")
        _abi.check(_abi.lib().rbrt_gpu_render_accum_device(scene.handle(), cam.to_c(), spp, R.render.make_opts(
            seed=seed, shard_mode=_abi.SHARD_SAMPLES, shard_rank=r, shard_count=world), buf.data_ptr(), torch.cuda.current_stream().cuda_stream, None))
        a = buf.cpu().numpy().reshape(H, W, 4)[..., :3]
        total = a if total is None else (total + a).astype(np.float32)
    return (total * (np.float32(1.0) / np.float32(spp))).astype(np.float32)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_collective_render_equals_one_gpu(gpu, comm, world):
    cam = S.example_camera(150, 101)                                   # ragged: partial tiles on both edges
    want_u8 = R.render_scene(cam, 5, S.small_mesh_scene(4), seed=12).pixels
    want_hdr = R.render_scene_hdr(cam, 5, S.small_mesh_scene(4), seed=12)
    want_samples = sample_shard_mean(S.small_mesh_scene(4), cam, 5, world, seed=12)
    info = comm(world)
    assert info["active"] == 1 and info["world"] == world and info["local_devices"] == world and info["transport"] == _abi.TRANSPORT_PEER
    scene = S.small_mesh_scene(4)                                      # created under the communicator: built once, replicated
    st = {}
    got = R.render_scene(cam, 5, scene, seed=12, stats=st)
    assert np.array_equal(got.pixels, want_u8)
    assert st["paths"] == 150 * 101 * 5
    hdr = R.render_scene_hdr(cam, 5, scene, seed=12)
    assert np.array_equal(hdr.view(np.uint32), want_hdr.view(np.uint32))
    # sample-range shards: rank 0's sums plus the other ranks' in rank order, then the 1/spp scale, all in f32
    hs = R.render_scene_hdr(cam, 5, scene, seed=12, shard_mode=_abi.SHARD_SAMPLES)
    assert np.array_equal(hs.view(np.uint32), want_samples.view(np.uint32))
    assert np.allclose(hs, want_hdr, rtol=1e-5, atol=1e-6)
    # an explicit shard placed by the host still works under a communicator, and a LOCAL scene is not sharded
    one = R.render_scene_hdr(cam, 5, scene, seed=12, shard_mode=_abi.SHARD_TILES, shard_rank=1, shard_count=2)
    assert one.any() and not np.array_equal(one, want_hdr)
    local = S.small_mesh_scene(4, local=True)
    assert np.array_equal(R.render_scene(cam, 5, local, seed=12).pixels, want_u8)
    scene.close(); local.close()


def test_collective_frames_device_and_pipeline(gpu, comm):
    """rbrt_gpu_render_frames_device (several frames per batch, device outputs) and the FramePipeline on top of it."""
    import torch
    cam_a, cam_b = S.example_camera(96, 64), S.quirk_camera(96, 64)
    base = S.small_mesh_scene(3)
    want = [R.render_scene(c, 4, base, seed=s).pixels for c, s in ((cam_a, 1), (cam_b, 2), (cam_a, 3))]
    comm(4)
    scene = S.small_mesh_scene(3)
    pipe = R.FramePipeline(96, 64, depth=2, frames_per_batch=2)
    out = []
    for k, (c, s) in enumerate(((cam_a, 1), (cam_b, 2), (cam_a, 3))):
        out += pipe.submit(c, 4, scene, tag=k, seed=s)
    out += pipe.drain()
    assert [t for _, t in out] == [0, 1, 2]
    for (img, t), w in zip(out, want):
        assert np.array_equal(img.pixels, w), f"frame {t}"
    scene.close()


def test_comm_errors(gpu, comm):
    lib = _abi.lib()
    assert lib.rbrt_gpu_init_multi(None, 0, 0) == _abi.E_INVALID
    assert lib.rbrt_gpu_init_multi(None, 1, 9) == _abi.E_INVALID
    devs = (C.c_int * 2)(0, 0)
    assert lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_NCCL) == _abi.E_INVALID      # NCCL cannot put two ranks on one GPU
    comm(2)
    assert lib.rbrt_gpu_init_multi(devs, 2, _abi.TRANSPORT_PEER) == _abi.E_INVALID      # already active
    assert lib.rbrt_gpu_init(0) == 0
