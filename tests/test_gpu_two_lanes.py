"""Two lanes (RBRT_OPT_SPLIT_BATCHES, render.cu render_accum): a lone frame's samples cut into at least two batches that alternate
between the caller's stream with wavefront pool p and an internal stream with pool 4 + p.  rbrt_gpu_render / rbrt_gpu_render_hdr
switch to it on their own from 2^26 paths per GPU, so it is what C3, every rank of C5 and the CLI at those sizes run.

The bar is the project's usual one: bit-identical HDR sums and u8 pixels.  Small frames are held against the CPU oracle; frames too
large for it against the one-lane render of the same frame (rbrt_gpu_render_accum_device without the flag, then
rbrt_gpu_finalize_device), which the rest of the suite pins to the oracle, plus an oracle pixel lattice.  Stats: rays / paths equal
the oracle's, and under RBRT_OPT_NO_TAIL_KERNEL (launch sequence fixed on the host) iterations = batches x (max_depth + 1), with the
batch count from planned_batches(), a restatement of the planner."""
import ctypes as C
import os

import numpy as np
import pytest

import rbrt_b200 as R
from rbrt_b200 import _abi
from rbrt_b200.vec3 import Vec3

from . import scenes as S
from .test_gpu_multi import sample_shard_mean
from .test_gpu_trace import mixed_element_scene

pytestmark = pytest.mark.gpu

T26 = 1 << 26                      # rbrt_gpu_render's switch: two lanes from 2^26 paths per GPU (api.cu render_host)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_same(got, ref, what):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    ne = (bits(got) != bits(ref)).reshape(-1, 4 if ref.ndim == 1 else ref.shape[-1]).any(axis=1)      # per pixel: sums [H*W*4], images [.., 3]
    assert not ne.any(), f"{what}: {int(ne.sum())} of {ne.size} pixels differ, first at pixel {int(np.argmax(ne))}"


def stream_ptr(stream=None):
    import torch
    return (stream or torch.cuda.current_stream()).cuda_stream


def accum(scene, cam, spp, **kw):
    """rbrt_gpu_render_accum_device on the current stream, with stats (so it blocks): (per-pixel sums [H*W*4], stats dict)."""
    import torch
    W, H = cam.img_width_pix, cam.img_height_pix
    buf = torch.empty(H * W * 4, dtype=torch.float32, device="cuda")
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_accum_device(scene.handle(), cam.to_c(), spp, R.render.make_opts(**kw), buf.data_ptr(),
                                                       stream_ptr(), st))
    return buf.cpu().numpy(), st.as_dict()


def finalize(sums, W, H, spp):
    """rbrt_gpu_finalize_device of host sums: (hdr [H,W,3] f32, rgb [H,W,3] u8)."""
    import torch
    a = torch.from_numpy(np.ascontiguousarray(sums, np.float32)).cuda()
    hdr = torch.empty(H * W * 3, dtype=torch.float32, device="cuda")
    rgb = torch.empty(H * W * 3, dtype=torch.uint8, device="cuda")
    _abi.check(_abi.lib().rbrt_gpu_finalize_device(a.data_ptr(), W, H, spp, rgb.data_ptr(), hdr.data_ptr(), stream_ptr()))
    return hdr.cpu().numpy().reshape(H, W, 3), rgb.cpu().numpy().reshape(H, W, 3)


def one_lane(scene, cam, spp, **kw):
    """The reference of a frame too large for the oracle: the one-lane sums, finalised on the device: (sums, hdr, rgb, stats)."""
    assert not kw.get("split")
    sums, st = accum(scene, cam, spp, **kw)
    hdr, rgb = finalize(sums, cam.img_width_pix, cam.img_height_pix, spp)
    return sums, hdr, rgb, st


def planned_batches(cam, spp, n_frames=1, batch_paths=0, max_depth=0, split=False, pool_limit=0,
                    shard_mode=_abi.SHARD_NONE, shard_rank=0, shard_count=0):
    """How many wavefront batches render_accum cuts a frame into (render.cu), restated.  batch_paths 0 (the default plan) is only
    restated for frames of at most 2^21 paths, which it holds in one batch (one per lane when split)."""
    W, H = cam.img_width_pix, cam.img_height_pix
    tiles = -(-W // 8) * -(-H // 4)                                    # 8 x 4 tiles: pixel SLOTS, not pixels
    rank, count, s0, s1 = 0, 1, 0, spp
    if shard_count > 1 and shard_mode == _abi.SHARD_TILES:
        rank, count = shard_rank, shard_count
    elif shard_count > 1 and shard_mode == _abi.SHARD_SAMPLES:
        s0, s1 = spp * shard_rank // shard_count, spp * (shard_rank + 1) // shard_count
    mine = (tiles - rank + count - 1) // count if tiles > rank else 0
    PF = mine * 32 * n_frames
    S_all = s1 - s0
    if not batch_paths:
        assert S_all * PF <= 1 << 21, "the default plan depends on free HBM above 2^21 paths: pin batch_paths"
        batch_paths = S_all * PF
    if pool_limit:
        batch_paths = min(batch_paths, max(pool_limit // (76 + 2 * max(max_depth or 50, 1)), 1))
    S_b = min(max(batch_paths // PF, 1), S_all)
    if split and S_all >= 2:
        S_b = min(S_b, (S_all + 1) // 2)                               # at least two batches, one per lane
    return -(-S_all // S_b)


_ORACLE = {}


def oracle_sums(oracle, key, scene, cam, spp, **kw):
    """The oracle's per-pixel sums of a frame, computed once per module (key names the scene)."""
    k = (key, cam.img_width_pix, cam.img_height_pix, spp, tuple(sorted(kw.items())))
    if k not in _ORACLE:
        st = {}
        sums = oracle.OracleScene.from_scene(scene).render_accum(cam.to_c(), spp, _abi.RenderOptsC(**kw), st)
        _ORACLE[k] = (sums, st)
    return _ORACLE[k]


@pytest.fixture
def pool_limit():
    lib = _abi.lib()
    yield lambda n: _abi.check(lib.rbrt_gpu_set_pool_limit(n))
    _abi.check(lib.rbrt_gpu_set_pool_limit(0))


@pytest.fixture
def comm():
    lib = _abi.lib()
    made = []

    def start(n):
        devs = (C.c_int * n)(*([0] * n))
        _abi.check(lib.rbrt_gpu_init_multi(devs, n, _abi.TRANSPORT_PEER))
        made.append(n)
    yield start
    if made:
        _abi.check(lib.rbrt_gpu_comm_destroy())
    R.gpu_init(0)


@pytest.fixture
def release_after():
    """Big frames leave pools of tens of GB behind: hand them back when the test is done."""
    yield
    import torch
    torch.cuda.synchronize()
    _abi.check(_abi.lib().rbrt_gpu_release_cache())


# ============================================================================== 1. small frames against the oracle
SCENES = {
    "mesh": (lambda: S.small_mesh_scene(4), lambda: S.example_camera(128, 96)),
    "ragged": (lambda: S.small_mesh_scene(4), lambda: S.example_camera(33, 17)),
    "spheres": (S.spheres_scene, lambda: S.example_camera(96, 64)),             # no mesh: the tail kernel right after k_generate
    "mixed": (mixed_element_scene, lambda: S.example_camera(96, 64)),           # BasicTriangle elements: the `et` kernels
    "quirk": (S.quirk_scene, lambda: S.quirk_camera(64, 48)),
}
_SCENE_CACHE = {}


def scene_of(name):
    if name not in _SCENE_CACHE:
        mk_scene, mk_cam = SCENES[name]
        _SCENE_CACHE[name] = (mk_scene(), mk_cam())
    return _SCENE_CACHE[name]


CASES = [("mesh", s) for s in (2, 3, 5, 8)] + [("ragged", s) for s in (1, 2, 3, 5, 8)] + [("spheres", s) for s in (2, 3, 5, 8)] \
    + [("mixed", s) for s in (2, 5)] + [("quirk", s) for s in (3, 8)]


@pytest.mark.parametrize("name,spp", CASES)
def test_small_frames_equal_the_oracle(gpu, oracle, name, spp):
    """Every batch plan of the lane logic: the default (one batch per lane), one sample per batch (spp batches ping-ponging), two
    samples per batch, W*H*3 paths; odd counts put a shorter last batch on lane 0 or lane 1; one sample falls back to one lane."""
    scene, cam = scene_of(name)
    W, H = cam.img_width_pix, cam.img_height_pix
    seed = 40 + spp
    ref, ost = oracle_sums(oracle, name, scene, cam, spp, seed=seed)
    PF = -(-W // 8) * -(-H // 4) * 32
    for bp in (0, PF, 2 * PF, W * H * 3):
        for extra in ({}, {"no_tail_kernel": True}):
            got, st = accum(scene, cam, spp, seed=seed, batch_paths=bp, split=True, **extra)
            what = f"{name} {W}x{H}x{spp} batch_paths {bp} {extra}"
            assert_same(got, ref, what)
            assert (st["rays"], st["paths"], st["nan_rays"]) == (ost["rays"], ost["paths"], ost["nan_rays"]), (what, st, ost)
            n = planned_batches(cam, spp, batch_paths=bp, split=True)
            assert n >= (2 if spp >= 2 else 1), (what, n)
            if extra:
                assert st["iterations"] == n * 51, (what, st["iterations"], n)


def test_pool_limit_forces_many_batches_on_both_lanes(gpu, oracle, pool_limit):
    scene, cam = scene_of("mesh")
    spp, seed = 8, 48
    ref, ost = oracle_sums(oracle, "mesh", scene, cam, spp, seed=seed)
    PF = 16 * 24 * 32
    per_path = 76 + 2 * 50
    for limit, want in ((1, 8), (3 * PF * per_path, 3), (3 * PF * per_path - 1, 4), (PF * per_path, 8)):
        pool_limit(limit)
        for extra in ({}, {"no_tail_kernel": True}):
            got, st = accum(scene, cam, spp, seed=seed, split=True, **extra)
            assert_same(got, ref, f"pool limit {limit} {extra}")
            assert st["rays"] == ost["rays"] and st["paths"] == ost["paths"]
            n = planned_batches(cam, spp, split=True, pool_limit=limit)
            assert n == want, (limit, n)
            if extra:
                assert st["iterations"] == n * 51, (limit, st["iterations"], n)


def test_options_pools_and_shards(gpu, oracle):
    """The brute-force integrator, no tail kernel, an early tail hand-over, pools 1-3 (second lanes 5-7), an explicit tile shard and an
    explicit sample shard whose range starts at 5 (rank 2 of 3 at 8 spp: samples 5, 6, 7)."""
    scene, cam = scene_of("mesh")
    W, H = 128, 96
    PF = 16 * 24 * 32
    ref, ost = oracle_sums(oracle, "mesh", scene, cam, 5, seed=45)
    ways = [{"trace_mode": _abi.TRACE_BRUTE}, {"trace_mode": _abi.TRACE_BRUTE, "batch_paths": PF}, {"no_tail_kernel": True, "batch_paths": PF},
            {"pool": 1}, {"pool": 2, "batch_paths": PF}, {"pool": 3, "batch_paths": 2 * PF}]
    for kw in ways:
        got, st = accum(scene, cam, 5, seed=45, split=True, **kw)
        assert_same(got, ref, f"{kw}")
        assert st["rays"] == ost["rays"] and st["paths"] == ost["paths"], kw
    os.environ["RBRT_TAIL_RAYS"] = "3000"                              # early hand-over: most of each batch runs in the tail kernel
    try:
        for bp in (0, PF):
            got, st = accum(scene, cam, 5, seed=45, split=True, batch_paths=bp)
            assert_same(got, ref, f"RBRT_TAIL_RAYS=3000 batch_paths {bp}")
            assert st["rays"] == ost["rays"]
    finally:
        del os.environ["RBRT_TAIL_RAYS"]
    # explicit tile shard
    sh = dict(shard_mode=_abi.SHARD_TILES, shard_rank=1, shard_count=3)
    ref_t, ost_t = oracle_sums(oracle, "mesh", scene, cam, 5, seed=45, **sh)
    for bp in (0, PF // 3):
        for extra in ({}, {"no_tail_kernel": True}):
            got, st = accum(scene, cam, 5, seed=45, split=True, batch_paths=bp, **sh, **extra)
            assert_same(got, ref_t, f"tile shard batch_paths {bp} {extra}")
            assert st["rays"] == ost_t["rays"] and st["paths"] == ost_t["paths"]
            if extra:
                assert st["iterations"] == planned_batches(cam, 5, batch_paths=bp, split=True, **sh) * 51
    # explicit sample shard that does not start at sample 0
    sh = dict(shard_mode=_abi.SHARD_SAMPLES, shard_rank=2, shard_count=3)
    ref_s, ost_s = oracle_sums(oracle, "mesh", scene, cam, 8, seed=48, **sh)
    assert ost_s["paths"] == W * H * 3
    for bp in (0, PF):
        for extra in ({}, {"no_tail_kernel": True}, {"pool": 2}):
            got, st = accum(scene, cam, 8, seed=48, split=True, batch_paths=bp, **sh, **extra)
            assert_same(got, ref_s, f"sample shard 2/3 batch_paths {bp} {extra}")
            assert st["rays"] == ost_s["rays"] and st["paths"] == ost_s["paths"]
            if extra.get("no_tail_kernel"):
                n = planned_batches(cam, 8, batch_paths=bp, split=True, **sh)
                assert n == (3 if bp else 2) and st["iterations"] == n * 51


def test_deep_paths_grow_the_second_lanes_pool(gpu, oracle):
    """max_depth 200 and 1024 grow depth_cap of pool 0 and of pool 4; then depth 50 again."""
    scene, cam = S.deep_path_scene(), S.deep_path_camera(32, 24)
    PF = 4 * 6 * 32
    for depth in (200, 1024, 50):
        ref, ost = oracle_sums(oracle, "deep", scene, cam, 3, seed=19, max_depth=depth)
        for bp in (0, PF):
            for extra in ({}, {"no_tail_kernel": True}):
                got, st = accum(scene, cam, 3, seed=19, max_depth=depth, split=True, batch_paths=bp, **extra)
                assert_same(got, ref, f"depth {depth} batch_paths {bp} {extra}")
                assert st["rays"] == ost["rays"] and st["paths"] == ost["paths"]
                if extra:
                    assert st["iterations"] == planned_batches(cam, 3, batch_paths=bp, split=True, max_depth=depth) * (depth + 1)


def frame_cams(n, w=64, h=48):
    from rbrt_b200 import synth
    cb = synth.example_camera_blueprint()
    return [R.Camera.new(Vec3(cb.camera_position.x + 0.3 * k, cb.camera_position.y + 0.1 * k, cb.camera_position.z), cb.camera_look_at,
                         cb.camera_up, h, w, cb.camera_focal_length_mm) for k in range(n)]


@pytest.mark.parametrize("n_frames", [2, 3, 4])
def test_several_frames_per_batch(gpu, oracle, n_frames):
    """rbrt_gpu_render_accum_device_frames and rbrt_gpu_render_frames_device with the flag: each frame equals its lone oracle render."""
    import torch
    lib = _abi.lib()
    scene = S.small_mesh_scene(3)
    cams = frame_cams(n_frames)
    W, H, spp = 64, 48, 3
    seeds = [70 + k for k in range(n_frames)]
    refs = [oracle_sums(oracle, f"frames{k}", scene, c, spp, seed=s) for k, (c, s) in enumerate(zip(cams, seeds))]
    cams_c = (_abi.CameraC * n_frames)(*[c.to_c() for c in cams])
    seeds_c = (C.c_uint64 * n_frames)(*seeds)
    PF = 8 * 12 * 32 * n_frames
    for bp in (0, PF):
        for extra in ({}, {"no_tail_kernel": True}):
            bufs = [torch.empty(H * W * 4, dtype=torch.float32, device="cuda") for _ in range(n_frames)]
            ptrs = (C.c_void_p * n_frames)(*[b.data_ptr() for b in bufs])
            st = _abi.StatsC()
            _abi.check(lib.rbrt_gpu_render_accum_device_frames(scene.handle(), cams_c, seeds_c, n_frames, spp,
                                                               R.render.make_opts(split=True, batch_paths=bp, **extra), ptrs, stream_ptr(), st))
            for k, (b, (ref, _)) in enumerate(zip(bufs, refs)):
                assert_same(b.cpu().numpy(), ref, f"frame {k} of {n_frames}, batch_paths {bp} {extra}")
            assert st.rays == sum(o["rays"] for _, o in refs) and st.paths == sum(o["paths"] for _, o in refs)
            if extra:
                assert st.iterations == planned_batches(cams[0], spp, n_frames=n_frames, batch_paths=bp, split=True) * 51
    hdrs = [torch.empty(H * W * 3, dtype=torch.float32, device="cuda") for _ in range(n_frames)]
    rgbs = [torch.empty(H * W * 3, dtype=torch.uint8, device="cuda") for _ in range(n_frames)]
    _abi.check(lib.rbrt_gpu_render_frames_device(scene.handle(), cams_c, seeds_c, n_frames, spp, R.render.make_opts(split=True, batch_paths=PF),
                                                 (C.c_void_p * n_frames)(*[r.data_ptr() for r in rgbs]),
                                                 (C.c_void_p * n_frames)(*[h.data_ptr() for h in hdrs]), stream_ptr(), None))
    torch.cuda.synchronize()
    for k, (ref, _) in enumerate(refs):
        rgb_ref, hdr_ref = oracle.finalize(ref, W, H, spp)
        assert_same(hdrs[k].cpu().numpy().reshape(H, W, 3), hdr_ref, f"render_frames_device frame {k} hdr")
        assert np.array_equal(rgbs[k].cpu().numpy().reshape(H, W, 3), rgb_ref), f"render_frames_device frame {k} u8"


def test_visit_counts_match_one_lane(gpu):
    """COUNT_VISITS totals under RBRT_OPT_NO_TAIL_KERNEL do not depend on the batch plan of one lane, so two lanes must give them too."""
    scene, cam = scene_of("mesh")
    PF = 16 * 24 * 32
    keys = ("rays", "node_visits", "tri_tests", "traversed_rays")
    one = [accum(scene, cam, 5, seed=3, count_visits=True, no_tail_kernel=True, batch_paths=bp)[1] for bp in (0, PF, 2 * PF)]
    want = {k: one[0][k] for k in keys}
    assert all({k: o[k] for k in keys} == want for o in one), one
    for bp in (0, PF, 2 * PF):
        st = accum(scene, cam, 5, seed=3, count_visits=True, no_tail_kernel=True, batch_paths=bp, split=True)[1]
        assert {k: st[k] for k in keys} == want, (bp, st)


# ============================================================================== 2. the automatic switch and its threshold
def lattice_check(oracle, scene, cam, spp, seed, hdr, stride, what):
    """The oracle on the pixel lattice (row % stride_y == 0, col % stride_x == 0) against a finalised frame."""
    sx, sy = stride if isinstance(stride, tuple) else (stride, stride)
    W, H = cam.img_width_pix, cam.img_height_pix
    _, sub = oracle.render_subset(oracle.OracleScene.from_scene(scene), cam.to_c(), spp, sx, sy, _abi.RenderOptsC(seed=seed), want_image=True)
    _, ref = oracle.finalize(sub, W, H, spp)
    assert_same(hdr[::sy, ::sx], ref[::sy, ::sx], f"{what}: oracle lattice")


@pytest.mark.parametrize("width,split", [(1024, True), (1023, False)])
def test_automatic_switch_at_two_to_the_26(gpu, oracle, release_after, width, split):
    """1024 x 1024 x 64 = 2^26 paths switches to two lanes, 1023 x 1024 x 64 does not; each image equals the one-lane render bit for
    bit and the oracle on a lattice.  With batch_paths pinned the plan is one batch, or one per lane."""
    scene, cam = S.spheres_scene(), S.example_camera(width, 1024)
    spp, seed = 64, 5
    assert (width * 1024 * spp >= T26) == split
    sums, hdr1, rgb1, st1 = one_lane(scene, cam, spp, seed=seed)
    st = {}
    hdr = R.render_scene_hdr(cam, spp, scene, stats=st, seed=seed)
    assert_same(hdr, hdr1, f"{width}x1024x64 render_scene_hdr vs one lane")
    assert st["rays"] == st1["rays"] and st["paths"] == st1["paths"] == width * 1024 * spp
    assert np.array_equal(R.render_scene(cam, spp, scene, seed=seed).pixels, rgb1), f"{width}x1024x64 render_scene vs one lane"
    lattice_check(oracle, scene, cam, spp, seed, hdr, 32, f"{width}x1024x64")
    kw = dict(seed=seed, max_depth=3, no_tail_kernel=True, batch_paths=1 << 27)
    _, hdr_d1, _, _ = one_lane(scene, cam, spp, **kw)
    st = {}
    assert_same(R.render_scene_hdr(cam, spp, scene, stats=st, **kw), hdr_d1, f"{width}x1024x64 depth 3")
    assert st["iterations"] == (2 if split else 1) * 4, st


@pytest.mark.parametrize("width,split", [(1024, True), (1023, False)])
def test_automatic_switch_divides_by_the_shard_count(gpu, release_after, width, split):
    """An explicit tile shard of two: each shard holds 2^26 paths of a 1024 x 1024 x 128 frame (two lanes), or fewer at 1023."""
    scene, cam = S.spheres_scene(), S.example_camera(width, 1024)
    spp = 128
    for kw in (dict(seed=6), dict(seed=6, max_depth=3, no_tail_kernel=True, batch_paths=1 << 27)):
        sh = dict(shard_mode=_abi.SHARD_TILES, shard_rank=1, shard_count=2, **kw)
        _, hdr1, rgb1, st1 = one_lane(scene, cam, spp, **sh)
        st = {}
        assert_same(R.render_scene_hdr(cam, spp, scene, stats=st, **sh), hdr1, f"{width} shard 1/2 {kw}")
        assert st["rays"] == st1["rays"] and st["paths"] == st1["paths"]
        if "no_tail_kernel" in kw:
            assert st["iterations"] == (2 if split else 1) * 4, st
        else:
            assert np.array_equal(R.render_scene(cam, spp, scene, **sh).pixels, rgb1)


# ============================================================================== 3. production shapes
def test_c3_two_lanes_equal_one_lane(gpu, oracle, release_after):
    """C3 (1920 x 1080 x 64 = 132.7 M paths) as rbrt_gpu_render_hdr issues it: two lanes on their own."""
    scene, cam = S.big_scene(8)
    spp, seed = 64, 2024
    sums, hdr1, rgb1, st1 = one_lane(scene, cam, spp, seed=seed)
    st = {}
    hdr = R.render_scene_hdr(cam, spp, scene, stats=st, seed=seed)
    assert_same(hdr, hdr1, "C3 two lanes vs one lane")
    assert st["rays"] == st1["rays"] and st["paths"] == st1["paths"] == 1920 * 1080 * 64 and st["nan_rays"] == st1["nan_rays"]
    assert np.array_equal(R.render_scene(cam, spp, scene, seed=seed).pixels, rgb1), "C3 u8"
    lattice_check(oracle, scene, cam, spp, seed, hdr, 120, "C3")     # 16 x 9 pixels


def test_c5_sample_shard_two_lanes_equal_one_lane(gpu, release_after):
    """C5 (3840 x 2160), sample shard rank 3 of 8 at 384 spp: 48 samples, at least three batches (the plan holds at most 2^27 paths)."""
    scene, cam = S.big_scene(9)
    sh = dict(seed=9, shard_mode=_abi.SHARD_SAMPLES, shard_rank=3, shard_count=8)
    a1, st1 = accum(scene, cam, 384, **sh)
    a2, st2 = accum(scene, cam, 384, split=True, **sh)
    assert_same(a2, a1, "C5 sample shard 3/8: two lanes vs one lane")
    assert st2["rays"] == st1["rays"] and st2["paths"] == st1["paths"] == 3840 * 2160 * 48
    assert (a1 > 0).any()


# ============================================================================== 4. ordering against the other users of the streams and pools
def test_enqueue_only_split_frames_around_an_update_and_destroy(gpu, oracle):
    import torch
    from .test_gpu_update import scale, twist
    scene = S.small_mesh_scene(3)
    a = scene.triangle_meshes[0].triangles.copy()
    b = scale(twist(a, 1.5), 1.3)
    c = S.example_camera(96, 64)
    spp, seed = 5, 11
    ref = {g: oracle.OracleScene.from_scene(R.Scene(list(scene.elements), [R.TriangleMesh(t, scene.triangle_meshes[0].material)]))
           .render_accum(c.to_c(), spp, _abi.RenderOptsC(seed=seed)) for g, t in (("A", a), ("B", b))}
    lib = _abi.lib()
    streams = [torch.cuda.Stream() for _ in range(3)]
    bufs = [torch.empty(64 * 96 * 4, dtype=torch.float32, device="cuda") for _ in range(3)]

    def enqueue(k):
        _abi.check(lib.rbrt_gpu_render_accum_device(scene.handle(), c.to_c(), spp, R.render.make_opts(seed=seed, pool=k, split=True,
                                                    batch_paths=12 * 16 * 32), bufs[k].data_ptr(), streams[k].cuda_stream, None))
    enqueue(0)
    scene.update_mesh(0, b)
    enqueue(1)
    scene.update_mesh(0, a)
    enqueue(2)
    scene.update_mesh(0, b)
    scene.close()                                                         # destroyed with three frames and an update in flight
    torch.cuda.synchronize()
    for k, g in enumerate("ABA"):
        assert_same(bufs[k].cpu().numpy(), ref[g], f"frame {k} on {g}")
    assert (bits(ref["A"]) != bits(ref["B"])).any()


def test_other_users_of_the_second_lanes_pool(gpu, oracle):
    """On one side stream, pool 0, enqueue-only: a split render, the variance render (its second lane is pool 4 on another internal
    stream), a split render with a larger batch (pool 4 grows), a split render with a larger max_depth (depth_cap grows)."""
    import torch
    scene, cam = S.small_mesh_scene(3), S.example_camera(64, 48)
    W, H = 64, 48
    PF = 8 * 12 * 32
    var_want = R.render_scene_hdr_variance(cam, 8, scene, splits=4, seed=31)
    jobs = [dict(spp=4, seed=30, batch_paths=PF), None, dict(spp=6, seed=32), dict(spp=4, seed=33, max_depth=200)]
    refs = [None if j is None else oracle_sums(oracle, "mesh3", scene, cam, j["spp"], seed=j["seed"], max_depth=j.get("max_depth", 0))[0]
            for j in jobs]
    lib = _abi.lib()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        bufs = [torch.empty(H * W * 4, dtype=torch.float32, device="cuda") for _ in jobs]
    out = []
    for j, b in zip(jobs, bufs):
        if j is None:
            out.append(R.render_hdr_variance_device(cam, 8, scene, splits=4, stream=s, seed=31))
            continue
        kw = {k: v for k, v in j.items() if k != "spp"}
        _abi.check(lib.rbrt_gpu_render_accum_device(scene.handle(), cam.to_c(), j["spp"], R.render.make_opts(split=True, **kw), b.data_ptr(),
                                                    s.cuda_stream, None))
        out.append(b)
    s.synchronize()
    for k, (o, ref) in enumerate(zip(out, refs)):
        if ref is None:
            assert_same(o[0].cpu().numpy(), var_want[0], "variance render: mean")
            assert_same(o[1].cpu().numpy(), var_want[1], "variance render: variance")
        else:
            assert_same(o.cpu().numpy(), ref, f"split render {k} ({jobs[k]})")


def test_two_split_frames_in_flight(gpu, oracle):
    import torch
    scene, cam = S.small_mesh_scene(3), S.example_camera(96, 64)
    refs = [oracle_sums(oracle, "mesh3", scene, cam, 6, seed=60 + p)[0] for p in range(2)]
    lib = _abi.lib()
    streams = [torch.cuda.Stream() for _ in range(2)]
    for rnd in range(2):
        bufs = []
        for p in range(2):
            with torch.cuda.stream(streams[p]):
                bufs.append(torch.empty(64 * 96 * 4, dtype=torch.float32, device="cuda"))
            _abi.check(lib.rbrt_gpu_render_accum_device(scene.handle(), cam.to_c(), 6, R.render.make_opts(seed=60 + p, pool=p, split=True,
                                                        batch_paths=(1 + rnd) * 12 * 16 * 32), bufs[p].data_ptr(), streams[p].cuda_stream, None))
        torch.cuda.synchronize()
        for p in range(2):
            assert_same(bufs[p].cpu().numpy(), refs[p], f"round {rnd}, pool {p}")


def test_release_cache_between_split_renders(gpu, oracle):
    """rbrt_gpu_release_cache destroys the lanes; the next split render must create them again."""
    import torch
    scene, cam = S.small_mesh_scene(3), S.example_camera(64, 48)
    ref, ost = oracle_sums(oracle, "mesh3", scene, cam, 4, seed=30, max_depth=0)
    for step in range(2):
        got, st = accum(scene, cam, 4, seed=30, split=True, batch_paths=8 * 12 * 32, no_tail_kernel=True)
        assert_same(got, ref, f"render {step}")
        assert st["iterations"] == 4 * 51 and st["rays"] == ost["rays"]
        torch.cuda.synchronize()
        _abi.check(_abi.lib().rbrt_gpu_release_cache())


# ============================================================================== 5. the collective render with two lanes
@pytest.mark.parametrize("world", [2, 3])
def test_collective_render_on_two_lanes(gpu, comm, release_after, world):
    """Emulated ranks on one device through the PEER transport, each rank's share 2^26 paths: the switch fires inside every rank's
    render_accum and all ranks share device 0's lanes.  Tile shards equal the one-GPU render; sample shards equal the rank-order f32 sum
    of the explicit sample-shard sums, scaled by 1/spp (k_sum_peers, then k_finalize)."""
    W = H = 1024
    spp = 64 * world
    assert W * H * spp // world == T26
    cam = S.example_camera(W, H)
    base = S.spheres_scene()
    _, hdr1, rgb1, st1 = one_lane(base, cam, spp, seed=8)
    want_samples = sample_shard_mean(base, cam, spp, world, seed=8)
    plan_kw = dict(seed=8, max_depth=3, no_tail_kernel=True, batch_paths=1 << 27)
    _, hdr_d1, _, _ = one_lane(base, cam, spp, **plan_kw)
    base.close()
    comm(world)
    scene = S.spheres_scene()                                          # created under the communicator: built once, replicated
    st = {}
    assert_same(R.render_scene_hdr(cam, spp, scene, stats=st, seed=8), hdr1, f"world {world} tile shards")
    assert st["rays"] == st1["rays"] and st["paths"] == st1["paths"]
    assert np.array_equal(R.render_scene(cam, spp, scene, seed=8).pixels, rgb1), f"world {world} tile shards u8"
    st = {}
    assert_same(R.render_scene_hdr(cam, spp, scene, stats=st, **plan_kw), hdr_d1, f"world {world} depth 3")
    assert st["iterations"] == 2 * 4, st                               # every rank: one batch per lane
    assert_same(R.render_scene_hdr(cam, spp, scene, seed=8, shard_mode=_abi.SHARD_SAMPLES), want_samples, f"world {world} sample shards")
    scene.close()
