"""FramePipeline — a SEQUENCE of render_scene calls kept in flight on one GPU.

A frame of the wavefront tracer ends with a sparse phase: the last bounce iterations and the tail kernel are bounded
by the latency of their longest path (C3: ~2.7 ms of a 36 ms frame on one GPU, ~1.7 ms of the 6.4 ms a rank spends on
its eighth of the frame), during which most of the GPU idles; and a rank's share of a frame on 8 GPUs is small enough
that its launches run well below the dense rate.  The reference renders one image per process, so nothing can hide
that there; a host that renders a sequence of images (an animation, a camera sweep, progressive refinement) can:

* `depth` frames (groups) in flight: each is enqueued on its own stream with its own pool of wavefront state
  (RBRT_OPT_POOL_*), so the dense first bounces of the next one fill the SMs the previous one's tail leaves empty;
* `frames_per_batch` frames of the same scene rendered TOGETHER in the same wavefront batches
  (rbrt_gpu_render_accum_device_frames), which gives the kernels of a small shard the size they have on fewer GPUs.

Every frame is computed by the same kernels on the same inputs as a lone render_scene call — each path keeps its own
(pixel, sample, frame) identity — so images stay bit-identical (tests).

    pipe = FramePipeline(width, height, depth=2, frames_per_batch=1)
    for cam, scene in frames:
        for image, tag in pipe.submit(cam, spp, scene, tag=...):     # frames that finished meanwhile, in order
            ...
    rest = pipe.drain()

Scene updates: a frame renders the scene as it was when the frame was SUBMITTED.  The library orders every update after the
frames already enqueued against the scene, but a group that is still being collected (frames_per_batch > 1) has not been
enqueued yet; so Scene.update_mesh / update_mesh_device / update_elements first launch the pending group of every live pipeline
that holds frames of that scene.  The frames that left a pipeline on that occasion are returned by its next submit / flush / drain.

Multi-GPU: under a library communicator (rbrt_gpu_init_multi, or rbrt_b200.dist.init_comm() for one process per GPU) every
rank calls submit() in the same order; a group is ONE call of rbrt_gpu_render_frames_device — shard render, per-GPU
finalise, gather on rank 0, all enqueued on the group's stream — and rank 0 gets the images.
"""
import ctypes as C
import weakref

from . import _abi
from .render import ImageBuffer, make_opts

_live = weakref.WeakSet()      # every FramePipeline, for launch_pending


def launch_pending(handle):
    """Launch the pending group of every pipeline that holds frames of the scene with this library handle (before an update)."""
    hv = handle.value if hasattr(handle, "value") else handle
    for p in list(_live):
        if p._pending and p._pending_hv == hv:
            p._early = [*p._early, *p._launch()]


class _Slot:
    def __init__(self, torch, n_px, fpb, host_output, hdr):
        self.stream = torch.cuda.Stream()
        self.out = torch.empty((fpb, n_px * 3), dtype=torch.float32 if hdr else torch.uint8, device="cuda")
        self.host = torch.empty((fpb, n_px * 3), dtype=self.out.dtype, pin_memory=True) if host_output else None
        self.done = torch.cuda.Event()
        self.busy = False
        self.keep = None       # the scene (and anything else) that must outlive the group in flight
        self.tags = []


class FramePipeline:
    _early = ()                  # frames that left the pipeline while an update launched the pending group (launch_pending)

    def __init__(self, width, height, depth=2, host_output=True, hdr=False, shard_mode=_abi.SHARD_TILES, frames_per_batch=1):
        import torch
        if depth not in (1, 2, 3, 4):
            raise ValueError("depth must be 1..4 (the library keeps four pools of wavefront state per device)")
        if not 1 <= frames_per_batch <= _abi.MAX_FRAMES:
            raise ValueError(f"frames_per_batch must be 1..{_abi.MAX_FRAMES}")
        self._torch = torch
        self.width, self.height, self.depth, self.hdr, self.fpb = int(width), int(height), depth, hdr, int(frames_per_batch)
        self._lib = _abi.lib()
        info = _abi.CommInfoC()
        _abi.check(self._lib.rbrt_gpu_comm_info(info))
        self.world = info.world if info.active else 1
        self.rank = info.rank if info.active else 0
        self.shard_mode = shard_mode
        self._slots = [self._make_slot(host_output and self.rank == 0) for _ in range(depth)]
        self._n = 0                  # groups launched
        self._pending = []           # frames of the group being collected: (cam_c, seed, tag)
        self._pending_key = None     # (scene, spp, opts) the pending frames share
        self._pending_hv = None
        _live.add(self)

    # ------------------------------------------------------------------ internals
    def _make_slot(self, host_output):
        return _Slot(self._torch, self.width * self.height, self.fpb, host_output, self.hdr)

    def _collect(self, slot):
        """Wait for the group in `slot`; returns its frames as [(image, tag)] (rank 0: images; other ranks: None)."""
        slot.done.synchronize()
        slot.busy = False
        tags, slot.tags, slot.keep = slot.tags, [], None
        res = []
        for k, tag in enumerate(tags):
            img = None
            if self.rank == 0:
                if slot.host is not None:
                    arr = slot.host[k].numpy().reshape(self.height, self.width, 3).copy()
                    img = arr if self.hdr else ImageBuffer(arr)
                else:
                    with self._torch.cuda.stream(slot.stream):   # a copy ordered before the slot's next group overwrites it
                        img = slot.out[k].clone()
                    img.record_stream(self._torch.cuda.current_stream())   # the caller reads it on ITS stream: keep the block until then
            res.append((img, tag))
        if self.rank == 0 and slot.host is None and tags:
            slot.stream.synchronize()                          # the copies above (the group itself finished long ago)
        return res

    def _launch(self):
        """Enqueue the pending group on the next slot; returns the frames of the group that slot held before."""
        frames, (scene, spp, opt_items) = self._pending, self._pending_key
        self._pending, self._pending_key = [], None
        slot = self._slots[self._n % self.depth]
        finished = self._collect(slot) if slot.busy else []
        self._enqueue(slot, frames, scene, spp, dict(opt_items))
        slot.busy, slot.keep, slot.tags = True, (scene, [f[0] for f in frames]), [f[2] for f in frames]
        self._n += 1
        return finished

    def _enqueue(self, slot, frames, scene, spp, opts):
        """Enqueue one group of frames (render -> finalise -> [gather on rank 0] -> [copy to pinned host memory]) on the slot's stream."""
        torch = self._torch
        opts.setdefault("shard_mode", self.shard_mode if self.world > 1 else _abi.SHARD_NONE)
        if self.depth == 1:
            opts.setdefault("split", True)                    # one group at a time: let the library overlap the group's own batches (two lanes)
        o = make_opts(pool=self._n % self.depth, **opts)    # shard_count 0 (default): the library shards over its communicator
        handle = scene.handle() if hasattr(scene, "handle") else scene
        nf = len(frames)
        s = slot.stream
        with torch.cuda.stream(s):
            cams = (_abi.CameraC * nf)(*[f[0] for f in frames])
            seeds = (C.c_uint64 * nf)(*[int(f[1]) & 0xFFFFFFFFFFFFFFFF for f in frames])
            outs = (C.c_void_p * nf)(*[slot.out[k].data_ptr() for k in range(nf)])
            rgb, hdr = (None, outs) if self.hdr else (outs, None)
            # stats = NULL: the call only enqueues (no event synchronisation inside the library)
            _abi.check(self._lib.rbrt_gpu_render_frames_device(handle, cams, seeds, nf, int(spp), o, rgb, hdr, s.cuda_stream, None))
            if self.rank == 0 and slot.host is not None:
                slot.host[:nf].copy_(slot.out[:nf], non_blocking=True)
            slot.done.record(s)

    # ------------------------------------------------------------------ API
    def submit(self, cam, num_samples, scene, tag=None, seed=0, **opts):
        """Queue render_scene(cam, num_samples, scene) and return at once.  Returns the list of (image, tag) of the frames
        that left the pipeline meanwhile (possibly empty), in submission order.  `scene` must stay alive (not closed) until
        its frame has been returned; it is held here until then.  Frames are launched in groups of `frames_per_batch`
        that share scene, sample count and options; a frame that differs in one of them starts a new group."""
        cam_c = cam.to_c() if hasattr(cam, "to_c") else cam
        if (int(cam_c.img_width_pix), int(cam_c.img_height_pix)) != (self.width, self.height):
            raise ValueError("camera size differs from the pipeline's")
        h = scene.handle() if hasattr(scene, "handle") else scene
        hv = h.value if hasattr(h, "value") else int(h)       # the same scene = the same library handle
        key = (scene, int(num_samples), tuple(sorted(opts.items())))
        finished, self._early = list(self._early), ()
        if self._pending and (self._pending_hv != hv or self._pending_key[1:] != key[1:]):
            finished += self._launch()
        self._pending_hv = hv
        self._pending.append((cam_c, seed, tag))
        self._pending_key = key
        if len(self._pending) == self.fpb:
            finished += self._launch()
        return finished

    def flush(self):
        """Launch a partially filled group now; returns the frames that left the pipeline meanwhile."""
        early, self._early = list(self._early), ()
        return early + (self._launch() if self._pending else [])

    def drain(self):
        """Launch what is pending and wait for everything in flight; returns the (image, tag) in submission order."""
        out = self.flush()
        for k in range(self.depth):
            slot = self._slots[(self._n + k) % self.depth]
            if slot.busy:
                out += self._collect(slot)
        return out

    def wait_on(self, stream=None):
        """Make `stream` (default: the current stream) wait for everything launched so far — for device-side timing."""
        torch = self._torch
        stream = stream or torch.cuda.current_stream()
        for slot in self._slots:
            if slot.busy:
                stream.wait_event(slot.done)
