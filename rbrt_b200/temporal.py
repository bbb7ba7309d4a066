"""TemporalAccumulator — temporal accumulation of a frame sequence on the GPU (rbrt_gpu_temporal_accumulate_device, DESIGN.md section 15).

Each step folds one frame (colour, its variance, and the first-hit AOVs of the same camera and seed) into the history of the frames
before it: the history is reprojected through the previous camera and kept where depth, normal and sample 0's hit ids agree.  The
accumulator owns two sets of output tensors and uses them in turn (the library refuses to accumulate in place), and keeps the previous
camera and guides.

    acc = TemporalAccumulator(width, height)
    for cam, seed in frames:
        hdr, var = render_hdr_variance_device(cam, spp, scene, splits=4, seed=seed)
        aovs = render_aovs_device(cam, aov_spp, scene, seed=seed, passes=("depth", "normal", "ids"))
        hdr_t, var_t, length = acc.step(cam, hdr, var, aovs)      # valid until the step after next
                                                                  # (motion=render_motion_device(cam, acc.camera, scene): per-object motion)
        out, _ = denoise_variance_device(hdr_t, var_t, {**aovs, **albedo}, ...)

The returned tensors are the accumulator's own: they are overwritten two steps later, so clone what must outlive that.
"""
from . import render


class TemporalAccumulator:
    def __init__(self, width, height, alpha_min=0.1, sigma_depth=0.02, normal_min=0.9, stream=None):
        self.width, self.height = int(width), int(height)
        self.opts = dict(alpha_min=alpha_min, sigma_depth=sigma_depth, normal_min=normal_min)
        self.stream = stream
        self._sets = [None, None]          # the two sets of (hdr, var, length) tensors, allocated on first use
        self._next = 0
        self._history = None

    def reset(self):
        """Forget the history: the next step is a first frame."""
        self._history = None

    def _outputs(self, torch, with_var, device):
        s = self._sets[self._next]
        if s is None or (s[1] is None) == with_var or s[0].device != device:
            H, W = self.height, self.width
            s = (torch.empty((H, W, 3), dtype=torch.float32, device=device),
                 torch.empty((H, W, 3), dtype=torch.float32, device=device) if with_var else None,
                 torch.empty((H, W), dtype=torch.float32, device=device))
            self._sets[self._next] = s
        self._next ^= 1
        return s

    @property
    def camera(self):
        """The history's camera (None before the first step or after reset): the prev_cam of the next frame's render_motion*."""
        return self._history["cam"] if self._history is not None else None

    def step(self, cam, hdr, var, aovs, motion=None):
        """Fold the frame at camera `cam` (hdr, var [H,W,3] CUDA tensors, var may be None; aovs with depth, normal, hit_kind and
        elem_idx) into the history.  motion: None, or (motion, prev_dist) of render_motion_device for cam against the history's camera
        and the snapshot taken at the history's frame; the history is then reprojected along each pixel's motion where it is finite.
        Returns (hdr, var or None, length) tensors, enqueued on the accumulator's stream (default: the current stream)."""
        import torch
        if (cam.img_width_pix, cam.img_height_pix) != (self.width, self.height):
            raise ValueError(f"the camera's image is {cam.img_width_pix} x {cam.img_height_pix}, the accumulator's {self.width} x {self.height}")
        stream = self.stream or torch.cuda.current_stream()
        if self._history is not None and (var is None) != (self._history["var"] is None):
            self._history = None                                            # a change between with and without variance restarts
        with torch.cuda.stream(stream):
            outs = self._outputs(torch, var is not None, stream.device)
        out = render._temporal(cam, hdr, var, aovs, self._history, **self.opts, device=True, outs=outs, stream=stream, motion=motion)
        guides = {k: aovs[k] for k in ("depth", "normal", "hit_kind", "elem_idx")}
        self._history = {"cam": cam, "hdr": out[0], "var": out[1], "length": out[2], "aovs": guides}
        return out
