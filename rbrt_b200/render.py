"""render_scene — host mirror of rbrt_lib::render_scene (lib.rs:75-124) over the C-ABI.

`render_scene(cam, num_samples, scene)` is the call a user of rbrt makes (main.rs:82); it returns an
ImageBuffer (RGB8, row-major, `.save(path)`), like `image::ImageBuffer<Rgb<u8>, Vec<u8>>`.
All buffers that cross this call are HOST buffers; device copies happen inside the library.
"""
import os
import struct

import numpy as np

from . import _abi
from .png import encode_png


class ImageBuffer:
    """Row-major RGB8 image = image::ImageBuffer<Rgb<u8>, Vec<u8>> (lib.rs:116-123)."""

    def __init__(self, pixels):
        self.pixels = np.ascontiguousarray(pixels, dtype=np.uint8)

    @property
    def height(self):
        return self.pixels.shape[0]

    @property
    def width(self):
        return self.pixels.shape[1]

    def get_pixel(self, x, y):
        return tuple(int(v) for v in self.pixels[y, x])

    def save(self, path):  # main.rs:86: format chosen by extension
        ext = os.path.splitext(path)[1].lower()
        if ext == ".png":
            data = encode_png(self.pixels)
        elif ext in (".ppm", ".pnm"):
            data = b"P6\n%d %d\n255\n" % (self.width, self.height) + self.pixels.tobytes()
        elif ext == ".bmp":                                  # 24-bit BI_RGB: bottom-up rows of BGR, padded to 4 bytes (as rbrt_cli.cpp)
            w, h = self.width, self.height
            stride = (3 * w + 3) & ~3
            rows = np.zeros((h, stride), np.uint8)
            rows[:, :3 * w] = self.pixels[::-1, :, ::-1].reshape(h, 3 * w)
            hdr = struct.pack("<2sIII", b"BM", 54 + stride * h, 0, 54) + struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, 0, stride * h, 2835, 2835, 0, 0)
            data = hdr + rows.tobytes()
        elif ext == ".tga":                                  # uncompressed true-colour, top-left origin, BGR
            if self.width > 65535 or self.height > 65535:
                raise ValueError(f"Unable to save target img to {path}! image too large for TGA")
            data = struct.pack("<BBBHHBHHHHBB", 0, 0, 2, 0, 0, 0, 0, 0, self.width, self.height, 24, 0x20) + np.ascontiguousarray(self.pixels[:, :, ::-1]).tobytes()
        elif ext in (".tif", ".tiff"):                       # baseline TIFF: little-endian, one uncompressed RGB strip
            data = encode_tiff(self.pixels)
        elif ext == ".qoi":
            data = encode_qoi(self.pixels)
        else:
            raise ValueError(f"Unable to save target img to {path}! unsupported extension {ext!r}")
        with open(path, "wb") as f:
            f.write(data)


def encode_tiff(pixels):
    """Baseline TIFF 6.0 (as rbrt_cli.cpp writes it): header, the pixel strip, then the IFD with the ten required RGB tags."""
    h, w = pixels.shape[:2]
    n = 3 * w * h
    ifd_at = 8 + n + (n & 1)
    bits_at = ifd_at + 2 + 10 * 12 + 4
    tags = [(256, 4, 1, w), (257, 4, 1, h), (258, 3, 3, bits_at), (259, 3, 1, 1), (262, 3, 1, 2), (273, 4, 1, 8), (277, 3, 1, 3),
            (278, 4, 1, h), (279, 4, 1, n), (284, 3, 1, 1)]
    ifd = struct.pack("<H", len(tags)) + b"".join(struct.pack("<HHII", t, ty, c, v) for t, ty, c, v in tags) + struct.pack("<I", 0)
    return struct.pack("<2sHI", b"II", 42, ifd_at) + pixels.tobytes() + b"\0" * (n & 1) + ifd + struct.pack("<HHH", 8, 8, 8)


def encode_qoi(pixels):
    """QOI (qoiformat.org), 3 channels: the ops in the encoder's usual order run / index / diff / luma / rgb (as rbrt_cli.cpp)."""
    h, w = pixels.shape[:2]
    out = bytearray(struct.pack(">4sIIBB", b"qoif", w, h, 3, 0))
    index = [None] * 64                                      # (slots start as RGBA 0,0,0,0: they never equal a pixel, whose alpha is 255)
    pr, pg, pb = 0, 0, 0
    run = 0
    flat = pixels.reshape(-1, 3).tolist()
    last = len(flat) - 1
    for i, (r, g, b) in enumerate(flat):
        if (r, g, b) == (pr, pg, pb):
            run += 1
            if run == 62 or i == last:
                out.append(0xC0 | (run - 1)); run = 0
            continue
        if run:
            out.append(0xC0 | (run - 1)); run = 0
        k = (r * 3 + g * 5 + b * 7 + 255 * 11) % 64
        if index[k] == (r, g, b):
            out.append(k)
        else:
            index[k] = (r, g, b)
            dr, dg, db = ((r - pr + 128) & 255) - 128, ((g - pg + 128) & 255) - 128, ((b - pb + 128) & 255) - 128
            if -2 <= dr <= 1 and -2 <= dg <= 1 and -2 <= db <= 1:
                out.append(0x40 | (dr + 2) << 4 | (dg + 2) << 2 | (db + 2))
            elif -32 <= dg <= 31 and -8 <= dr - dg <= 7 and -8 <= db - dg <= 7:
                out += bytes((0x80 | (dg + 32), (dr - dg + 8) << 4 | (db - dg + 8)))
            else:
                out += bytes((0xFE, r, g, b))
        pr, pg, pb = r, g, b
    return bytes(out) + b"\0" * 7 + b"\1"


def make_opts(seed=0, max_depth=0, trace_mode=_abi.TRACE_BVH, shard_mode=_abi.SHARD_NONE, shard_rank=0, shard_count=0,
              batch_paths=0, integrator=0, count_visits=False, time_kernels=False, no_tail_kernel=False, pool=0, split=False):
    return _abi.RenderOptsC(int(seed) & 0xFFFFFFFFFFFFFFFF, max_depth, trace_mode, shard_mode, shard_rank, shard_count,
                            batch_paths, integrator,
                            (_abi.OPT_COUNT_VISITS if count_visits else 0) | (_abi.OPT_TIME_KERNELS if time_kernels else 0)
                            | (_abi.OPT_NO_TAIL_KERNEL if no_tail_kernel else 0) | ((int(pool) & 3) << _abi.OPT_POOL_SHIFT)
                            | (_abi.OPT_SPLIT_BATCHES if split else 0))


def render_scene(cam, num_samples, scene, stats=None, **opts):
    """= rbrt_lib::render_scene(cam, num_samples, scene) (lib.rs:75-79)."""
    print("Starting rendering...")  # lib.rs:80
    W, H = cam.img_width_pix, cam.img_height_pix
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render(scene.handle(), cam.to_c(), int(num_samples), make_opts(**opts),
                                          rgb.ctypes.data, st))
    print("\rRendering 100% complete!")  # lib.rs:114
    if stats is not None:
        stats.update(st.as_dict())
    return ImageBuffer(rgb)


def render_scene_hdr(cam, num_samples, scene, stats=None, **opts):
    """The pre-gamma mean colour `color * (1.0 / num_samples)` (lib.rs:101) as [H,W,3] f32."""
    W, H = cam.img_width_pix, cam.img_height_pix
    hdr = np.empty((H, W, 3), dtype=np.float32)
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_hdr(scene.handle(), cam.to_c(), int(num_samples), make_opts(**opts),
                                              hdr.ctypes.data, st))
    if stats is not None:
        stats.update(st.as_dict())
    return hdr


def primary_rays(cam, seed=0, sample_idx=0):
    """The renderer's own primary rays (cam.rs:64-82 with the Philox stream of one sample): [H*W,6] f32."""
    rays = np.empty((cam.img_width_pix * cam.img_height_pix, 6), dtype=np.float32)
    _abi.check(_abi.lib().rbrt_gpu_primary_rays(cam.to_c(), int(seed), int(sample_idx), rays.ctypes.data))
    return rays


# ---- first-hit AOVs (rbrt_gpu_render_aov*, include/rbrt_gpu.h and DESIGN.md section 11) ----------------------------------
AOV_PASSES = ("depth", "normal", "albedo", "coverage", "ids")
# pass -> [(plane, numpy dtype, components)]; "ids" is sample 0's hit_kind / elem_idx / tri_idx
_AOV_PLANES = {"depth": [("depth", np.float32, 1)], "normal": [("normal", np.float32, 3)], "albedo": [("albedo", np.float32, 3)],
               "coverage": [("coverage", np.float32, 1)],
               "ids": [("hit_kind", np.int32, 1), ("elem_idx", np.uint32, 1), ("tri_idx", np.uint32, 1)]}


def _aov_planes(passes):
    if isinstance(passes, str):
        passes = (passes,)
    unknown = [p for p in passes if p not in _AOV_PLANES]
    if unknown:
        raise ValueError(f"unknown AOV pass(es) {unknown}; choose from {AOV_PASSES}")
    return [pl for p in dict.fromkeys(passes) for pl in _AOV_PLANES[p]]


def render_aovs(cam, num_samples, scene, seed=0, passes=AOV_PASSES, stats=None):
    """First-hit AOVs of the render's own camera rays: a dict of numpy arrays, [H,W] for depth / coverage / hit_kind / elem_idx /
    tri_idx and [H,W,3] for normal / albedo ("ids" gives the last three).  Blocks until they are on the host."""
    W, H = cam.img_width_pix, cam.img_height_pix
    out, arrays = _abi.AovOutC(), {}
    for name, dt, k in _aov_planes(passes):
        arrays[name] = np.empty((H, W, k) if k > 1 else (H, W), dtype=dt)
        setattr(out, name, arrays[name].ctypes.data)
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_aov(scene.handle(), cam.to_c(), int(num_samples), int(seed) & 0xFFFFFFFFFFFFFFFF, out, st))
    if stats is not None:
        stats.update(st.as_dict())
    return arrays


def render_aovs_device(cam, num_samples, scene, seed=0, passes=AOV_PASSES, stream=None):
    """The same as CUDA tensors on the scene's first device, enqueued on `stream` (default: the current stream); returns without
    synchronising."""
    import torch
    stream = stream or torch.cuda.current_stream()
    W, H = cam.img_width_pix, cam.img_height_pix
    tdt = {np.float32: torch.float32, np.int32: torch.int32, np.uint32: torch.uint32}
    out, tensors = _abi.AovOutC(), {}
    handle = scene.handle()
    with torch.cuda.stream(stream):
        for name, dt, k in _aov_planes(passes):
            tensors[name] = torch.empty((H, W, k) if k > 1 else (H, W), dtype=tdt[dt], device=stream.device)
            setattr(out, name, tensors[name].data_ptr())
    _abi.check(_abi.lib().rbrt_gpu_render_aov_device(handle, cam.to_c(), int(num_samples), int(seed) & 0xFFFFFFFFFFFFFFFF, out,
                                                     stream.cuda_stream, None))
    return tensors


# ---- guided denoising (rbrt_gpu_denoise*, include/rbrt_gpu.h and DESIGN.md section 13) --------------------------------------
def _denoise_inputs(hdr, aovs, is_tensor):
    """(H, W) of the colour [H,W,3] and the guides depth [H,W], normal and albedo [H,W,3]: contiguous float32 (CUDA tensors for the device
    variant, numpy arrays otherwise), or ValueError."""
    planes = {"hdr": hdr}
    for k in ("depth", "normal", "albedo"):
        if k not in aovs:
            raise ValueError(f"the guides need the {k!r} AOV (render_aovs with passes including it)")
        planes[k] = aovs[k]
    if getattr(hdr, "ndim", 0) != 3 or hdr.shape[2] != 3:
        raise ValueError("hdr must be [H, W, 3]")
    H, W = hdr.shape[:2]
    for k, v in planes.items():
        want = (H, W) if k == "depth" else (H, W, 3)
        if is_tensor(v) is not True or tuple(v.shape) != want:
            raise ValueError(f"{k} must be a contiguous float32 {'CUDA tensor' if is_tensor is _is_cuda_f32 else 'numpy array'} of shape {want}")
    return H, W


def _is_numpy_f32(v):
    return isinstance(v, np.ndarray) and v.dtype == np.float32 and v.flags.c_contiguous


def _is_cuda_f32(v):
    import torch
    return isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float32 and v.is_contiguous()


def _denoise_opts(levels, sigma_depth, sigma_luminance):
    return _abi.DenoiseOptsC(int(levels), float(sigma_depth), float(sigma_luminance))


def _denoise(hdr, var, aovs, levels, sigma_depth, sigma_luminance, device, stats=None, stream=None):
    """denoise (var None) and denoise_variance, on numpy arrays or, with device=True, on CUDA tensors enqueued on `stream`."""
    is_tensor = _is_cuda_f32 if device else _is_numpy_f32
    H, W = _denoise_inputs(hdr, aovs, is_tensor)
    if var is not None:
        _variance_input(var, hdr, is_tensor)
    if device:
        import torch
        stream = stream or torch.cuda.current_stream()
        with torch.cuda.stream(stream):
            out = torch.empty((H, W, 3), dtype=torch.float32, device=stream.device)
            rgb = torch.empty((H, W, 3), dtype=torch.uint8, device=stream.device)
        ptr, tail = (lambda a: a.data_ptr()), (stream.cuda_stream, None)
    else:
        out = np.empty((H, W, 3), dtype=np.float32)
        rgb = np.empty((H, W, 3), dtype=np.uint8)
        st = _abi.StatsC()
        ptr, tail = (lambda a: a.ctypes.data), (st,)
    lib = _abi.lib()
    if var is None:
        call, planes = (lib.rbrt_gpu_denoise_device if device else lib.rbrt_gpu_denoise), (ptr(hdr),)
    else:
        call, planes = (lib.rbrt_gpu_denoise_variance_device if device else lib.rbrt_gpu_denoise_variance), (ptr(hdr), ptr(var))
    g = _abi.AovOutC(depth=ptr(aovs["depth"]), normal=ptr(aovs["normal"]), albedo=ptr(aovs["albedo"]))
    _abi.check(call(W, H, *planes, g, _denoise_opts(levels, sigma_depth, sigma_luminance), ptr(out), ptr(rgb), *tail))
    if device:
        return out, rgb
    if stats is not None:
        stats.update(st.as_dict())
    return out, ImageBuffer(rgb)


def denoise(hdr, aovs, levels=0, sigma_depth=0.0, sigma_luminance=0.0, stats=None):
    """Denoise a render_scene_hdr image [H,W,3] guided by render_aovs planes of the same camera and seed (depth, normal, albedo; guides
    with at most the image's samples line up with it pixel for pixel).  Returns (hdr_out [H,W,3] float32, ImageBuffer of its tonemap).
    levels / sigmas: 0 = the defaults (4 levels).  Blocks until the result is on the host."""
    return _denoise(hdr, None, aovs, levels, sigma_depth, sigma_luminance, False, stats=stats)


def denoise_device(hdr, aovs, levels=0, sigma_depth=0.0, sigma_luminance=0.0, stream=None):
    """The same on CUDA tensors (render_aovs_device's planes) of the current render device: returns (hdr_out [H,W,3] float32,
    rgb [H,W,3] uint8) tensors, enqueued on `stream` (default: the current stream) without synchronising."""
    return _denoise(hdr, None, aovs, levels, sigma_depth, sigma_luminance, True, stream=stream)


# ---- per-pixel variance and variance-guided denoising (rbrt_gpu_render_hdr_variance*, rbrt_gpu_denoise_variance*; DESIGN.md section 14)
def render_scene_hdr_variance(cam, num_samples, scene, splits=4, stats=None, **opts):
    """The pre-gamma mean colour [H,W,3] f32 of num_samples samples, rendered as `splits` sample-range shards (2..16, dividing
    num_samples), and the unbiased variance of that mean per pixel and channel [H,W,3] f32, from the spread of the shards' means.
    Returns (hdr, var); blocks until both are on the host."""
    W, H = cam.img_width_pix, cam.img_height_pix
    hdr = np.empty((H, W, 3), dtype=np.float32)
    var = np.empty((H, W, 3), dtype=np.float32)
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_hdr_variance(scene.handle(), cam.to_c(), int(num_samples), int(splits), make_opts(**opts),
                                                       hdr.ctypes.data, var.ctypes.data, st))
    if stats is not None:
        stats.update(st.as_dict())
    return hdr, var


def render_hdr_variance_device(cam, num_samples, scene, splits=4, stream=None, **opts):
    """The same as CUDA tensors on the scene's first device, enqueued on `stream` (default: the current stream) without synchronising."""
    import torch
    stream = stream or torch.cuda.current_stream()
    W, H = cam.img_width_pix, cam.img_height_pix
    handle = scene.handle()
    with torch.cuda.stream(stream):
        hdr = torch.empty((H, W, 3), dtype=torch.float32, device=stream.device)
        var = torch.empty((H, W, 3), dtype=torch.float32, device=stream.device)
    _abi.check(_abi.lib().rbrt_gpu_render_hdr_variance_device(handle, cam.to_c(), int(num_samples), int(splits), make_opts(**opts),
                                                              hdr.data_ptr(), var.data_ptr(), stream.cuda_stream, None))
    return hdr, var


def _variance_input(var, hdr, is_tensor):
    if is_tensor(var) is not True or tuple(var.shape) != tuple(hdr.shape):
        raise ValueError(f"var must be a contiguous float32 {'CUDA tensor' if is_tensor is _is_cuda_f32 else 'numpy array'} of the shape of hdr")


def denoise_variance(hdr, var, aovs, levels=0, sigma_depth=0.0, sigma_luminance=0.0, stats=None):
    """Denoise a render_scene_hdr_variance frame [H,W,3] with its variance [H,W,3], guided by render_aovs planes of the same camera and
    seed (depth, normal, albedo).  Returns (hdr_out [H,W,3] float32, ImageBuffer of its tonemap).  levels / sigmas: 0 = this filter's
    defaults (5 levels).  Blocks until the result is on the host."""
    return _denoise(hdr, var, aovs, levels, sigma_depth, sigma_luminance, False, stats=stats)


def denoise_variance_device(hdr, var, aovs, levels=0, sigma_depth=0.0, sigma_luminance=0.0, stream=None):
    """The same on CUDA tensors of the current render device: returns (hdr_out [H,W,3] float32, rgb [H,W,3] uint8) tensors, enqueued on
    `stream` (default: the current stream) without synchronising."""
    return _denoise(hdr, var, aovs, levels, sigma_depth, sigma_luminance, True, stream=stream)


# ---- temporal accumulation (rbrt_gpu_temporal_accumulate*; include/rbrt_gpu.h and DESIGN.md section 15) ----------------------------
_TEMPORAL_GUIDES = (("depth", 1, "float32"), ("normal", 3, "float32"), ("hit_kind", 1, "int32"), ("elem_idx", 1, "uint32"))


def _temporal_plane(what, v, H, W, k, dtype, device):
    shape = (H, W, k) if k > 1 else (H, W)
    if device:
        import torch
        ok = isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == getattr(torch, dtype) and v.is_contiguous()
    else:
        ok = isinstance(v, np.ndarray) and v.dtype == np.dtype(dtype) and v.flags.c_contiguous
    if not ok or tuple(v.shape) != shape:
        raise ValueError(f"{what} must be a contiguous {dtype} {'CUDA tensor' if device else 'numpy array'} of shape {shape}")
    return v.data_ptr() if device else v.ctypes.data


def _temporal(cam, hdr, var, aovs, history, alpha_min, sigma_depth, normal_min, device, outs, stream=None, stats=None, motion=None):
    """temporal_accumulate (numpy) and, with device=True, temporal_accumulate_device; outs = (hdr_out, var_out, len_out) or None.
    motion: None, or (motion [H,W,2], prev_dist [H,W]) of render_motion*: the _motion variants."""
    W, H = cam.img_width_pix, cam.img_height_pix
    if var is not None and history is not None and history.get("var") is None:
        raise ValueError("with var, the history needs the var it returned")
    ptr = lambda what, v, k=3, dt="float32": _temporal_plane(what, v, H, W, k, dt, device)
    planes = [ptr("hdr", hdr), ptr("var", var) if var is not None else None]

    def guides(what, g):
        missing = [k for k, *_ in _TEMPORAL_GUIDES if k not in g]
        if missing:
            raise ValueError(f"the {what} need the AOVs {missing} (render_aovs with passes depth, normal and ids)")
        return _abi.AovOutC(**{k: ptr(f"{what}[{k!r}]", g[k], n, dt) for k, n, dt in _TEMPORAL_GUIDES})

    g = guides("guides", aovs)
    h = None
    if history is not None:
        h = _abi.TemporalHistoryC(cam=history["cam"].to_c(), hdr=ptr("history hdr", history["hdr"]),
                                  var=ptr("history var", history["var"]) if var is not None else None,
                                  length=ptr("history length", history["length"], 1), guides=guides("history guides", history["aovs"]))
    opts = _abi.TemporalOptsC(float(alpha_min), float(sigma_depth), float(normal_min))
    if outs is None:
        if device:
            import torch
            with torch.cuda.stream(stream):
                outs = (torch.empty((H, W, 3), dtype=torch.float32, device=stream.device),
                        torch.empty((H, W, 3), dtype=torch.float32, device=stream.device) if var is not None else None,
                        torch.empty((H, W), dtype=torch.float32, device=stream.device))
        else:
            outs = (np.empty((H, W, 3), np.float32), np.empty((H, W, 3), np.float32) if var is not None else None, np.empty((H, W), np.float32))
    optr = [ptr("hdr_out", outs[0]), ptr("var_out", outs[1]) if outs[1] is not None else None, ptr("len_out", outs[2], 1)]
    lib = _abi.lib()
    mo = None if motion is None else _abi.MotionOutC(ptr("motion", motion[0], 2), ptr("prev_dist", motion[1], 1))
    if device:
        if mo is None:
            _abi.check(lib.rbrt_gpu_temporal_accumulate_device(W, H, cam.to_c(), *planes, g, h, opts, *optr, stream.cuda_stream, None))
        else:
            _abi.check(lib.rbrt_gpu_temporal_accumulate_motion_device(W, H, cam.to_c(), *planes, g, h, mo, opts, *optr, stream.cuda_stream,
                                                                      None))
    else:
        st = _abi.StatsC()
        if mo is None:
            _abi.check(lib.rbrt_gpu_temporal_accumulate(W, H, cam.to_c(), *planes, g, h, opts, *optr, st))
        else:
            _abi.check(lib.rbrt_gpu_temporal_accumulate_motion(W, H, cam.to_c(), *planes, g, h, mo, opts, *optr, st))
        if stats is not None:
            stats.update(st.as_dict())
    return outs


def temporal_accumulate(cam, hdr, aovs, var=None, history=None, alpha_min=0.1, sigma_depth=0.02, normal_min=0.9, stats=None, motion=None):
    """Fold the frame hdr [H,W,3] (with its variance var [H,W,3], optional) rendered at camera `cam` into a history: each pixel's
    history is reprojected through the previous camera and blended with the frame where depth, normal and sample 0's hit ids agree.
    aovs: render_aovs planes of the same camera and seed with depth, normal, hit_kind and elem_idx.  history: None for the first frame,
    else a dict with the previous call's results and inputs: cam, hdr, var (with var), length and aovs.  Returns (hdr_out, var_out or
    None, length [H,W]) numpy float32 arrays; blocks until they are on the host.  motion: (motion, prev_dist) of render_motion for cam
    against the history's camera and the snapshot taken at the history's frame: each pixel is reprojected along its motion where
    that is finite (moving objects keep their history), through the cameras otherwise."""
    return _temporal(cam, hdr, var, aovs, history, alpha_min, sigma_depth, normal_min, False, None, stats=stats, motion=motion)


def temporal_accumulate_device(cam, hdr, aovs, var=None, history=None, alpha_min=0.1, sigma_depth=0.02, normal_min=0.9, stream=None,
                               motion=None):
    """The same on CUDA tensors of the current render device (render_aovs_device's planes; motion: render_motion_device's): returns
    (hdr_out, var_out or None, length) tensors, enqueued on `stream` (default: the current stream) without synchronising."""
    import torch
    stream = stream or torch.cuda.current_stream()
    return _temporal(cam, hdr, var, aovs, history, alpha_min, sigma_depth, normal_min, True, None, stream=stream, motion=motion)


# ---- per-object motion vectors (rbrt_gpu_render_motion*; include/rbrt_gpu.h and DESIGN.md section 16) -------------------------------
def render_motion(cam, prev_cam, scene, stats=None):
    """Per pixel of cam's image, the screen motion [H,W,2] f32 from the pixel-centre ray's hit in cam to where that surface point was
    in prev_cam at the scene's latest snapshot (Scene.snapshot), and the distance [H,W] f32 from prev_cam's position to that previous
    point; (NaN, NaN) and +inf for a miss.  Returns (motion, prev_dist); blocks until they are on the host."""
    W, H = cam.img_width_pix, cam.img_height_pix
    motion = np.empty((H, W, 2), dtype=np.float32)
    prev_dist = np.empty((H, W), dtype=np.float32)
    st = _abi.StatsC()
    _abi.check(_abi.lib().rbrt_gpu_render_motion(scene.handle(), cam.to_c(), prev_cam.to_c(), _abi.MotionOutC(motion.ctypes.data, prev_dist.ctypes.data),
                                                 st))
    if stats is not None:
        stats.update(st.as_dict())
    return motion, prev_dist


def render_motion_device(cam, prev_cam, scene, stream=None):
    """The same as CUDA tensors on the scene's first device, enqueued on `stream` (default: the current stream) without synchronising."""
    import torch
    stream = stream or torch.cuda.current_stream()
    W, H = cam.img_width_pix, cam.img_height_pix
    handle = scene.handle()
    with torch.cuda.stream(stream):
        motion = torch.empty((H, W, 2), dtype=torch.float32, device=stream.device)
        prev_dist = torch.empty((H, W), dtype=torch.float32, device=stream.device)
    _abi.check(_abi.lib().rbrt_gpu_render_motion_device(handle, cam.to_c(), prev_cam.to_c(),
                                                        _abi.MotionOutC(motion.data_ptr(), prev_dist.data_ptr()), stream.cuda_stream, None))
    return motion, prev_dist
