"""Scene — host mirror of rbrt_lib::scene::Scene (scene.rs:12-16): `elements` (spheres and BasicTriangles, any `Intersectable` of the reference that has a GPU twin),
`triangle_meshes`, `lights` (dead in the reference, scene.rs:7-10).  The GPU scene (flattened SoA buffers
+ one LBVH per mesh) is created lazily on first use and owned by this object.

Animation: `update_mesh` / `update_mesh_device` / `update_elements` change the scene in place (rbrt_gpu_scene_update_*): same
triangle counts, same element kinds, no new device block and, by default, each mesh's tree refit rather than rebuilt.  Frames
submitted before an update render the old geometry, frames submitted after it the new one (also through a FramePipeline, whose
pending group is launched first).  The host mirror (`triangle_meshes`, `elements`) follows, so the CPU oracle sees the new scene."""
import ctypes as C

import numpy as np

from . import _abi
from .mesh import TriangleMesh


class _DeviceTriangles(TriangleMesh):
    """Host mirror of vertices handed in on the device (update_mesh_device): a device snapshot, copied to the host when first read."""

    def __init__(self, snapshot, stream, material):
        self._snap, self._stream, self._host = snapshot, stream, None
        self.material = material

    @property
    def triangles(self):
        if self._host is None:
            import torch
            with torch.cuda.stream(self._stream):
                self._host = self._snap.cpu().numpy().reshape(-1, 3, 3)
            self._snap = self._stream = None
        return self._host


def element_arrays(elements):
    """Scene.elements (spheres and BasicTriangles, in order) -> the arrays rbrt_gpu_scene_create_elements takes."""
    from .triangle import BasicTriangle
    sph = [e for e in elements if not isinstance(e, BasicTriangle)]
    tri = [e for e in elements if isinstance(e, BasicTriangle)]
    order, si, ti = [], 0, 0
    for e in elements:
        if isinstance(e, BasicTriangle):
            order.append(_abi.ElementRefC(_abi.ELEM_TRIANGLE, ti)); ti += 1
        else:
            order.append(_abi.ElementRefC(_abi.ELEM_SPHERE, si)); si += 1
    return ((_abi.ElementRefC * max(len(order), 1))(*order), (_abi.SphereDescC * max(len(sph), 1))(*[s.to_c() for s in sph]),
            (_abi.TriangleDescC * max(len(tri), 1))(*[t.to_c() for t in tri]), len(order), len(sph), len(tri))


QUERY_PASSES = ("t", "dist", "kind", "elem_idx", "tri_idx", "point", "normal")
NEAREST_PASSES = ("dist", "kind", "elem_idx", "tri_idx", "point", "normal", "uv")
WINDING_PASSES = ("winding", "inside")


class Scene:
    def __init__(self, elements=None, triangle_meshes=None, lights=None, simd_lanes=8, leaf_size=0, box_pad_rel=0.0, local=False, sah=True, broadcast=False):
        self.elements = list(elements or [])
        self.triangle_meshes = list(triangle_meshes or [])
        self.lights = list(lights or [])
        self.simd_lanes, self.leaf_size, self.box_pad_rel = simd_lanes, leaf_size, box_pad_rel
        self.local, self.sah, self.broadcast = local, sah, broadcast     # RBRT_SCENE_LOCAL / RBRT_SCENE_NO_SAH / RBRT_SCENE_BROADCAST
        self._handle = None

    # ---- GPU handle -----------------------------------------------------------------------
    def handle(self):
        if self._handle is None:
            lib = _abi.lib()
            order, spheres, tris, ne, ns, nt = element_arrays(self.elements)
            nm = len(self.triangle_meshes)
            meshes = (_abi.MeshDescC * max(nm, 1))(*[m.to_c() for m in self.triangle_meshes])
            opts = _abi.SceneOptsC(self.simd_lanes, self.leaf_size, self.box_pad_rel,
                                   (_abi.SCENE_LOCAL if self.local else 0) | (0 if self.sah else _abi.SCENE_NO_SAH)
                                   | (_abi.SCENE_BROADCAST if self.broadcast else 0))
            h = C.c_void_p()
            _abi.check(lib.rbrt_gpu_scene_create_elements(order, ne, spheres, ns, tris, nt, meshes, nm, opts, C.byref(h)))
            self._handle = h
        return self._handle

    def info(self):
        out = _abi.SceneInfoC()
        _abi.check(_abi.lib().rbrt_gpu_scene_info(self.handle(), out))
        return out.as_dict()

    def close(self):
        if self._handle is not None:
            _abi.lib().rbrt_gpu_scene_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- updates in place (rbrt_gpu_scene_update_*) ----------------------------------------------
    def _before_update(self):
        from .pipeline import launch_pending
        launch_pending(self._handle)                                   # frames already submitted keep the old geometry

    def update_mesh(self, i, triangles, material=None, rebuild=False):
        """New world-space vertices [N,3,3] for mesh i (N = its triangle count), optionally a new material; rebuild=True builds the
        mesh's tree afresh instead of refitting it.  Returns once the vertices have been read."""
        tris = np.ascontiguousarray(triangles, dtype=np.float32).reshape(-1, 3, 3)   # (held by the mirror like TriangleMesh holds it)
        i = int(i)
        mat = material if material is not None else (self.triangle_meshes[i].material if 0 <= i < len(self.triangle_meshes) else None)
        if self._handle is not None:
            self._before_update()
            _abi.check(_abi.lib().rbrt_gpu_scene_update_mesh(self._handle, i, tris.ctypes.data, len(tris),
                                                             C.byref(material.to_c()) if material is not None else None,
                                                             _abi.UPDATE_REBUILD if rebuild else _abi.UPDATE_REFIT))
        self.triangle_meshes[i] = TriangleMesh(tris, mat)

    def update_mesh_device(self, i, tensor, material=None, rebuild=False, stream=None):
        """The same from a CUDA float32 tensor [N,3,3] on the scene's device, read in order on `stream` (default: the current stream),
        which then waits for the update: the tensor may be overwritten by work enqueued on that stream afterwards."""
        import torch
        if not (isinstance(tensor, torch.Tensor) and tensor.is_cuda and tensor.dtype == torch.float32):
            raise TypeError("update_mesh_device takes a CUDA float32 tensor of shape [N,3,3]")
        t = tensor.reshape(-1, 3, 3)
        stream = stream or torch.cuda.current_stream()
        i = int(i)
        mat = material if material is not None else (self.triangle_meshes[i].material if 0 <= i < len(self.triangle_meshes) else None)
        with torch.cuda.stream(stream):
            t = t.contiguous()
            snap = t.clone()                                           # the mirror's copy, taken before the caller may overwrite `tensor`
        if self._handle is not None:
            self._before_update()
            _abi.check(_abi.lib().rbrt_gpu_scene_update_mesh_device(self._handle, i, t.data_ptr(), t.shape[0],
                                                                    C.byref(material.to_c()) if material is not None else None,
                                                                    _abi.UPDATE_REBUILD if rebuild else _abi.UPDATE_REFIT,
                                                                    stream.cuda_stream))
        self.triangle_meshes[i] = _DeviceTriangles(snap, stream, mat)

    def update_elements(self, elements):
        """New Scene.elements: the same number, the same kinds (Sphere / BasicTriangle) in the same order; positions, sizes and
        materials may change."""
        elements = list(elements)
        if self._handle is not None:
            self._before_update()
            order, spheres, tris, ne, ns, nt = element_arrays(elements)
            _abi.check(_abi.lib().rbrt_gpu_scene_update_elements(self._handle, order, ne, spheres, ns, tris, nt))
        self.elements = elements

    # ---- motion vectors (rbrt_gpu_scene_snapshot, DESIGN.md section 16) ---------------------------
    def snapshot(self, stream=None):
        """Record the scene's current geometry as "the previous frame" of render_motion*, enqueued on `stream` (a torch.cuda.Stream;
        default: the legacy default stream).  It sees every update made before it; later updates wait for it."""
        _abi.check(_abi.lib().rbrt_gpu_scene_snapshot(self.handle(), stream.cuda_stream if stream is not None else None))

    # ---- Scene::hit (scene.rs:19-43) for caller-supplied rays ----------------------------------
    def hit(self, rays, trace_mode=_abi.TRACE_BVH, stats=None):
        """rays: [N,6] f32 (origin xyz, direction xyz). Returns a structured array (HIT_DTYPE)."""
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
        hits = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
        st = _abi.StatsC()
        _abi.check(_abi.lib().rbrt_gpu_trace_rays(self.handle(), rays.ctypes.data, len(rays), trace_mode,
                                                  hits.ctypes.data, st))
        if stats is not None:
            stats.update(st.as_dict())
        return hits

    # ---- ray queries on device memory (rbrt_gpu_query_*_device, DESIGN.md section 12) ---------------
    def _query_rays(self, rays, stream):
        import torch
        if not (isinstance(rays, torch.Tensor) and rays.is_cuda and rays.dtype == torch.float32 and rays.dim() == 2 and rays.shape[1] == 6
                and rays.is_contiguous()):
            raise ValueError("rays must be a contiguous float32 CUDA tensor of shape [N,6] (origin xyz, direction xyz)")
        stream = stream or torch.cuda.current_stream(rays.device)
        if stream.device != rays.device:
            raise ValueError(f"rays are on {rays.device}, the stream on {stream.device}")
        return stream

    @staticmethod
    def _query_check(rc, stats, st):
        if rc == _abi.E_INVALID:                                       # a refused argument (rays or outputs on another device, ...)
            raise ValueError(_abi.lib().rbrt_last_error().decode("utf-8", "replace"))
        _abi.check(rc)
        if stats is not None:
            stats.update(st.as_dict())

    def intersect_device(self, rays, passes=None, stream=None, stats=None):
        """Scene::hit for the rays of a CUDA tensor [N,6] on the scene's device: a dict of CUDA tensors t, dist, kind (RBRT_HIT_*),
        elem_idx, tri_idx [N] and point, normal [N,3], each bit for bit the field `hit` reports (`passes`: a subset of those names).
        Enqueued on `stream` (default: the rays' current stream); returns without synchronising unless `stats` (a dict) is given."""
        import torch
        stream = self._query_rays(rays, stream)
        names = QUERY_PASSES if passes is None else ((passes,) if isinstance(passes, str) else tuple(dict.fromkeys(passes)))
        unknown = [p for p in names if p not in QUERY_PASSES]
        if unknown or not names:
            raise ValueError(f"unknown or no pass(es) {unknown}; choose from {QUERY_PASSES}")
        n = rays.shape[0]
        handle = self.handle()
        out, tensors = _abi.QueryOutC(), {}
        with torch.cuda.stream(stream):
            for name in names:
                dt = torch.int32 if name == "kind" else (torch.uint32 if name in ("elem_idx", "tri_idx") else torch.float32)
                tensors[name] = torch.empty((n, 3) if name in ("point", "normal") else (n,), dtype=dt, device=rays.device)
                setattr(out, name, tensors[name].data_ptr())
        st = _abi.StatsC()
        rc = _abi.lib().rbrt_gpu_query_closest_device(handle, rays.data_ptr(), n, out, stream.cuda_stream, st if stats is not None else None)
        self._query_check(rc, stats, st)
        return tensors

    def occluded_device(self, rays, max_dist=None, stream=None, stats=None):
        """Occlusion for the rays of a CUDA tensor [N,6]: a uint8 CUDA tensor [N], 1 where `hit` reports a hit with dist < max_dist
        (strict; max_dist a float32 CUDA tensor [N], None = +inf), 2 for a NaN ray, 0 otherwise.  Enqueued like intersect_device."""
        import torch
        stream = self._query_rays(rays, stream)
        n = rays.shape[0]
        if max_dist is not None and not (isinstance(max_dist, torch.Tensor) and max_dist.device == rays.device and max_dist.dtype == torch.float32
                                         and tuple(max_dist.shape) == (n,) and max_dist.is_contiguous()):
            raise ValueError("max_dist must be None or a contiguous float32 CUDA tensor [N] on the rays' device")
        handle = self.handle()
        with torch.cuda.stream(stream):
            occ = torch.empty(n, dtype=torch.uint8, device=rays.device)
        st = _abi.StatsC()
        rc = _abi.lib().rbrt_gpu_query_occluded_device(handle, rays.data_ptr(), n, max_dist.data_ptr() if max_dist is not None else None,
                                                         occ.data_ptr(), stream.cuda_stream, st if stats is not None else None)
        self._query_check(rc, stats, st)
        return occ

    # ---- nearest-surface queries on device memory (rbrt_gpu_query_nearest_device, DESIGN.md section 17) ----------
    def nearest_device(self, points, max_dist=None, passes=None, stream=None, stats=None):
        """The nearest surface of the scene to each point of a contiguous float32 CUDA tensor [N,3] on the scene's device: a dict of CUDA
        tensors dist, kind (RBRT_HIT_*), elem_idx, tri_idx [N], point, normal [N,3] and uv [N,2] (`passes`: a subset of those names).
        max_dist: None (+inf) or a float32 CUDA tensor [N]; only surfaces closer than it (strict) count, and a point without one gets
        kind RBRT_HIT_NONE and dist +inf.  Enqueued on `stream` (default: the points' current stream); returns without synchronising
        unless `stats` (a dict) is given."""
        import torch
        points, stream = self._device_points(points, stream)
        n = points.shape[0]
        if max_dist is not None and not (isinstance(max_dist, torch.Tensor) and max_dist.device == points.device
                                         and max_dist.dtype == torch.float32 and tuple(max_dist.shape) == (n,) and max_dist.is_contiguous()):
            raise ValueError("max_dist must be None or a contiguous float32 CUDA tensor [N] on the points' device")
        names = NEAREST_PASSES if passes is None else ((passes,) if isinstance(passes, str) else tuple(dict.fromkeys(passes)))
        unknown = [p for p in names if p not in NEAREST_PASSES]
        if unknown or not names:
            raise ValueError(f"unknown or no pass(es) {unknown}; choose from {NEAREST_PASSES}")
        handle = self.handle()
        out, tensors = _abi.NearestOutC(), {}
        with torch.cuda.stream(stream):
            for name in names:
                dt = torch.int32 if name == "kind" else (torch.uint32 if name in ("elem_idx", "tri_idx") else torch.float32)
                shape = (n, 3) if name in ("point", "normal") else ((n, 2) if name == "uv" else (n,))
                tensors[name] = torch.empty(shape, dtype=dt, device=points.device)
                setattr(out, name, tensors[name].data_ptr())
        st = _abi.StatsC()
        rc = _abi.lib().rbrt_gpu_query_nearest_device(handle, points.data_ptr(), n, max_dist.data_ptr() if max_dist is not None else None,
                                                       out, stream.cuda_stream, st if stats is not None else None)
        self._query_check(rc, stats, st)
        return tensors

    @staticmethod
    def _device_points(points, stream):
        """(points, stream) of a query on points: a contiguous float32 CUDA tensor [N,3], and the stream (default: its current one)."""
        import torch
        if not (isinstance(points, torch.Tensor) and points.is_cuda and points.dtype == torch.float32 and points.dim() == 2
                and points.shape[1] == 3 and points.is_contiguous()):
            raise ValueError("points must be a contiguous float32 CUDA tensor of shape [N,3]")
        stream = stream or torch.cuda.current_stream(points.device)
        if stream.device != points.device:
            raise ValueError(f"points are on {points.device}, the stream on {stream.device}")
        return points, stream

    # ---- inside tests on device memory (rbrt_gpu_query_winding_device, DESIGN.md section 18) ---------------------------
    def winding_device(self, points, beta=None, passes=None, stream=None, stats=None):
        """The generalized winding number of the scene at each point of a contiguous float32 CUDA tensor [N,3] on the scene's device: a
        dict of CUDA tensors winding (float32 [N]) and inside (uint8 [N], |winding| > 0.5); `passes`: a subset of those names.  beta: None
        (the default 2.0), > 1, or float('inf') for the exact sum over every triangle.  Enqueued on `stream` (default: the points'
        current stream); returns without synchronising unless `stats` (a dict) is given."""
        import torch
        points, stream = self._device_points(points, stream)
        n = points.shape[0]
        names = WINDING_PASSES if passes is None else ((passes,) if isinstance(passes, str) else tuple(dict.fromkeys(passes)))
        unknown = [p for p in names if p not in WINDING_PASSES]
        if unknown or not names:
            raise ValueError(f"unknown or no pass(es) {unknown}; choose from {WINDING_PASSES}")
        handle = self.handle()
        out, tensors = _abi.WindingOutC(), {}
        with torch.cuda.stream(stream):
            for name in names:
                tensors[name] = torch.empty(n, dtype=torch.float32 if name == "winding" else torch.uint8, device=points.device)
                setattr(out, name, tensors[name].data_ptr())
        st = _abi.StatsC()
        rc = _abi.lib().rbrt_gpu_query_winding_device(handle, points.data_ptr(), n, _abi.WindingOptsC(0.0 if beta is None else float(beta)),
                                                       out, stream.cuda_stream, st if stats is not None else None)
        self._query_check(rc, stats, st)
        return tensors

    def signed_distance_device(self, points, max_dist=None, beta=None, stream=None):
        """The signed distance to the scene at each point (float32 CUDA tensor [N]): nearest_device's `dist`, negated where
        winding_device's `inside` is set; both calls run on one stream.  max_dist (None, a float, or a float32 CUDA tensor [N]) bounds
        the nearest search: a point with no surface closer than it gets +inf outside and -inf inside, which narrow-band SDF sampling
        can take as "beyond the band, on this side"."""
        import torch
        points, stream = self._device_points(points, stream)
        if max_dist is not None and not isinstance(max_dist, torch.Tensor):
            with torch.cuda.stream(stream):
                max_dist = torch.full((points.shape[0],), float(max_dist), dtype=torch.float32, device=points.device)
        dist = self.nearest_device(points, max_dist=max_dist, passes="dist", stream=stream)["dist"]
        inside = self.winding_device(points, beta=beta, passes="inside", stream=stream)["inside"]
        with torch.cuda.stream(stream):
            return torch.where(inside.bool(), -dist, dist)


def scatter(items, seed=0):
    """Parity hook for RayScattering::scatter (materials.rs:4-12).  items: iterable of (material, in_ray_direction(3),
    hit_point(3), hit_normal(3), pixel, sample, bounce); returns (scattered [N] i32, attenuation [N,3], out_dir [N,3])."""
    items = list(items)
    n = len(items)
    arr = (_abi.ScatterInC * max(n, 1))()
    for k, (mat, d, p, nrm, pixel, sample, bounce) in enumerate(items):
        a = arr[k]
        a.material = mat.to_c()
        a.in_ray.origin = _abi.Vec3C(0.0, 0.0, 0.0)
        a.in_ray.direction = _abi.Vec3C(*[float(x) for x in d])
        a.hit_point = _abi.Vec3C(*[float(x) for x in p])
        a.hit_normal = _abi.Vec3C(*[float(x) for x in nrm])
        a.pixel, a.sample, a.bounce = int(pixel), int(sample), int(bounce)
    out = (_abi.ScatterOutC * max(n, 1))()
    _abi.check(_abi.lib().rbrt_gpu_scatter(C.cast(arr, C.c_void_p), n, int(seed) & 0xFFFFFFFFFFFFFFFF, C.cast(out, C.c_void_p)))
    sc = np.array([out[k].scattered for k in range(n)], np.int32)
    att = np.array([[out[k].attenuation.x, out[k].attenuation.y, out[k].attenuation.z] for k in range(n)], np.float32).reshape(n, 3)
    od = np.array([[out[k].out_ray.direction.x, out[k].out_ray.direction.y, out[k].out_ray.direction.z] for k in range(n)], np.float32).reshape(n, 3)
    return sc, att, od
