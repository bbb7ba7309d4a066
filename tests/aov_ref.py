"""numpy restatement of the first-hit AOV rules (include/rbrt_gpu.h, DESIGN.md section 11): from the closest hits of each sample's camera
rays, in sample order, with float32 accumulators.  Bit-exact against rbrt_gpu_render_aov by construction of the rules."""
import numpy as np

from rbrt_b200 import _abi


def albedo_tables(scene):
    """Per element and per mesh: the albedo a hit contributes ((1,1,1) for Dielectric), as the f32 the library receives."""
    def alb(m):
        c = m.to_c()
        return [1.0, 1.0, 1.0] if c.kind == _abi.MAT_DIELECTRIC else [c.albedo.x, c.albedo.y, c.albedo.z]
    el = np.array([alb(e.material) for e in scene.elements], np.float32).reshape(-1, 3)
    me = np.array([alb(m.material) for m in scene.triangle_meshes], np.float32).reshape(-1, 3)
    return el, me


def compose(hits, el_alb, mesh_alb, shape=None):
    """hits: one HIT_DTYPE array per sample, s = 0 .. S-1 (all of the same length).  Returns the passes as a dict of arrays
    (reshaped to `shape` = (H, W) if given)."""
    S, n = len(hits), len(hits[0])
    f32 = np.float32
    depth, nrm, alb = np.zeros(n, f32), np.zeros((n, 3), f32), np.zeros((n, 3), f32)
    n_hit = np.zeros(n, np.int64)
    for h in hits:
        m = h["kind"] != _abi.HIT_NONE
        nv = h["normal"].astype(f32, copy=True)
        sph = h["kind"] == _abi.HIT_SPHERE
        x, y, z = nv[sph, 0], nv[sph, 1], nv[sph, 2]
        ln = np.sqrt((x * x + y * y) + z * z)                               # len3, f32
        with np.errstate(invalid="ignore", divide="ignore"):
            nv[sph] = nv[sph] / ln[:, None]
        a = np.zeros((n, 3), f32)
        mesh = m & (h["kind"] == _abi.HIT_MESH)
        elem = m & ~mesh
        a[mesh] = mesh_alb[h["elem_idx"][mesh]]
        a[elem] = el_alb[h["elem_idx"][elem]]
        with np.errstate(invalid="ignore", over="ignore"):
            depth[m] = depth[m] + h["dist"][m]
            nrm[m] = nrm[m] + nv[m]
            alb[m] = alb[m] + a[m]
        n_hit += m
    k = n_hit.astype(f32)
    hit = n_hit > 0
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        out = {"depth": np.where(hit, depth / np.where(hit, k, f32(1)), f32(np.inf)).astype(f32),
               "normal": np.where(hit[:, None], nrm / np.where(hit, k, f32(1))[:, None], f32(0)).astype(f32),
               "albedo": np.where(hit[:, None], alb / np.where(hit, k, f32(1))[:, None], f32(0)).astype(f32),
               "coverage": (k / f32(S)).astype(f32)}
    out["hit_kind"] = hits[0]["kind"].astype(np.int32)
    out["elem_idx"] = hits[0]["elem_idx"].astype(np.uint32)
    out["tri_idx"] = hits[0]["tri_idx"].astype(np.uint32)
    if shape is not None:
        out = {key: v.reshape(tuple(shape) + v.shape[1:]) for key, v in out.items()}
    return out


def expected(cam, n_samples, scene, seed=0, oracle=None):
    """The passes composed from the parity hooks: the renderer's primary rays + Scene::hit for every sample (the GPU's hooks, or the
    CPU oracle's primary_rays + OracleScene.hit when `oracle` is given)."""
    import rbrt_b200 as R
    if oracle is None:
        hits = [scene.hit(R.primary_rays(cam, seed, s)) for s in range(n_samples)]
    else:
        osc = oracle.OracleScene.from_scene(scene)
        hits = [osc.hit(oracle.primary_rays(cam.to_c(), seed, s)) for s in range(n_samples)]
    return compose(hits, *albedo_tables(scene), shape=(cam.img_height_pix, cam.img_width_pix))


def mismatches(got, want):
    """Planes that differ bit for bit (uint32 views, so NaN and +-inf compare too): {name: number of differing values}."""
    bad = {}
    for k, w in want.items():
        if k not in got:
            continue
        g = np.ascontiguousarray(got[k])
        w = np.ascontiguousarray(w)
        assert g.shape == w.shape, (k, g.shape, w.shape)
        ne = int((g.view(np.uint32) != w.view(np.uint32)).sum())
        if ne:
            bad[k] = ne
    return bad
