// harness.cpp — TEST INFRASTRUCTURE (tests/test_device_source_on_host.py): the product's device headers compiled for the host.
//
// rbrt_b200/csrc/{common,intersect,shade}.cuh hold the per-ray arithmetic of the hot path — Scene::hit with its sphere,
// BasicTriangle, bounding-box and Moeller-Trumbore tests, camera rays, the three scatter()s, Philox, sky, `as u8`.  Here those
// headers are compiled by g++ (-ffp-contract=off, the cuda_runtime.h stand-in of this directory) and driven by the plainest
// possible loop: one ray at a time, brute force over the triangles (`scene_hit<true>`, the kernel `rbrt_gpu_trace_rays` runs
// in RBRT_TRACE_BRUTE mode) or the one-lane BVH traversal (`scene_hit<false>`, RBRT_TRACE_BVH mode) over a tree built here,
// recursion of lib.rs:43-73 unrolled into a loop.  The tests compare the result bit for bit with
// the oracle and the golden fixtures, so a slip in one of those headers shows up in the CPU-only test run of every round and
// not only on the GPU box.  What this does NOT cover: the device compiler (nvcc / ptxas — `__fmul_rn` and friends on the
// device against plain `*` under -ffp-contract=off here), the GPU's LBVH build, the warp-voted traversal and the wavefront machinery of render.cu.
// Those are the GPU tests' business.  This is not a fallback: nothing under rbrt_b200/ can reach it.
//
// The scene is flattened here the way api.cu / bvh_build.cu (k_emit_tris) lay it out for the kernels: element records,
// {v0, e1, e2} + original index per tested triangle (N_eff of the lane rule), unit normals, exact AABB over all triangles.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "intersect.cuh"
#include "cull.cuh"
#include "shade.cuh"
#include "../../include/rbrt_gpu.h"

using namespace rbrt;

float hd_rcp_error = 0.0f;
unsigned hd_rcp_calls = 0;

namespace {

struct HostScene {
    std::vector<uint4> nodes;                                  // 4 x uint4 per 4-wide node, all meshes (MeshDev::node_base)
    std::vector<float4> spheres, etris, tris, normals, mat;
    std::vector<uint32_t> elem_kind, mat_kind;
    std::vector<MeshDev> meshes;
    SceneDev dev;
};

uint64_t tested_triangles(uint64_t n, uint32_t lanes) {            // mesh.rs:136-144 + triangle.rs:167,296 (as api.cu)
    uint64_t r = n % lanes, total = n + r, tested = (total / lanes) * lanes;
    return tested < n ? tested : n;
}

// ---- a 4-wide BVH in the node format of intersect.cuh, built on the host -----------------------------------------------------
// The product builds its tree on the GPU (bvh_build.cu: Morton LBVH -> refit + rotations -> 4-wide collapse), which cannot run
// here.  What CAN be checked without a GPU is the product's TRAVERSAL source (ray_slabs, the PRMT decode, bvh4_step, leaf_step,
// the prune bounds, scene_hit<false>'s t_limit) — on any valid tree in that format.  This builder makes one: median splits of
// the centroid range, two binary levels folded into one node (largest box first, like collapse_node), boxes = triangle AABBs +
// the pad, quantised onto the mesh's 16-bit grid OUTWARD plus one step, by the formulas of bvh_build.cu (k_mesh_setup, quant_lo /
// quant_hi).  It shares no code with the GPU builder; a traversal that agrees with the brute-force loop on it for every ray has
// its own arithmetic right.
struct Box { float lo[3], hi[3]; };
inline void grow(Box& b, const Box& o) { for (int k = 0; k < 3; ++k) { b.lo[k] = fminf(b.lo[k], o.lo[k]); b.hi[k] = fmaxf(b.hi[k], o.hi[k]); } }
inline Box empty_box() { Box b; for (int k = 0; k < 3; ++k) { b.lo[k] = INFINITY; b.hi[k] = -INFINITY; } return b; }
inline float half_area(const Box& b) { float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2]; return dx * dy + dy * dz + dz * dx; }
inline uint32_t quant_lo(float v, float org, float step) {
    float q = floorf((v - org) / step) - 1.0f;
    while (q > 0.0f && fmaf(q, step, org) > v) q -= 1.0f;
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}
inline uint32_t quant_hi(float v, float org, float step) {
    float q = ceilf((v - org) / step) + 1.0f;
    while (q < 65535.0f && fmaf(q, step, org) < v) q += 1.0f;
    return (uint32_t)fminf(fmaxf(q, 0.0f), 65535.0f);
}

// rbrt_scene_opts.box_pad_rel as api.cu resolves it (default 2e-5); HD_BOX_PAD_REL overrides it for experiments
inline float pad_rel() { const char* e = getenv("HD_BOX_PAD_REL"); return e ? (float)atof(e) : 2e-5f; }

struct TreeBuilder {
    const std::vector<Box>& tb;                                // per triangle (already padded), in the order `order` lists them
    std::vector<uint32_t>& order;
    uint32_t leaf_size;
    const float* step;                                         // the grid step of k_mesh_setup's BuildParams (md.qstep may be NaN)
    const MeshDev& md;
    std::vector<uint4>& out; size_t base;                      // nodes of this mesh start at out[4 * base]
    struct Part { uint32_t a, b; Box box; };                   // triangles order[a..b)
    Part part(uint32_t a, uint32_t b) const { Part p{a, b, empty_box()}; for (uint32_t i = a; i < b; ++i) grow(p.box, tb[order[i]]); return p; }
    void split(const Part& p, Part& l, Part& r) {
        Box cb = empty_box();
        for (uint32_t i = p.a; i < p.b; ++i) { const Box& t = tb[order[i]]; Box c; for (int k = 0; k < 3; ++k) c.lo[k] = c.hi[k] = 0.5f * (t.lo[k] + t.hi[k]); grow(cb, c); }
        int ax = 0; for (int k = 1; k < 3; ++k) if (cb.hi[k] - cb.lo[k] > cb.hi[ax] - cb.lo[ax]) ax = k;
        const uint32_t mid = p.a + (p.b - p.a) / 2;
        std::nth_element(order.begin() + p.a, order.begin() + mid, order.begin() + p.b,
                         [&](uint32_t x, uint32_t y) { return tb[x].lo[ax] + tb[x].hi[ax] < tb[y].lo[ax] + tb[y].hi[ax]; });
        l = part(p.a, mid); r = part(mid, p.b);
    }
    // writes the node of `p` (more than leaf_size triangles) into slot `slot`
    void node(const Part& p, uint32_t slot) {
        std::vector<Part> kids(2);
        split(p, kids[0], kids[1]);
        for (int round = 0; round < 2; ++round) {
            int best = -1; float best_a = -1.0f;
            for (size_t k = 0; k < kids.size(); ++k) if (kids[k].b - kids[k].a > leaf_size && half_area(kids[k].box) > best_a) { best_a = half_area(kids[k].box); best = (int)k; }
            if (best < 0) break;
            Part l, r; split(kids[best], l, r);
            kids[best] = l; kids.push_back(r);
        }
        uint32_t q[4][3]; int32_t refs[4];
        for (size_t k = 0; k < 4; ++k) {
            if (k < kids.size()) {
                for (int c = 0; c < 3; ++c) q[k][c] = quant_lo(kids[k].box.lo[c], md.qorg[c], step[c]) | (quant_hi(kids[k].box.hi[c], md.qorg[c], step[c]) << 16);
                if (kids[k].b - kids[k].a > leaf_size) { const uint32_t child = (uint32_t)(out.size() / 4 - base); out.resize(out.size() + 4); refs[k] = (int32_t)child; node(kids[k], child); }
                else refs[k] = make_leaf_ref(kids[k].a, kids[k].b - kids[k].a);
            } else { q[k][0] = q[k][1] = q[k][2] = 0x0000FFFFu; refs[k] = make_leaf_ref(0, 1); }      // unused slot: inverted box
        }
        uint4* o = out.data() + 4 * (base + slot);
        o[0] = make_uint4(q[0][0], q[0][1], q[0][2], q[1][0]); o[1] = make_uint4(q[1][1], q[1][2], q[2][0], q[2][1]);
        o[2] = make_uint4(q[2][2], q[3][0], q[3][1], q[3][2]); o[3] = make_uint4((uint32_t)refs[0], (uint32_t)refs[1], (uint32_t)refs[2], (uint32_t)refs[3]);
    }
};

void flatten(HostScene& hs, const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, const rbrt_triangle_desc* btris,
             const rbrt_mesh_desc* meshes, uint32_t nm, uint32_t lanes, uint32_t leaf_size = 0) {   // leaf_size > 0: also build the trees
    hs.spheres.resize(ne); hs.elem_kind.resize(ne); hs.mat.resize(ne + nm); hs.mat_kind.resize(ne + nm);
    uint32_t n_et = 0;
    for (uint32_t i = 0; i < ne; ++i) {
        rbrt_material m;
        if (order[i].kind == RBRT_ELEM_SPHERE) {
            const rbrt_sphere_desc& s = spheres[order[i].index];
            hs.spheres[i] = make_float4(s.center.x, s.center.y, s.center.z, s.radius);
            hs.elem_kind[i] = RBRT_ELEM_SPHERE; m = s.material;
        } else {                                                    // BasicTriangle::new (triangle.rs:19-27)
            const rbrt_triangle_desc& t = btris[order[i].index];
            f3 a = mk3(t.corners[0].x, t.corners[0].y, t.corners[0].z), b = mk3(t.corners[1].x, t.corners[1].y, t.corners[1].z), c = mk3(t.corners[2].x, t.corners[2].y, t.corners[2].z);
            f3 e1 = b - a, e2 = c - a, n = norm3(cross3(e1, e2));
            uint32_t ti = (uint32_t)(hs.etris.size() / 4);
            hs.spheres[i] = make_float4(__uint_as_float(ti), 0.0f, 0.0f, 0.0f);
            hs.etris.push_back(make_float4(a.x, a.y, a.z, 0.0f)); hs.etris.push_back(make_float4(e1.x, e1.y, e1.z, 0.0f));
            hs.etris.push_back(make_float4(e2.x, e2.y, e2.z, 0.0f)); hs.etris.push_back(make_float4(n.x, n.y, n.z, 0.0f));
            hs.elem_kind[i] = RBRT_ELEM_TRIANGLE; m = t.material; ++n_et;
        }
        hs.mat[i] = make_float4(m.albedo.x, m.albedo.y, m.albedo.z, m.param); hs.mat_kind[i] = m.kind;
    }
    hs.meshes.resize(nm);
    for (uint32_t mi = 0; mi < nm; ++mi) {
        const rbrt_mesh_desc& m = meshes[mi];
        hs.mat[ne + mi] = make_float4(m.material.albedo.x, m.material.albedo.y, m.material.albedo.z, m.material.param); hs.mat_kind[ne + mi] = m.material.kind;
        MeshDev md; memset(&md, 0, sizeof(md));
        const uint64_t n_eff = tested_triangles(m.num_triangles, lanes);
        md.tri_base = (uint32_t)(hs.tris.size() / 3); md.n_tris = (uint32_t)n_eff; md.nrm_base = (uint32_t)hs.normals.size(); md.elem = ne + mi;
        for (int k = 0; k < 3; ++k) { md.lo[k] = 3.40282347e+38f; md.hi[k] = -3.40282347e+38f; }        // k_aabb_init: an axis with no number keeps them
        for (uint64_t t = 0; t < m.num_triangles; ++t) {
            const float* v = m.tri_vertices + 9 * t;
            for (int c = 0; c < 3; ++c) for (int k = 0; k < 3; ++k) { md.lo[k] = fminf(md.lo[k], v[3 * c + k]); md.hi[k] = fmaxf(md.hi[k], v[3 * c + k]); }   // aabbox.rs:62-88
        }
        std::vector<uint32_t> order(n_eff);
        for (uint32_t t = 0; t < n_eff; ++t) order[t] = t;
        md.node_base = (uint32_t)(hs.nodes.size() / 4); md.root_ref = make_leaf_ref(0, 1);
        if (leaf_size && n_eff) {                                    // grid as k_mesh_setup lays it, then the tree; triangles go out in tree order
            float mx = 0.0f, grid_step[3];
            for (int k = 0; k < 3; ++k) { mx = fmaxf(mx, fmaxf(fabsf(md.lo[k]), fabsf(md.hi[k]))); mx = fmaxf(mx, md.hi[k] - md.lo[k]); }
            const float pad = pad_rel() > 0.0f ? fmaxf(pad_rel() * mx, (getenv("HD_NO_PAD_FLOOR") ? 0.0f : (getenv("HD_PAD_FLOOR") ? (float)atof(getenv("HD_PAD_FLOOR")) : 4.7683716e-7f) * (mx + 1000.0f))) : 0.0f;   // k_mesh_setup
            for (int k = 0; k < 3; ++k) {
                float ext = (md.hi[k] + pad) - (md.lo[k] - pad), step = ext / 65500.0f;
                if (!(step > 1e-30f)) step = 1e-30f;
                md.qorg[k] = (md.lo[k] - pad) - 8.0f * step;
                grid_step[k] = step;                                                                                  // the nodes are quantised on this grid...
                md.qstep[k] = step <= RBRT_QSTEP_MAX ? step : NAN;                                                    // ...the traversal reads NaN where it would overflow
            }
            std::vector<Box> tb(n_eff);
            for (uint32_t t = 0; t < n_eff; ++t) {
                const float* v = m.tri_vertices + 9 * (size_t)t;
                Box b;
                for (int k = 0; k < 3; ++k) {                                                                         // k_emit_tris' padded box
                    b.lo[k] = fminf(v[k], fminf(v[3 + k], v[6 + k])) - pad; b.hi[k] = fmaxf(v[k], fmaxf(v[3 + k], v[6 + k])) + pad;
                }
                tb[t] = b;
            }
            TreeBuilder B{tb, order, leaf_size, grid_step, md, hs.nodes, md.node_base};
            if (n_eff <= leaf_size) md.root_ref = make_leaf_ref(0, (uint32_t)n_eff);
            else { hs.nodes.resize(hs.nodes.size() + 4); md.root_ref = 0; B.node(B.part(0, (uint32_t)n_eff), 0); }
        }
        hs.normals.resize(md.nrm_base + n_eff);
        for (uint32_t pos = 0; pos < n_eff; ++pos) {
            const uint32_t t = order[pos];
            const float* v = m.tri_vertices + 9 * (size_t)t;
            f3 v0 = mk3(v[0], v[1], v[2]), e1 = mk3(v[3], v[4], v[5]) - v0, e2 = mk3(v[6], v[7], v[8]) - v0;        // mesh.rs:57-60
            f3 n = norm3(cross3(e1, e2));                                                                             // triangle.rs:30-34
            hs.tris.push_back(make_float4(v0.x, v0.y, v0.z, __uint_as_float(t)));                                       // BVH order, original index alongside
            hs.tris.push_back(make_float4(e1.x, e1.y, e1.z, 0.0f)); hs.tris.push_back(make_float4(e2.x, e2.y, e2.z, 0.0f));
            hs.normals[md.nrm_base + t] = make_float4(n.x, n.y, n.z, 0.0f);                                             // original order
        }
        hs.meshes[mi] = md;
    }
    SceneDev& d = hs.dev;
    d.spheres = hs.spheres.data(); d.etris = hs.etris.data(); d.elem_kind = hs.elem_kind.data(); d.tris = hs.tris.data();
    d.nodes = reinterpret_cast<const float4*>(hs.nodes.data());
    d.normals = hs.normals.data(); d.mat = hs.mat.data(); d.mat_kind = hs.mat_kind.data(); d.meshes = hs.meshes.data();
    d.n_spheres = ne; d.n_meshes = nm; d.n_etris = n_et;
}

f3 hit_normal(const SceneDev& S, const Hit& h, f3 p) {
    if (h.kind == 0) return element_normal(S, h.elem, p);                                        // sphere: p - c (sphere.rs:56); BasicTriangle: its normal
    float4 nn = S.normals[S.meshes[h.elem].nrm_base + h.tri];                                     // mesh.rs:253-257
    return mk3(nn.x, nn.y, nn.z);
}

// Scene::hit with the traversal the trace kernels run (traverse_voted: one node visit or ONE triangle test per step, leaf_step_one +
// the branch-free tri_intersect_masks), for a "warp" of one lane.  The frame around it — spheres first, then per mesh the box test,
// the limit from the best hit so far, closing the mesh — restates what k_trace does per ray (render.cu, start_mesh / the loop head).
Hit scene_hit_voted(const SceneDev& S, f3 o, f3 d, TraceCounters* cnt) {
    Hit best; best.kind = -1; best.elem = 0; best.tri = 0; best.t = 0.0f; best.dist = 0.0f;
    float closest = 3.40282347e+38f;
    for (uint32_t i = 0; i < S.n_spheres; ++i) {
        float t, dist;
        int r = element_intersect(S, i, o, d, t, dist);
        if (r < 0) { best.kind = -2; return best; }
        if (r && dist < closest) { closest = dist; best.kind = 0; best.elem = i; best.t = t; best.dist = dist; }
    }
    for (uint32_t mi = 0; mi < S.n_meshes; ++mi) {
        const MeshDev& M = S.meshes[mi];
        if (M.n_tris == 0 || !mesh_bbox_hit(M, o, d)) continue;
        float t_limit = RBRT_T_CAP;
        if (closest < 3.0e38f) {
            float dl = len3(d), omax = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z));
            float lim = (closest * 1.001f + 1e-5f * (omax + closest) + 1e-6f) / dl;
            if (lim == lim) t_limit = fminf(t_limit, lim);
        }
        float t_prune = t_limit, best_t = 1000000.0f; uint32_t best_idx = 0xFFFFFFFFu;
        const uint4* nodes = reinterpret_cast<const uint4*>(S.nodes) + 4 * (size_t)M.node_base;
        const RaySlabs R = ray_slabs(M, o, d);
        int32_t lstack[RBRT_STACK]; const StackL stack = {lstack};
        int sp = 0; stack.put(sp++, RBRT_SENTINEL);
        int32_t cur = M.root_ref;
        uint32_t n_nodes = 0, n_tris = 0;
        traverse_voted<true, false>(nodes, S.tris, M.tri_base, R, o, d, t_limit, stack, sp, cur, best_t, best_idx, t_prune, 1, n_nodes, n_tris);
        if (cnt) { cnt->nodes += n_nodes; cnt->tris += n_tris; }
        if (best_idx == 0xFFFFFFFFu) continue;
        f3 p = o + best_t * d;
        float dist = len3(o - p);
        if (dist > RBRT_MIN_DIST && dist < RBRT_MAX_DIST && dist < closest) { closest = dist; best.kind = 1; best.elem = mi; best.tri = best_idx; best.t = best_t; best.dist = dist; }
    }
    return best;
}

}  // namespace

extern "C" {

void hd_set_rcp_error(float e) { hd_rcp_error = e; hd_rcp_calls = 0; }

// Scene::hit for caller-supplied rays, records filled as k_trace_rays (render.cu) fills them
int hd_trace_rays(const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, const rbrt_triangle_desc* btris, const rbrt_mesh_desc* meshes,
                  uint32_t nm, uint32_t lanes, uint32_t leaf_size /* 0: brute force; 1..8: through a 4-wide BVH with such leaves; + 16: the voted traversal */,
                  const rbrt_ray* rays, uint64_t n, rbrt_hit* hits, uint64_t* node_visits, uint64_t* tri_tests) {
    const bool voted = (leaf_size & 16u) != 0; leaf_size &= 15u;
    HostScene hs; flatten(hs, order, ne, spheres, btris, meshes, nm, lanes, leaf_size);
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    uint64_t nodes_total = 0, tris_total = 0;
    for (uint64_t i = 0; i < n; ++i) {
        f3 o = mk3(rays[i].origin.x, rays[i].origin.y, rays[i].origin.z), d = mk3(rays[i].direction.x, rays[i].direction.y, rays[i].direction.z);
        Hit h = !leaf_size ? scene_hit<true>(hs.dev, o, d, &cnt) : (voted ? scene_hit_voted(hs.dev, o, d, &cnt) : scene_hit<false>(hs.dev, o, d, &cnt));
        nodes_total += cnt.nodes; tris_total += cnt.tris; cnt.nodes = 0; cnt.tris = 0;
        rbrt_hit out; memset(&out, 0, sizeof(out));
        out.kind = h.kind >= 0 ? h.kind : RBRT_HIT_NONE;
        if (h.kind >= 0) {
            f3 p = o + h.t * d, nrm = hit_normal(hs.dev, h, p);
            if (h.kind == 0 && hs.dev.n_etris && hs.elem_kind[h.elem]) out.kind = RBRT_HIT_TRIANGLE;
            out.elem_idx = h.elem; out.tri_idx = h.tri; out.t = h.t; out.dist = h.dist;
            out.point = rbrt_vec3{p.x, p.y, p.z}; out.normal = rbrt_vec3{nrm.x, nrm.y, nrm.z};
        }
        hits[i] = out;
    }
    if (node_visits) *node_visits = nodes_total;
    if (tri_tests) *tri_tests = tris_total;
    return 0;
}

// render_scene (lib.rs:75-124) with the product's device functions: hdr_out H x W x 3 (pre-gamma mean), rgb_out H x W x 3
int hd_render(const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, const rbrt_triangle_desc* btris, const rbrt_mesh_desc* meshes,
              uint32_t nm, uint32_t lanes, uint32_t leaf_size /* as hd_trace_rays: 0 brute force, 1..8 BVH, + 16 voted */, const rbrt_camera* cam, uint32_t spp,
              uint64_t seed, uint32_t max_depth, float* hdr_out, uint8_t* rgb_out, uint64_t* rays_out, uint64_t* nan_out) {
    const bool voted = (leaf_size & 16u) != 0; leaf_size &= 15u;
    HostScene hs; flatten(hs, order, ne, spheres, btris, meshes, nm, lanes, leaf_size);
    const SceneDev& S = hs.dev;
    CamDev c;
    const rbrt_vec3* src[4] = {&cam->position, &cam->right, &cam->up, &cam->img_center_point};
    float* dst[4] = {c.pos, c.right, c.up, c.center};
    for (int k = 0; k < 4; ++k) { dst[k][0] = src[k]->x; dst[k][1] = src[k]->y; dst[k][2] = src[k]->z; }
    c.mm_per_pix_hor = cam->mm_per_pix_hor; c.mm_per_pix_vert = cam->mm_per_pix_vert; c.width = cam->img_width_pix; c.height = cam->img_height_pix;
    RngKey key; key.k0 = (uint32_t)seed; key.k1 = (uint32_t)(seed >> 32);
    if (!max_depth) max_depth = 50;                                                               // lib.rs:99
    uint64_t rays = 0, nans = 0;
    std::vector<uint32_t> hist(max_depth + 1);
    const float inv_spp = XDIV(1.0f, (float)spp);                                                 // lib.rs:101: multiply by the reciprocal
    for (uint32_t row = 0; row < c.height; ++row)
        for (uint32_t col = 0; col < c.width; ++col) {
            const uint32_t pixel = row * c.width + col;
            f3 acc = mk3(0.0f, 0.0f, 0.0f);
            for (uint32_t s = 0; s < spp; ++s) {
                f3 o, d;
                camera_ray(c, row, col, key, pixel, s, o, d);
                f3 color = mk3(0.0f, 0.0f, 0.0f);
                for (uint32_t it = 0;; ++it) {                                                     // `it` scatters lie behind this ray
                    ++rays;
                    Hit h = !leaf_size ? scene_hit<true>(S, o, d, nullptr) : (voted ? scene_hit_voted(S, o, d, nullptr) : scene_hit<false>(S, o, d, nullptr));
                    if (h.kind == -2) { ++nans; break; }                                          // the reference panics (sphere.rs:33); the product ends the path black
                    if (h.kind < 0) {                                                             // miss: sky, then att_1 * (att_2 * (... * sky)) (lib.rs:62-71)
                        color = sky(d);
                        for (int k = (int)it - 1; k >= 0; --k) {
                            float4 m = S.mat[hist[k]];
                            color = (S.mat_kind[hist[k]] == 2u ? mk3(1.0f, 1.0f, 1.0f) : mk3(m.x, m.y, m.z)) * color;
                        }
                        break;
                    }
                    if (it >= max_depth) break;                                                   // depth == 0: black, scatter() not called (lib.rs:54-55)
                    f3 p = o + h.t * d, nrm = hit_normal(S, h, p), out_d;
                    const uint32_t elem = h.kind == 0 ? h.elem : S.meshes[h.elem].elem;
                    if (!scatter(S.mat_kind[elem], S.mat[elem], d, p, nrm, key, pixel, s, it + 1, out_d)) break;   // absorbed (metal.rs:24)
                    hist[it] = elem; o = p; d = out_d;
                }
                acc = acc + color;                                                                // lib.rs:96-100, samples in order
            }
            f3 mean = acc * inv_spp;
            float* hp = hdr_out + 3 * (size_t)pixel; hp[0] = mean.x; hp[1] = mean.y; hp[2] = mean.z;
            uint8_t* rp = rgb_out + 3 * (size_t)pixel;                                            // lib.rs:118-120
            rp[0] = as_u8(XMUL(XSQRT(mean.x), 256.0f)); rp[1] = as_u8(XMUL(XSQRT(mean.y), 256.0f)); rp[2] = as_u8(XMUL(XSQRT(mean.z), 256.0f));
        }
    if (rays_out) *rays_out = rays;
    if (nan_out) *nan_out = nans;
    return 0;
}

// scatter() in isolation, as rbrt_gpu_scatter / k_scatter_kat call it (bounce index and Philox key given by the caller)
int hd_scatter(const rbrt_scatter_in* in, uint64_t n, uint64_t seed, rbrt_scatter_out* out) {
    RngKey key; key.k0 = (uint32_t)seed; key.k1 = (uint32_t)(seed >> 32);
    for (uint64_t i = 0; i < n; ++i) {
        const rbrt_scatter_in& q = in[i];
        f3 od;
        const bool ok = scatter(q.material.kind, make_float4(q.material.albedo.x, q.material.albedo.y, q.material.albedo.z, q.material.param),
                                mk3(q.in_ray.direction.x, q.in_ray.direction.y, q.in_ray.direction.z), mk3(q.hit_point.x, q.hit_point.y, q.hit_point.z),
                                mk3(q.hit_normal.x, q.hit_normal.y, q.hit_normal.z), key, q.pixel, q.sample, q.bounce, od);
        memset(&out[i], 0, sizeof(out[i]));
        out[i].scattered = ok ? 1 : 0;
        const bool glass = q.material.kind == 2u;                                                 // attenuation: albedo, or (1,1,1) for dielectrics (dielectric.rs:19)
        out[i].attenuation = glass ? rbrt_vec3{1.0f, 1.0f, 1.0f} : q.material.albedo;
        out[i].out_ray.origin = q.hit_point; out[i].out_ray.direction = rbrt_vec3{od.x, od.y, od.z};
    }
    return 0;
}

// The camera-ray culling of stage A (cull.cuh) against the exact tests it stands in front of.  For sphere s and its m directions
// (normalised here the way camera_ray normalises): skipped = outside_double_cone, hit = sphere_intersect != 0 (a NaN counts as "must be tested").
// axis_scale / w_shift perturb the cone record the way the device's approximate rsqrtf may.  out = {pairs, skipped, skipped AND hit, hit}.
int hd_cull_spheres(const float* origin, const float* spheres, uint32_t n, const float* dirs, uint32_t m, float axis_scale, float w_shift, uint64_t* out) {
    const f3 o = mk3(origin[0], origin[1], origin[2]);
    uint64_t pairs = 0, skipped = 0, wrong = 0, hits = 0;
    for (uint32_t s = 0; s < n; ++s) {
        const float4 sp = make_float4(spheres[4 * s], spheres[4 * s + 1], spheres[4 * s + 2], spheres[4 * s + 3]);
        float4 q = cone_of_sphere(o, sp.x, sp.y, sp.z, fabsf(sp.w));
        if (q.w != -2.0f) { q.x *= axis_scale; q.y *= axis_scale; q.z *= axis_scale; q.w += w_shift; }
        for (uint32_t k = 0; k < m; ++k) {
            const float* dv = dirs + 3 * ((size_t)s * m + k);
            const f3 d = norm3(mk3(dv[0], dv[1], dv[2]));
            float t, dist;
            const bool hit = sphere_intersect(sp, o, d, t, dist) != 0, skip = outside_double_cone(q, d);
            ++pairs; skipped += skip; hits += hit; wrong += skip && hit;
        }
    }
    out[0] = pairs; out[1] = skipped; out[2] = wrong; out[3] = hits;
    return 0;
}

// The same for mesh boxes: boxes = n x {lo xyz, hi xyz}; skipped = outside_cone of the box's bounding sphere (as k_generate builds it), hit = mesh_bbox_hit
int hd_cull_boxes(const float* origin, const float* boxes, uint32_t n, const float* dirs, uint32_t m, float axis_scale, float w_shift, uint64_t* out) {
    const f3 o = mk3(origin[0], origin[1], origin[2]);
    uint64_t pairs = 0, skipped = 0, wrong = 0, hits = 0;
    for (uint32_t b = 0; b < n; ++b) {
        MeshDev M; memset(&M, 0, sizeof(M));
        for (int k = 0; k < 3; ++k) { M.lo[k] = boxes[6 * b + k]; M.hi[k] = boxes[6 * b + 3 + k]; }
        const float hx = 0.5f * (M.hi[0] - M.lo[0]), hy = 0.5f * (M.hi[1] - M.lo[1]), hz = 0.5f * (M.hi[2] - M.lo[2]);
        float4 q = cone_of_sphere(o, M.lo[0] + hx, M.lo[1] + hy, M.lo[2] + hz, 1.001f * sqrtf(hx * hx + hy * hy + hz * hz) + 1e-6f);
        if (q.w != -2.0f) { q.x *= axis_scale; q.y *= axis_scale; q.z *= axis_scale; q.w += w_shift; }
        for (uint32_t k = 0; k < m; ++k) {
            const float* dv = dirs + 3 * ((size_t)b * m + k);
            const f3 d = norm3(mk3(dv[0], dv[1], dv[2]));
            const bool hit = mesh_bbox_hit(M, o, d), skip = outside_cone(q, d);
            ++pairs; skipped += skip; hits += hit; wrong += skip && hit;
        }
    }
    out[0] = pairs; out[1] = skipped; out[2] = wrong; out[3] = hits;
    return 0;
}

// fast_div (common.cuh: the pixel mapping's division by launch-invariant divisors): mismatches against `/` over the given dividends and divisors
uint64_t hd_fastdiv_mismatches(const uint32_t* divisors, uint32_t nd, const uint32_t* dividends, uint32_t nn) {
    uint64_t bad = 0;
    for (uint32_t i = 0; i < nd; ++i) {
        const FastDiv f = make_fastdiv(divisors[i]);
        for (uint32_t k = 0; k < nn; ++k) bad += fast_div(dividends[k], f) != dividends[k] / divisors[i];
    }
    return bad;
}

// shard_pixel (common.cuh) over ALL ranks of a tile-sharded W x H image, ShardDev filled as make_shard (render.cu) fills it:
// visits[row * W + col] += 1 for every (rank, j) that maps to a pixel.  A correct mapping leaves every entry at exactly 1.
int hd_shard_visits(uint32_t W, uint32_t H, uint32_t count, uint32_t* visits, uint32_t* max_paths_per_rank) {
    CamDev cam; memset(&cam, 0, sizeof(cam)); cam.width = W; cam.height = H;
    uint32_t most = 0;
    for (uint32_t rank = 0; rank < count; ++rank) {
        ShardDev sh; memset(&sh, 0, sizeof(sh));
        sh.rank = rank; sh.count = count;
        sh.tiles_x = (W + 7) / 8; sh.fd_tiles_x = make_fastdiv(sh.tiles_x); sh.tiles_total = sh.tiles_x * ((H + 3) / 4);
        sh.tiles_mine = sh.tiles_total > sh.rank ? (sh.tiles_total - sh.rank + sh.count - 1) / sh.count : 0;
        const uint32_t P = sh.tiles_mine * 32;
        most = P > most ? P : most;
        for (uint32_t j = 0; j < P; ++j) {
            uint32_t row, col;
            if (shard_pixel(sh, cam, j, row, col)) { if (row >= H || col >= W) return 1; ++visits[(size_t)row * W + col]; }
        }
        uint32_t row, col;                                         // one past the rank's range must not map to a pixel of ANOTHER rank's tile inside the image...
        (void)shard_pixel(sh, cam, P, row, col);                   // (...it may: the kernels never ask; just make sure it does not crash)
    }
    if (max_paths_per_rank) *max_paths_per_rank = most;
    return 0;
}

}  // extern "C"
