// query_harness.cpp — TEST INFRASTRUCTURE (tests/test_query_host.py): the occlusion rule of rbrt_b200/csrc/query.cuh compiled for the host.
//
// harness.cpp (included whole: its scene flattening and host-built 4-wide trees) runs Scene::hit from the product's device headers; this
// adds query.cuh's occluded_ray, the one-lane form of what the occlusion kernel does per ray (elements, the early-exit rule, the voted
// traversal with the exit step), and beside it the definition it must equal: Scene::hit (scene_hit, brute force or BVH) composed with the
// strict max_dist compare.  Nothing under rbrt_b200/ can reach it.
#include "harness.cpp"
#include "query.cuh"

extern "C" {

// occ_out[i] = occluded_ray for ray i (leaf_size 1..8: over a host-built tree of such leaves), ref_out[i] = the composition:
// 2 for a NaN ray, 1 for a hit with dist < max_dist[i], else 0, with Scene::hit by brute force (ref_bvh 0) or by the BVH (ref_bvh 1).
int hd_occluded(const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, const rbrt_triangle_desc* btris, const rbrt_mesh_desc* meshes,
                uint32_t nm, uint32_t lanes, uint32_t leaf_size, const rbrt_ray* rays, const float* max_dist, uint64_t n, int ref_bvh,
                uint8_t* occ_out, uint8_t* ref_out, uint64_t* node_visits) {
    HostScene hs; flatten(hs, order, ne, spheres, btris, meshes, nm, lanes, leaf_size);
    int32_t lstack[RBRT_STACK]; const StackL stack = {lstack};
    TraceCounters cnt; cnt.nodes = 0; cnt.tris = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const f3 o = mk3(rays[i].origin.x, rays[i].origin.y, rays[i].origin.z), d = mk3(rays[i].direction.x, rays[i].direction.y, rays[i].direction.z);
        occ_out[i] = (uint8_t)occluded_ray(hs.dev, o, d, max_dist[i], stack, &cnt);
        const Hit h = ref_bvh ? scene_hit<false>(hs.dev, o, d, nullptr) : scene_hit<true>(hs.dev, o, d, nullptr);
        ref_out[i] = h.kind == -2 ? 2 : (h.kind >= 0 && h.dist < max_dist[i] ? 1 : 0);
    }
    if (node_visits) *node_visits = cnt.nodes;
    return 0;
}

}  // extern "C"
