// point_harness.cpp — TEST INFRASTRUCTURE (tests/test_point_host.py): the per-candidate routines and the prune bound of the nearest-surface
// module, rbrt_b200/csrc/point.cuh, compiled for the host with the cuda_runtime.h stand-in of this directory.  The tests compare the results
// bit for bit with tests/point_ref.py.  Nothing under rbrt_b200/ can reach it.
#include "point.cuh"

using namespace rbrt;

extern "C" {

// n triangles: p[3n], rec[9n] = v0, e1, e2.  Outputs d2[n], q[3n], uv[2n].
int hd_triangle(uint32_t n, const float* p, const float* rec, float* d2, float* q, float* uv) {
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        const float* r = rec + 9 * (size_t)i;
        f3 qq; float u, v;
        d2[i] = closest_on_triangle(mk3(a[0], a[1], a[2]), mk3(r[0], r[1], r[2]), mk3(r[3], r[4], r[5]), mk3(r[6], r[7], r[8]), qq, u, v);
        q[3 * i] = qq.x; q[3 * i + 1] = qq.y; q[3 * i + 2] = qq.z; uv[2 * i] = u; uv[2 * i + 1] = v;
    }
    return 0;
}

// n spheres: p[3n], s[4n] = {c, r}.  Outputs d2[n], q[3n].
int hd_sphere(uint32_t n, const float* p, const float* s, float* d2, float* q) {
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        const float* c = s + 4 * (size_t)i;
        f3 qq;
        d2[i] = closest_on_sphere(mk3(a[0], a[1], a[2]), make_float4(c[0], c[1], c[2], c[3]), qq);
        q[3 * i] = qq.x; q[3 * i + 1] = qq.y; q[3 * i + 2] = qq.z;
    }
    return 0;
}

// n boxes: p[3n], box[6n] = lo, hi; md[n], best[n]; mesh[6n] = the mesh box that sets the scale.  Outputs box_d2[n], prune_d2[n], acc[n].
int hd_prune(uint32_t n, const float* p, const float* box, const float* md, const float* best, const float* mesh, float* box_d2, float* prune_d2,
             int32_t* acc) {
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        const float* b = box + 6 * (size_t)i;
        const f3 pp = mk3(a[0], a[1], a[2]);
        MeshDev M;
        memset(&M, 0, sizeof(M));
        for (int k = 0; k < 3; ++k) { M.lo[k] = mesh[6 * i + k]; M.hi[k] = mesh[6 * i + 3 + k]; }
        box_d2[i] = pt_box_d2(pp, b[0], b[1], b[2], b[3], b[4], b[5]);
        prune_d2[i] = pt_prune_d2(md[i], best[i], pt_scale(pp, M));
        acc[i] = pt_accept(best[i], md[i]);
    }
    return 0;
}

}  // extern "C"
