// winding_harness.cpp — TEST INFRASTRUCTURE (tests/test_winding_host.py): the terms, the far test, the expansion and the moments of the
// winding-number module, rbrt_b200/csrc/winding.cuh, compiled for the host with the cuda_runtime.h stand-in of this directory.  The tests
// compare the results with float64 restatements (tests/winding_ref.py).  Nothing under rbrt_b200/ can reach it.
#include "winding.cuh"

using namespace rbrt;

extern "C" {

// n triangles: p[3n], rec[9n] = v0, e1, e2.  Output om[n].
int hd_tri(uint32_t n, const float* p, const float* rec, float* om) {
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        const float* r = rec + 9 * (size_t)i;
        om[i] = wind_tri(mk3(a[0], a[1], a[2]), mk3(r[0], r[1], r[2]), mk3(r[3], r[4], r[5]), mk3(r[6], r[7], r[8]));
    }
    return 0;
}

// n spheres: p[3n], s[4n] = {c, r}.  Output halves[n].
int hd_sphere(uint32_t n, const float* p, const float* s, int32_t* halves) {
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        const float* c = s + 4 * (size_t)i;
        halves[i] = wind_sphere(mk3(a[0], a[1], a[2]), make_float4(c[0], c[1], c[2], c[3]));
    }
    return 0;
}

// The record (16 floats) and area of cnt (1..8) triangle records tris[12 cnt] (3 float4 each, as the scene stores them).
int hd_leaf(uint32_t cnt, const float* tris, float* rec, double* area) {
    WindMom m;
    wind_leaf(reinterpret_cast<const float4*>(tris), cnt, m);
    wind_store(m, reinterpret_cast<float4*>(rec));
    *area = m.area;
    return 0;
}

// The merge of four child records rec[64] (R < 0: unused) with their areas; returns 0 when no child is used.
int hd_merge(const float* rec, const double* area, float* out, double* out_area) {
    float4 r[4][4];
    memcpy(r, rec, sizeof(r));
    WindMom m;
    if (!wind_merge(r, area, m)) return 0;
    wind_store(m, reinterpret_cast<float4*>(out));
    *out_area = m.area;
    return 1;
}

// n points p[3n] against one record rec[16]: far[n] (the test with beta) and om[n] (the expansion, evaluated whatever the test says).
int hd_far(uint32_t n, const float* p, const float* rec, float beta, int32_t* far, float* om) {
    const float4* r = reinterpret_cast<const float4*>(rec);
    for (uint32_t i = 0; i < n; ++i) {
        const float* a = p + 3 * (size_t)i;
        f3 u; float inv;
        far[i] = wind_far(mk3(a[0], a[1], a[2]), r[0], beta, u, inv);
        om[i] = wind_expand(u, inv, r[1], r[2], r[3]);
    }
    return 0;
}

}  // extern "C"
