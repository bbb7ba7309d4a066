// motion_harness.cpp — TEST INFRASTRUCTURE (tests/test_motion_host.py): the per-pixel code of the motion module, rbrt_b200/csrc/motion.cuh,
// and the motion variant of the temporal step, rbrt_b200/csrc/temporal.cuh, compiled for the host with the cuda_runtime.h stand-in of this
// directory and driven the way motion.cu's and temporal.cu's kernels drive them, with the arguments csrc/api.cu forms.  The tests compare
// the results bit for bit with tests/motion_ref.py.  Nothing under rbrt_b200/ can reach it.
#include "motion.cuh"

using namespace rbrt;

static CamDev cam_dev(const rbrt_camera& c) {
    CamDev d;
    const rbrt_vec3* v[4] = {&c.position, &c.right, &c.up, &c.img_center_point};
    float* o[4] = {d.pos, d.right, d.up, d.center};
    for (int k = 0; k < 4; ++k) { o[k][0] = v[k]->x; o[k][1] = v[k]->y; o[k][2] = v[k]->z; }
    d.mm_per_pix_hor = c.mm_per_pix_hor; d.mm_per_pix_vert = c.mm_per_pix_vert;
    d.width = c.img_width_pix; d.height = c.img_height_pix;
    return d;
}

extern "C" {

// n hits: tri[n] (1: a triangle, 0: a sphere), odt[7n] = o, d, t; cur / old [12n] = three float4 records each.  Outputs motion[2n], pd[n].
int hd_motion(uint32_t n, const rbrt_camera* cam, const rbrt_camera* prev, const int32_t* tri, const float* odt, const float* cur,
              const float* old, float* motion, float* pd) {
    const CamDev c = cam_dev(*cam), p = cam_dev(*prev);
    for (uint32_t i = 0; i < n; ++i) {
        const float* r = odt + 7 * (size_t)i;
        float4 cr[3], od[3];
        for (int k = 0; k < 3; ++k) {
            const float* a = cur + 12 * (size_t)i + 4 * k;
            const float* b = old + 12 * (size_t)i + 4 * k;
            cr[k] = make_float4(a[0], a[1], a[2], a[3]);
            od[k] = make_float4(b[0], b[1], b[2], b[3]);
        }
        mv_pixel(c, p, tri[i] != 0, mk3(r[0], r[1], r[2]), mk3(r[3], r[4], r[5]), r[6], cr, od, &motion[2 * i], &motion[2 * i + 1], &pd[i]);
    }
    return 0;
}

// The pixel-centre ray directions of cam, W*H*3.
int hd_pixel_dirs(const rbrt_camera* cam, float* dirs) {
    const CamDev c = cam_dev(*cam);
    for (uint32_t y = 0; y < c.height; ++y)
        for (uint32_t x = 0; x < c.width; ++x) {
            const f3 d = tp_pixel_dir(c, x, y);
            float* w = dirs + 3 * ((size_t)y * c.width + x);
            w[0] = d.x; w[1] = d.y; w[2] = d.z;
        }
    return 0;
}

// As hd_temporal (temporal_harness.cpp) with the motion planes mv[2]: motion W*H*2, prev_dist W*H.
int hd_temporal_motion(uint32_t W, uint32_t H, const rbrt_camera* cam, const rbrt_camera* prev, const void* const* in, const void* const* hist,
                       const void* const* mv, const float* opt, float* hdr_out, float* var_out, float* len_out) {
    TemporalArgs a;
    memset(&a, 0, sizeof(a));
    a.W = W; a.H = H;
    a.alpha_min = opt[0]; a.sigma_z = opt[1]; a.n_min = opt[2];
    a.cam = cam_dev(*cam);
    a.hdr = (const float*)in[0]; a.var = (const float*)in[1]; a.depth = (const float*)in[2]; a.normal = (const float*)in[3];
    a.kind = (const int32_t*)in[4]; a.elem = (const uint32_t*)in[5];
    a.motion = (const float*)mv[0]; a.prev_dist = (const float*)mv[1];
    if (prev) {
        a.history = 1;
        a.same_cam = memcmp(cam, prev, sizeof(rbrt_camera)) == 0;
        a.prev = cam_dev(*prev);
        a.h_hdr = (const float*)hist[0]; a.h_var = (const float*)hist[1]; a.h_len = (const float*)hist[2]; a.h_depth = (const float*)hist[3];
        a.h_normal = (const float*)hist[4]; a.h_kind = (const int32_t*)hist[5]; a.h_elem = (const uint32_t*)hist[6];
    }
    for (uint32_t y = 0; y < H; ++y)
        for (uint32_t x = 0; x < W; ++x) {
            const size_t p = (size_t)y * W + x;
            f3 o, v;
            float l;
            tp_pixel(a, x, y, &o, &v, &l);
            hdr_out[3 * p] = o.x; hdr_out[3 * p + 1] = o.y; hdr_out[3 * p + 2] = o.z;
            if (var_out) { var_out[3 * p] = v.x; var_out[3 * p + 1] = v.y; var_out[3 * p + 2] = v.z; }
            len_out[p] = l;
        }
    return 0;
}

}  // extern "C"
