// temporal_harness.cpp — TEST INFRASTRUCTURE (tests/test_temporal_host.py): the per-pixel code of the temporal module,
// rbrt_b200/csrc/temporal.cuh, compiled for the host with the cuda_runtime.h stand-in of this directory, and driven the way temporal.cu's
// kernel drives it, with the arguments csrc/api.cu forms (the cameras' fields, same_cam by a bitwise compare).  The tests compare the
// results bit for bit with tests/temporal_ref.py.  Nothing under rbrt_b200/ can reach it.
#include "temporal.cuh"

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

// in[7]: hdr, var (or NULL), depth, normal, hit_kind, elem_idx of the frame; hist[7]: hdr, var, length, depth, normal, hit_kind,
// elem_idx of the history (prev NULL: none); opt[3]: alpha_min, sigma_z, n_min.  Outputs W*H*3, W*H*3 (or NULL), W*H.
int hd_temporal(uint32_t W, uint32_t H, const rbrt_camera* cam, const rbrt_camera* prev, const void* const* in, const void* const* hist,
                const float* opt, float* hdr_out, float* var_out, float* len_out) {
    TemporalArgs a;
    memset(&a, 0, sizeof(a));
    a.W = W; a.H = H;
    a.alpha_min = opt[0]; a.sigma_z = opt[1]; a.n_min = opt[2];
    a.cam = cam_dev(*cam);
    a.hdr = (const float*)in[0]; a.var = (const float*)in[1]; a.depth = (const float*)in[2]; a.normal = (const float*)in[3];
    a.kind = (const int32_t*)in[4]; a.elem = (const uint32_t*)in[5];
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
