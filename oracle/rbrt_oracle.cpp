// rbrt_oracle.cpp — CPU ORACLE.  TEST INFRASTRUCTURE ONLY.
//
// A statement-for-statement CPU restatement of the hot path of baurst/rbrt (Rust), written
// because no Rust toolchain exists in the build image (cargo/rustc absent, no network), so the
// reference itself cannot be compiled or run.  Nothing under rbrt_b200/ may link, import or
// call this file; only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs use it,
// and only as the checker / the CPU number reported beside the GPU one.
//
// Build (oracle/Makefile):  g++ -O2 -mavx -ffp-contract=off -shared -fPIC   (NO -mfma, NO
// -ffast-math: Rust never contracts a*b+c, so neither may we; every f32 op below rounds once.)
//
// Pinning: the functions below are checked against every exact-equality unit test the
// reference holds for this path (tests/test_oracle_kat.py: sphere.rs:76-112,
// triangle.rs:449-475, aabbox.rs:95-108, materials.rs:43-59, dielectric.rs:93-115,
// vec3_avx.rs:60-110, vec3.rs:166-342).  What the reference's tests do NOT pin (ray-triangle
// t/index, BoundingBox::hit, camera rays, Scene::hit ordering, colorize, scatter, gamma) is
// pinned by this restatement only: for those rows "parity unpinned by reference tests".
//
// RNG: the reference draws from rand 0.8 `thread_rng()` (OS-seeded ChaCha, per rayon thread;
// call sites cam.rs:69,71, materials.rs:17-19,24-26, dielectric.rs:48), which cannot be seeded
// through rbrt's API, so no draw sequence exists to reproduce.  The oracle and the GPU path both
// use counter-based Philox4x32-10 keyed on (seed; pixel, sample, bounce, round) — implemented
// independently on each side — so that equal seeds give bit-identical images.  f32 conversion is
// rand 0.8's Standard: (u32 >> 8) * 2^-24 in [0,1).
//
// All citations are file:line in /root/reference/rbrt_lib/src/ unless noted.

#include <immintrin.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "../include/rbrt_gpu.h"

namespace {

// ------------------------------------------------------------------ vec3.rs:6-160
struct V3 { float x, y, z; };
inline V3 v3(float x, float y, float z) { return V3{x, y, z}; }
inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }   // vec3.rs:12-22
inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }   // vec3.rs:23-34
inline V3 operator*(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }   // vec3.rs:57-67
inline V3 operator*(float s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }      // vec3.rs:68-78
inline V3 operator*(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }      // vec3.rs:80-90
inline float sum(V3 a) { return a.x + a.y + a.z; }                                // vec3.rs:115-117
inline float dot(V3 a, V3 b) { return sum(a * b); }                               // vec3.rs:157-159
inline float length(V3 a) { return sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); }    // vec3.rs:111-113
inline V3 normalize(V3 a) { float l = length(a); return v3(a.x / l, a.y / l, a.z / l); }  // :119-126
inline V3 cross(V3 a, V3 b) {                                                     // vec3.rs:128-134
    return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
inline V3 rotate_point(V3 p, V3 rot) {                                            // vec3.rs:139-155
    float s_x = sinf(rot.x), s_y = sinf(rot.y), s_z = sinf(rot.z);
    float c_x = cosf(rot.x), c_y = cosf(rot.y), c_z = cosf(rot.z);
    float x = p.x, y = p.y, z = p.z;
    return v3((c_x * c_z - c_y * s_x * s_z) * x - (c_x * s_z + c_y * c_z * s_x) * y + s_x * s_y * z,
              (c_z * s_x + c_x * c_y * s_z) * x + (c_x * c_y * c_z - s_x * s_z) * y - c_x * s_y * z,
              s_y * s_z * x + c_z * s_y * y + c_y * z);
}
inline V3 from(rbrt_vec3 v) { return v3(v.x, v.y, v.z); }
inline rbrt_vec3 to(V3 v) { return rbrt_vec3{v.x, v.y, v.z}; }

struct Ray { V3 origin, direction; };                                             // ray.rs:4-7
inline V3 point_at(const Ray& r, float t) { return r.origin + t * r.direction; }  // ray.rs:10-12

// ------------------------------------------------------------------ Philox4x32-10
inline void philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
inline float u32_to_f32(uint32_t u) { return (float)(u >> 8) * (1.0f / 16777216.0f); }

// One path's RNG: key = seed, counter = (pixel, sample, bounce, round).  Every request site
// (camera jitter; one rejection round of random_point_in_unit_sphere; the dielectric coin) takes
// one Philox block and uses its first 2 / 3 / 1 words.
struct PathRng {
    uint32_t key[2]; uint32_t pixel, sample, bounce, round;
    void block(float* f, int n) {
        uint32_t c[4] = {pixel, sample, bounce, round}, o[4];
        philox4x32_10(c, key, o);
        for (int i = 0; i < n; ++i) f[i] = u32_to_f32(o[i]);
        ++round;
    }
    void next_bounce() { ++bounce; round = 0; }
};

// ------------------------------------------------------------------ cam.rs
rbrt_camera camera_new(V3 position, V3 look_at, V3 up, uint32_t h, uint32_t w, float focal) {  // cam.rs:22-62
    V3 right = normalize(cross(normalize(look_at), normalize(up)));
    float img_width_mm = 35.0f;
    float mm_per_pix_hor = img_width_mm / (float)w;
    float img_height_mm = (float)h * mm_per_pix_hor;
    float mm_per_pix_vert = img_height_mm / (float)h;
    V3 center = position + focal / 1000.0f * normalize(look_at);
    float hor_fov = 2.0f * atanf(2.0f * focal / img_width_mm);
    float vert_fov = 2.0f * atanf(2.0f * focal / img_height_mm);
    rbrt_camera c;
    c.hor_fov_rad = hor_fov; c.img_width_pix = w; c.img_height_mm = img_height_mm;
    c.vert_fov_rad = vert_fov; c.img_height_pix = h; c.img_width_mm = img_width_mm;
    c.position = to(position); c.focal_len_mm = focal; c.look_at = to(look_at); c.up = to(up);
    c.right = to(right); c.img_center_point = to(center);
    c.mm_per_pix_hor = mm_per_pix_hor; c.mm_per_pix_vert = mm_per_pix_vert;
    return c;
}

Ray get_ray_through_pixel(const rbrt_camera& c, uint32_t row, uint32_t col, PathRng& rng) {  // cam.rs:64-82
    float col_off = (float)col - (float)(c.img_width_pix / 2);
    float row_off = (float)row - (float)(c.img_height_pix / 2);
    float u[2]; rng.block(u, 2);                       // col draw before row draw (cam.rs:69,71)
    float col_mm = (col_off + u[0] - 0.5f) * c.mm_per_pix_hor;
    float row_mm = (row_off + u[1] - 0.5f) * c.mm_per_pix_vert;
    V3 target = from(c.img_center_point) + 0.001f * col_mm * from(c.right) - 0.001f * row_mm * from(c.up);
    V3 dir = normalize(target - from(c.position));
    return Ray{from(c.position), dir};
}

// ------------------------------------------------------------------ scene data
struct Material { uint32_t kind; V3 albedo; float param; };
struct Sphere { V3 center; float radius; Material mat; };

struct Mesh {                                           // mesh.rs:12-25
    std::vector<float> v0[3], e1[3], e2[3], nrm[3];     // the 12 SoA arrays the hot path touches
    std::vector<uint8_t> is_padding;
    V3 lo, hi;
    Material mat;
    size_t n_real;
};

struct HitInfo {                                        // lib.rs:31-36 (+ ids for the parity hook)
    V3 point, normal; const Material* mat; float dist;
    int kind; uint32_t elem, tri; float t;
};

// ------------------------------------------------------------------ sphere.rs:20-66
// returns 0 = None, 1 = Some, -1 = the reference would panic ("Encountered NAN", sphere.rs:33)
int sphere_intersect(const Sphere& s, const Ray& ray, float min_dist, float max_dist, HitInfo& out) {
    float a = dot(ray.direction, ray.direction);
    V3 l = ray.origin - s.center;
    float b = dot(ray.direction * 2.0f, l);
    float c = dot(l, l) - s.radius * s.radius;          // powf(2.0)
    float sol = b * b - 4.0f * a * c;
    if (sol != sol) return -1;
    int num_hits = sol < 0.0f ? 0 : (sol > 0.0f ? 2 : 1);
    if (num_hits == 0) return 0;
    float t = (-b - sqrtf(sol)) / (2.0f * a);
    if (num_hits == 2 && t < 0.0f) {
        t = (-b + sqrtf(sol)) / (2.0f * a);
        if (t < 0.0f) return 0;
    }
    V3 p = point_at(ray, t);
    float dist = length(ray.origin - p);
    if (dist < min_dist || dist > max_dist) return 0;
    out.normal = p - s.center; out.point = p; out.mat = &s.mat; out.dist = dist; out.t = t;
    return 1;
}

// ------------------------------------------------------------------ aabbox.rs
inline float rmin(float a, float b) { return fminf(a, b); }   // f32::min: NaN-ignoring (aabbox.rs:16-18)
inline float rmax(float a, float b) { return fmaxf(a, b); }   // f32::max (aabbox.rs:12-14)

bool bbox_hit(V3 lo, V3 hi, const Ray& ray) {                 // aabbox.rs:28-58
    float tlx = (lo.x - ray.origin.x) / ray.direction.x, tux = (hi.x - ray.origin.x) / ray.direction.x;
    float tly = (lo.y - ray.origin.y) / ray.direction.y, tuy = (hi.y - ray.origin.y) / ray.direction.y;
    float tlz = (lo.z - ray.origin.z) / ray.direction.z, tuz = (hi.z - ray.origin.z) / ray.direction.z;
    float t_min = rmax(rmax(rmin(tlx, tux), rmin(tly, tuy)), rmin(tlz, tuz));
    float t_max = rmin(rmin(rmax(tlx, tux), rmax(tly, tuy)), rmax(tlz, tuz));
    if (t_max < 0.0f) return false;
    if (t_min > t_max) return false;
    return true;
}

void compute_min_max_3d(const float* tris, size_t n, V3& lo, V3& hi) {   // aabbox.rs:62-88
    lo = v3(3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f);
    hi = v3(-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f);
    for (size_t i = 0; i < n * 3; ++i) {
        float x = tris[3 * i], y = tris[3 * i + 1], z = tris[3 * i + 2];
        if (x < lo.x) lo.x = x;
        if (y < lo.y) lo.y = y;
        if (z < lo.z) lo.z = z;
        if (x > hi.x) hi.x = x;
        if (y > hi.y) hi.y = y;
        if (z > hi.z) hi.z = z;
    }
}

V3 triangle_normal(V3 a, V3 b, V3 c) { return normalize(cross(b - a, c - a)); }   // triangle.rs:30-34

// ------------------------------------------------------------------ mesh.rs:41-74, 123-181
Mesh* mesh_new(const float* tris, size_t n, Material mat, unsigned lanes) {
    Mesh* m = new Mesh();
    m->mat = mat; m->n_real = n;
    compute_min_max_3d(tris, n, m->lo, m->hi);              // before padding (mesh.rs:61)
    size_t pad = lanes ? n % lanes : 0;                      // mesh.rs:136: the remainder, not the complement
    size_t total = n + pad;
    for (int k = 0; k < 3; ++k) { m->v0[k].resize(total); m->e1[k].resize(total); m->e2[k].resize(total); m->nrm[k].resize(total); }
    m->is_padding.assign(total, 0);
    for (size_t i = 0; i < total; ++i) {
        size_t src = i < n ? i : 0;                          // padding = copies of triangle 0 (mesh.rs:140-143)
        const float* t = tris + 9 * src;
        V3 a = v3(t[0], t[1], t[2]), b = v3(t[3], t[4], t[5]), c = v3(t[6], t[7], t[8]);
        V3 ea = b - a, eb = c - a, nn = triangle_normal(a, b, c);
        m->v0[0][i] = a.x; m->v0[1][i] = a.y; m->v0[2][i] = a.z;
        m->e1[0][i] = ea.x; m->e1[1][i] = ea.y; m->e1[2][i] = ea.z;
        m->e2[0][i] = eb.x; m->e2[1][i] = eb.y; m->e2[2][i] = eb.z;
        m->nrm[0][i] = nn.x; m->nrm[1][i] = nn.y; m->nrm[2][i] = nn.z;
        if (i >= n) m->is_padding[i] = 1;
    }
    return m;
}

// ------------------------------------------------------------------ vec3_avx.rs:10-45
inline __m256 avx_dot(__m256 ax, __m256 ay, __m256 az, __m256 bx, __m256 by, __m256 bz) {
    __m256 x = _mm256_mul_ps(ax, bx), y = _mm256_mul_ps(ay, by), z = _mm256_mul_ps(az, bz);
    return _mm256_add_ps(_mm256_add_ps(x, y), z);
}
inline void avx_cross(__m256 ax, __m256 ay, __m256 az, __m256 bx, __m256 by, __m256 bz,
                      __m256& cx, __m256& cy, __m256& cz) {
    cx = _mm256_sub_ps(_mm256_mul_ps(ay, bz), _mm256_mul_ps(az, by));
    cy = _mm256_sub_ps(_mm256_mul_ps(az, bx), _mm256_mul_ps(ax, bz));
    cz = _mm256_sub_ps(_mm256_mul_ps(ax, by), _mm256_mul_ps(ay, bx));
}
// vec3_sse.rs:10-44 (same shapes, 4 lanes)
inline __m128 sse_dot(__m128 ax, __m128 ay, __m128 az, __m128 bx, __m128 by, __m128 bz) {
    __m128 x = _mm_mul_ps(ax, bx), y = _mm_mul_ps(ay, by), z = _mm_mul_ps(az, bz);
    return _mm_add_ps(_mm_add_ps(x, y), z);
}
inline void sse_cross(__m128 ax, __m128 ay, __m128 az, __m128 bx, __m128 by, __m128 bz,
                      __m128& cx, __m128& cy, __m128& cz) {
    cx = _mm_sub_ps(_mm_mul_ps(ay, bz), _mm_mul_ps(az, by));
    cy = _mm_sub_ps(_mm_mul_ps(az, bx), _mm_mul_ps(ax, bz));
    cz = _mm_sub_ps(_mm_mul_ps(ax, by), _mm_mul_ps(ay, bx));
}

// ------------------------------------------------------------------ triangle.rs:392-410
bool find_smallest_bigger_than_eps(const float* params, size_t n, const uint8_t* is_pad, float eps,
                                   float& t_out, size_t& idx_out) {
    size_t min_idx = 0; float min_param = 1000000.0f;
    for (size_t i = 0; i < n; ++i) {
        float p = params[i];
        if (p > eps && p < min_param && !is_pad[i]) { min_param = p; min_idx = i; }
    }
    if (min_param > eps && min_param < 100000.0f) { t_out = min_param; idx_out = min_idx; return true; }
    return false;
}

// ------------------------------------------------------------------ triangle.rs:134-262 (AVX, 8 lanes)
bool triangle_soa_avx(const Mesh& m, const Ray& ray, float min_dist, std::vector<float>& params,
                      float& t_out, size_t& idx_out) {
    size_t total = m.v0[0].size();
    // the reference heap-allocates this Vec per ray (triangle.rs:142); the oracle reuses one per thread
    float eps_f = min_dist;
    __m256 eps = _mm256_set1_ps(eps_f), eps_frac = _mm256_set1_ps(1.0f / eps_f), neg_eps = _mm256_set1_ps(-eps_f);
    __m256 zero = _mm256_set1_ps(0.0f), one = _mm256_set1_ps(1.0f);
    __m256 ro_x = _mm256_set1_ps(ray.origin.x), ro_y = _mm256_set1_ps(ray.origin.y), ro_z = _mm256_set1_ps(ray.origin.z);
    __m256 rd_x = _mm256_set1_ps(ray.direction.x), rd_y = _mm256_set1_ps(ray.direction.y), rd_z = _mm256_set1_ps(ray.direction.z);
    size_t chunks = total / 8;                              // chunks_exact(8) (triangle.rs:167)
    if (params.size() != chunks * 8) params.resize(chunks * 8);
    for (size_t ch = 0; ch < chunks; ++ch) {
        size_t o = ch * 8;
        __m256 vax = _mm256_loadu_ps(&m.v0[0][o]), vay = _mm256_loadu_ps(&m.v0[1][o]), vaz = _mm256_loadu_ps(&m.v0[2][o]);
        __m256 eax = _mm256_loadu_ps(&m.e1[0][o]), eay = _mm256_loadu_ps(&m.e1[1][o]), eaz = _mm256_loadu_ps(&m.e1[2][o]);
        __m256 ebx = _mm256_loadu_ps(&m.e2[0][o]), eby = _mm256_loadu_ps(&m.e2[1][o]), ebz = _mm256_loadu_ps(&m.e2[2][o]);
        __m256 hx, hy, hz; avx_cross(rd_x, rd_y, rd_z, ebx, eby, ebz, hx, hy, hz);          // h = d x e2
        __m256 a = avx_dot(eax, eay, eaz, hx, hy, hz);                                         // a = e1 . h
        __m256 c1 = _mm256_and_ps(_mm256_cmp_ps(neg_eps, a, _CMP_LT_OQ), _mm256_cmp_ps(a, eps, _CMP_LT_OQ));
        __m256 f = _mm256_div_ps(one, a);
        __m256 sx = _mm256_sub_ps(ro_x, vax), sy = _mm256_sub_ps(ro_y, vay), sz = _mm256_sub_ps(ro_z, vaz);
        __m256 u = _mm256_mul_ps(f, avx_dot(sx, sy, sz, hx, hy, hz));
        __m256 c2 = _mm256_or_ps(_mm256_cmp_ps(u, zero, _CMP_LT_OQ), _mm256_cmp_ps(u, one, _CMP_GT_OQ));
        __m256 qx, qy, qz; avx_cross(sx, sy, sz, eax, eay, eaz, qx, qy, qz);                  // q = s x e1
        __m256 v = _mm256_mul_ps(f, avx_dot(rd_x, rd_y, rd_z, qx, qy, qz));
        __m256 c3 = _mm256_or_ps(_mm256_cmp_ps(v, zero, _CMP_LT_OQ), _mm256_cmp_ps(_mm256_add_ps(u, v), one, _CMP_GT_OQ));
        __m256 t = _mm256_mul_ps(f, avx_dot(ebx, eby, ebz, qx, qy, qz));
        __m256 c4 = _mm256_and_ps(_mm256_cmp_ps(t, eps, _CMP_GT_OQ), _mm256_cmp_ps(t, eps_frac, _CMP_LT_OQ));
        __m256 c123 = _mm256_or_ps(c1, _mm256_or_ps(c2, c3));
        __m256 has = _mm256_andnot_ps(c123, c4);
        __m256 res = _mm256_or_ps(_mm256_and_ps(has, t), _mm256_andnot_ps(has, _mm256_set1_ps(-1000.0f)));
        _mm256_storeu_ps(&params[o], res);
    }
    return find_smallest_bigger_than_eps(params.data(), params.size(), m.is_padding.data(), eps_f, t_out, idx_out);
}

// ------------------------------------------------------------------ triangle.rs:266-390 (SSE, 4 lanes)
bool triangle_soa_sse(const Mesh& m, const Ray& ray, float min_dist, std::vector<float>& params,
                      float& t_out, size_t& idx_out) {
    size_t total = m.v0[0].size();
    float eps_f = min_dist;
    __m128 eps = _mm_set1_ps(eps_f), eps_frac = _mm_set1_ps(1.0f / eps_f), neg_eps = _mm_set1_ps(-eps_f);
    __m128 zero = _mm_set1_ps(0.0f), one = _mm_set1_ps(1.0f);
    __m128 ro_x = _mm_set1_ps(ray.origin.x), ro_y = _mm_set1_ps(ray.origin.y), ro_z = _mm_set1_ps(ray.origin.z);
    __m128 rd_x = _mm_set1_ps(ray.direction.x), rd_y = _mm_set1_ps(ray.direction.y), rd_z = _mm_set1_ps(ray.direction.z);
    size_t chunks = total / 4;                              // chunks_exact(4) (triangle.rs:296)
    if (params.size() != chunks * 4) params.resize(chunks * 4);
    for (size_t ch = 0; ch < chunks; ++ch) {
        size_t o = ch * 4;
        __m128 vax = _mm_loadu_ps(&m.v0[0][o]), vay = _mm_loadu_ps(&m.v0[1][o]), vaz = _mm_loadu_ps(&m.v0[2][o]);
        __m128 eax = _mm_loadu_ps(&m.e1[0][o]), eay = _mm_loadu_ps(&m.e1[1][o]), eaz = _mm_loadu_ps(&m.e1[2][o]);
        __m128 ebx = _mm_loadu_ps(&m.e2[0][o]), eby = _mm_loadu_ps(&m.e2[1][o]), ebz = _mm_loadu_ps(&m.e2[2][o]);
        __m128 hx, hy, hz; sse_cross(rd_x, rd_y, rd_z, ebx, eby, ebz, hx, hy, hz);
        __m128 a = sse_dot(eax, eay, eaz, hx, hy, hz);
        __m128 c1 = _mm_and_ps(_mm_cmplt_ps(neg_eps, a), _mm_cmplt_ps(a, eps));
        __m128 f = _mm_div_ps(one, a);
        __m128 sx = _mm_sub_ps(ro_x, vax), sy = _mm_sub_ps(ro_y, vay), sz = _mm_sub_ps(ro_z, vaz);
        __m128 u = _mm_mul_ps(f, sse_dot(sx, sy, sz, hx, hy, hz));
        __m128 c2 = _mm_or_ps(_mm_cmplt_ps(u, zero), _mm_cmpgt_ps(u, one));
        __m128 qx, qy, qz; sse_cross(sx, sy, sz, eax, eay, eaz, qx, qy, qz);
        __m128 v = _mm_mul_ps(f, sse_dot(rd_x, rd_y, rd_z, qx, qy, qz));
        __m128 c3 = _mm_or_ps(_mm_cmplt_ps(v, zero), _mm_cmpgt_ps(_mm_add_ps(u, v), one));
        __m128 t = _mm_mul_ps(f, sse_dot(ebx, eby, ebz, qx, qy, qz));
        __m128 c4 = _mm_and_ps(_mm_cmpgt_ps(t, eps), _mm_cmplt_ps(t, eps_frac));
        __m128 c123 = _mm_or_ps(c1, _mm_or_ps(c2, c3));
        __m128 has = _mm_andnot_ps(c123, c4);
        __m128 res = _mm_or_ps(_mm_and_ps(has, t), _mm_andnot_ps(has, _mm_set1_ps(-1000.0f)));
        _mm_storeu_ps(&params[o], res);
    }
    return find_smallest_bigger_than_eps(params.data(), params.size(), m.is_padding.data(), eps_f, t_out, idx_out);
}

// triangle.rs:9-28 (BasicTriangle) — a single triangle as an element of Scene.elements
struct BasicTri { V3 corners[3]; V3 normal; V3 edges[2]; Material mat; };

// triangle.rs:92-130
bool basic_triangle_intersect_w_ray(const Ray& ray, const V3 vertices[3], const V3 edges[2], float min_dist, float max_dist, float& t_out) {
    float eps = min_dist;
    V3 h = cross(ray.direction, edges[1]);
    float a = dot(edges[0], h);
    if (-eps < a && a < eps) return false;
    float f = 1.0f / a;
    V3 s = ray.origin - vertices[0];
    float u = f * dot(s, h);
    if (!(0.0f <= u && u <= 1.0f)) return false;                          // !(0.0..=1.0).contains(&u): NaN is not contained
    V3 q = cross(s, edges[0]);
    float v = f * dot(ray.direction, q);
    if (v < 0.0f || u + v > 1.0f) return false;
    float t = f * dot(edges[1], q);
    if (t > eps) {
        V3 p = point_at(ray, t);
        float dist = length(ray.origin - p);
        if (dist < min_dist || dist > max_dist) return false;
        t_out = t;
        return true;
    }
    return false;
}

// triangle.rs:412-441 (impl Intersectable for BasicTriangle)
int basic_triangle_intersect(const BasicTri& tr, const Ray& ray, float min_dist, float max_dist, HitInfo& out) {
    float t;
    if (!basic_triangle_intersect_w_ray(ray, tr.corners, tr.edges, min_dist, max_dist, t)) return 0;
    V3 p = point_at(ray, t);
    float dist = length(ray.origin - p);
    if (dist < min_dist || dist > max_dist) return 0;
    out.point = p; out.normal = tr.normal; out.mat = &tr.mat; out.dist = dist; out.t = t;
    return 1;
}

struct Element { uint32_t kind; uint32_t index; };                        // entry of Scene.elements: sphere or BasicTriangle

struct Scene {
    std::vector<Element> elements;                                        // iteration order of scene.rs:23-31
    std::vector<BasicTri> btris;
    std::vector<Sphere> spheres;
    std::vector<Mesh*> meshes;
    unsigned lanes = 8;
    ~Scene() { for (auto* m : meshes) delete m; }
};

// ------------------------------------------------------------------ mesh.rs:225-268
bool mesh_intersect(const Scene& sc, const Mesh& m, const Ray& ray, float min_dist, float max_dist,
                    std::vector<float>& scratch, HitInfo& out) {
    if (!bbox_hit(m.lo, m.hi, ray)) return false;
    float t; size_t idx;
    bool ok = sc.lanes == 4 ? triangle_soa_sse(m, ray, min_dist, scratch, t, idx)
                            : triangle_soa_avx(m, ray, min_dist, scratch, t, idx);
    if (!ok) return false;
    V3 p = point_at(ray, t);
    float dist = length(ray.origin - p);
    if (dist > min_dist && dist < max_dist) {
        out.point = p; out.normal = v3(m.nrm[0][idx], m.nrm[1][idx], m.nrm[2][idx]);
        out.mat = &m.mat; out.dist = dist; out.t = t; out.tri = (uint32_t)idx;
        return true;
    }
    return false;
}

// ------------------------------------------------------------------ scene.rs:19-43
// returns 1 hit, 0 miss, -1 NaN panic
int scene_hit(const Scene& sc, const Ray& ray, float min_dist, float max_dist,
              std::vector<float>& scratch, HitInfo& best) {
    bool found = false; float closest = 3.40282347e+38f;
    for (size_t i = 0; i < sc.elements.size(); ++i) {
        HitInfo h; h.tri = 0;
        const Element& e = sc.elements[i];
        int r = e.kind == RBRT_ELEM_SPHERE ? sphere_intersect(sc.spheres[e.index], ray, min_dist, max_dist, h)
                                           : basic_triangle_intersect(sc.btris[e.index], ray, min_dist, max_dist, h);
        if (r < 0) return -1;
        if (r && h.dist < closest) {
            closest = h.dist; best = h; best.kind = e.kind == RBRT_ELEM_SPHERE ? RBRT_HIT_SPHERE : RBRT_HIT_TRIANGLE; best.elem = (uint32_t)i; found = true;
        }
    }
    for (size_t i = 0; i < sc.meshes.size(); ++i) {
        HitInfo h;
        if (mesh_intersect(sc, *sc.meshes[i], ray, min_dist, max_dist, scratch, h) && h.dist < closest) {
            closest = h.dist; best = h; best.kind = RBRT_HIT_MESH; best.elem = (uint32_t)i; found = true;
        }
    }
    return found ? 1 : 0;
}

// ------------------------------------------------------------------ materials.rs
V3 random_point_in_unit_sphere(PathRng& rng) {                 // materials.rs:14-30
    float u[3]; rng.block(u, 3);
    V3 p = 2.0f * v3(u[0], u[1], u[2]) - v3(1.0f, 1.0f, 1.0f);
    while (length(p) > 1.0f) {
        rng.block(u, 3);
        p = 2.0f * v3(u[0], u[1], u[2]) - v3(1.0f, 1.0f, 1.0f);
    }
    return p;
}
V3 reflect(V3 d, V3 n) {                                       // materials.rs:32-37
    V3 du = normalize(d), nu = normalize(n);
    V3 r = du - 2.0f * nu * dot(du, nu);
    return normalize(r);
}
inline float powi2(float x) { return x * x; }
inline float powi5(float x) { float x2 = x * x; float x4 = x2 * x2; return x * x4; }   // llvm.powi: square-and-multiply
float schlick(float cosine, float ref_index) {                 // dielectric.rs:63-66
    float r0 = powi2((1.0f - ref_index) / (1.0f + ref_index));
    return r0 + (1.0f - r0) * powi5(1.0f - cosine);
}
bool refract(V3 d, V3 n, float ni_over_nt, V3& out) {          // dielectric.rs:68-85
    V3 vu = normalize(d), nu = normalize(n);
    float c = dot(vu, nu);
    float discr = 1.0f - powi2(ni_over_nt) * (1.0f - powi2(c));
    if (discr > 0.0f) { out = ni_over_nt * (vu - nu * c) - sqrtf(discr) * nu; return true; }
    return false;
}

bool scatter(const Material& m, const Ray& in, const HitInfo& h, PathRng& rng, V3& att, Ray& out) {
    if (m.kind == RBRT_MAT_LAMBERTIAN) {                       // lambertian.rs:11-24
        V3 target = h.point + normalize(h.normal) + random_point_in_unit_sphere(rng);
        out.direction = normalize(target - h.point);
        out.origin = h.point;
        att = m.albedo;
        return true;
    } else if (m.kind == RBRT_MAT_METAL) {                     // metal.rs:12-25
        V3 refl = reflect(in.direction, h.normal);
        out.direction = normalize(refl + m.param * random_point_in_unit_sphere(rng));
        out.origin = h.point;
        att = m.albedo;
        return dot(out.direction, h.normal) > 0.0f;
    } else {                                                   // dielectric.rs:11-60
        float ref_idx = m.param;
        att = v3(1.0f, 1.0f, 1.0f);
        V3 refl = reflect(in.direction, h.normal);
        V3 outward; float ni_over_nt, cosine;
        float a = dot(normalize(in.direction), normalize(h.normal));
        if (a > 0.0f) { outward = -1.0f * h.normal; ni_over_nt = ref_idx; cosine = ref_idx * a; }
        else { outward = h.normal; ni_over_nt = 1.0f / ref_idx; cosine = -a; }
        V3 refr = v3(0, 0, 0);
        float reflect_prob = refract(in.direction, outward, ni_over_nt, refr) ? schlick(cosine, ref_idx) : 1.0f;
        float u[1]; rng.block(u, 1);
        out.origin = h.point;
        out.direction = (u[0] < reflect_prob) ? refl : refr;
        return true;
    }
}

// ------------------------------------------------------------------ lib.rs:43-73
struct Counters { uint64_t rays = 0, nan_rays = 0; };

// Iterative form of the recursion: the product att_1 * (att_2 * (... * leaf)) is evaluated
// innermost-first exactly as the recursion unwinds (lib.rs:62).  `atts` holds at least `depth` entries:
// a path scatters at most `depth` times.
V3 colorize(Ray ray, const Scene& sc, V3 bg, uint32_t depth, PathRng& rng, std::vector<float>& scratch, std::vector<V3>& atts, Counters& cnt) {
    int n_att = 0;
    V3 leaf;
    for (;;) {
        HitInfo h; h.tri = 0;
        cnt.rays++;
        int r = scene_hit(sc, ray, 0.001f, 2000.0f, scratch, h);
        if (r < 0) { cnt.nan_rays++; leaf = v3(0, 0, 0); break; }   // reference panics; we end the path black
        if (r == 1) {
            Ray next{v3(0, 0, 0), v3(0, 0, 0)}; V3 att = v3(0, 0, 0);
            rng.next_bounce();
            if (depth > 0 && scatter(*h.mat, ray, h, rng, att, next)) {
                atts[n_att++] = att; ray = next; depth -= 1;
                continue;
            }
            leaf = v3(0, 0, 0);
            break;
        }
        float t = 0.5f * (ray.direction.y + 1.0f);                   // lib.rs:69-70
        leaf = t * v3(1.0f, 1.0f, 1.0f) + (1.0f - t) * bg;
        break;
    }
    for (int i = n_att - 1; i >= 0; --i) leaf = atts[i] * leaf;
    return leaf;
}

inline uint8_t as_u8(float v) {                                      // Rust `as u8`: saturating, NaN -> 0
    if (!(v == v)) return 0;
    if (v <= 0.0f) return 0;
    if (v >= 255.0f) return 255;
    return (uint8_t)v;
}

thread_local std::string g_err;
int fail(int code, const char* msg) { g_err = msg; return code; }

struct ShardPlan { uint32_t s0, s1; bool tiles; uint32_t rank, count; };

// Pixel ownership under tile sharding: 8x4-pixel tiles, linear tile id t owned by rank t % count.
inline bool owns_pixel(const ShardPlan& sp, uint32_t row, uint32_t col, uint32_t width) {
    if (!sp.tiles) return true;
    uint32_t tiles_x = (width + 7) / 8;
    uint32_t tile = (row / 4) * tiles_x + (col / 8);
    return tile % sp.count == sp.rank;
}

// lib.rs:75-114: threads over image columns (rayon stand-in), rows and samples serial.
int render_sum(const Scene& sc, const rbrt_camera& cam, uint32_t spp, const rbrt_render_opts* o,
               std::vector<V3>& sum /* row-major */, rbrt_stats* stats, unsigned threads_req,
               uint32_t stride_x = 1, uint32_t stride_y = 1) {
    uint32_t W = cam.img_width_pix, H = cam.img_height_pix;
    if (!W || !H || !spp) return fail(RBRT_E_INVALID, "empty image or zero samples");
    uint64_t seed = o ? o->seed : 0;
    uint32_t depth = (o && o->max_depth) ? o->max_depth : 50;
    if (depth > 1024) return fail(RBRT_E_INVALID, "max_depth > 1024");     // the product's limit (render.cu)
    ShardPlan sp{0, spp, false, 0, 1};
    if (o && o->shard_count > 1) {
        if (o->shard_rank >= o->shard_count) return fail(RBRT_E_INVALID, "shard_rank >= shard_count");
        sp.rank = o->shard_rank; sp.count = o->shard_count;
        if (o->shard_mode == RBRT_SHARD_TILES) sp.tiles = true;
        else if (o->shard_mode == RBRT_SHARD_SAMPLES) {
            sp.s0 = (uint32_t)((uint64_t)spp * sp.rank / sp.count);
            sp.s1 = (uint32_t)((uint64_t)spp * (sp.rank + 1) / sp.count);
        }
    }
    sum.assign((size_t)W * H, v3(0, 0, 0));
    unsigned nthreads = threads_req ? threads_req : std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint32_t> next_col{0};
    std::atomic<uint64_t> rays{0}, nans{0}, paths{0};
    auto t0 = std::chrono::steady_clock::now();
    auto worker = [&]() {
        std::vector<float> scratch; std::vector<V3> atts(depth); Counters cnt; uint64_t np = 0;
        V3 bg = v3(0.05f, 0.05f, 0.8f);                              // lib.rs:89-93
        for (;;) {
            uint32_t col = next_col.fetch_add(stride_x);
            if (col >= W) break;
            for (uint32_t row = 0; row < H; row += stride_y) {
                if (!owns_pixel(sp, row, col, W)) continue;
                V3 color = v3(0, 0, 0);
                for (uint32_t s = sp.s0; s < sp.s1; ++s) {
                    PathRng rng{{(uint32_t)seed, (uint32_t)(seed >> 32)}, row * W + col, s, 0, 0};
                    Ray ray = get_ray_through_pixel(cam, row, col, rng);
                    V3 c = colorize(ray, sc, bg, depth, rng, scratch, atts, cnt);
                    color = color + c;                                // lib.rs:99
                    ++np;
                }
                sum[(size_t)row * W + col] = color;
            }
        }
        rays += cnt.rays; nans += cnt.nan_rays; paths += np;
    };
    std::vector<std::thread> pool;
    for (unsigned i = 1; i < nthreads; ++i) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
    double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rays = rays; stats->paths = paths; stats->nan_rays = nans;
        stats->ms_total = ms; stats->ms_device = ms; stats->launches = nthreads;   // launches := threads used
    }
    return RBRT_OK;
}

unsigned g_threads = 0;

}  // namespace

// ====================================================================== C ABI (rbrt_ref_*)
extern "C" {

const char* rbrt_ref_last_error(void) { return g_err.c_str(); }
const char* rbrt_ref_version(void) { return "rbrt oracle (C++/AVX restatement of baurst/rbrt), test infrastructure"; }
int rbrt_ref_set_threads(unsigned n) { g_threads = n; return 0; }
unsigned rbrt_ref_hardware_threads(void) { return std::max(1u, std::thread::hardware_concurrency()); }

int rbrt_ref_camera_new(rbrt_vec3 position, rbrt_vec3 look_at, rbrt_vec3 up, uint32_t h, uint32_t w,
                        float focal, rbrt_camera* out) {
    if (!out) return fail(RBRT_E_INVALID, "null out");
    *out = camera_new(from(position), from(look_at), from(up), h, w, focal);
    return RBRT_OK;
}

int rbrt_ref_transform_vertices(float* xyz, uint64_t n, float scale, rbrt_vec3 rot, rbrt_vec3 tr) {
    for (uint64_t i = 0; i < n; ++i) {                                // mesh.rs:102-112
        V3 p = v3(xyz[3 * i] * scale, xyz[3 * i + 1] * scale, xyz[3 * i + 2] * scale);
        V3 q = rotate_point(p, from(rot)) + from(tr);
        xyz[3 * i] = q.x; xyz[3 * i + 1] = q.y; xyz[3 * i + 2] = q.z;
    }
    return RBRT_OK;
}

int rbrt_ref_scene_create_elements(const rbrt_element_ref* order, uint32_t ne, const rbrt_sphere_desc* spheres, uint32_t ns,
                                   const rbrt_triangle_desc* triangles, uint32_t nt, const rbrt_mesh_desc* meshes, uint32_t nm,
                                   const rbrt_scene_opts* opts, rbrt_scene** out) {
    if (!out || (ne && !order) || (ns && !spheres) || (nt && !triangles) || (nm && !meshes)) return fail(RBRT_E_INVALID, "null argument");
    Scene* sc = new Scene();
    sc->lanes = (opts && opts->simd_lanes) ? opts->simd_lanes : 8;
    if (sc->lanes != 8 && sc->lanes != 4) { delete sc; return fail(RBRT_E_INVALID, "simd_lanes must be 8 or 4"); }
    for (uint32_t i = 0; i < ns; ++i) {
        const auto& s = spheres[i];
        if (s.material.kind > 2) { delete sc; return fail(RBRT_E_INVALID, "unknown material kind"); }
        sc->spheres.push_back(Sphere{from(s.center), s.radius, Material{s.material.kind, from(s.material.albedo), s.material.param}});
    }
    for (uint32_t i = 0; i < nt; ++i) {                                  // BasicTriangle::new (triangle.rs:19-27)
        const auto& t = triangles[i];
        if (t.material.kind > 2) { delete sc; return fail(RBRT_E_INVALID, "unknown material kind"); }
        BasicTri b;
        for (int k = 0; k < 3; ++k) b.corners[k] = from(t.corners[k]);
        b.normal = triangle_normal(b.corners[0], b.corners[1], b.corners[2]);
        b.edges[0] = b.corners[1] - b.corners[0]; b.edges[1] = b.corners[2] - b.corners[0];
        b.mat = Material{t.material.kind, from(t.material.albedo), t.material.param};
        sc->btris.push_back(b);
    }
    for (uint32_t i = 0; i < ne; ++i) {
        if ((order[i].kind == RBRT_ELEM_SPHERE && order[i].index >= ns) || (order[i].kind == RBRT_ELEM_TRIANGLE && order[i].index >= nt) || order[i].kind > 1) {
            delete sc; return fail(RBRT_E_INVALID, "bad element");
        }
        sc->elements.push_back(Element{order[i].kind, order[i].index});
    }
    for (uint32_t i = 0; i < nm; ++i) {
        const auto& m = meshes[i];
        if (m.material.kind > 2) { delete sc; return fail(RBRT_E_INVALID, "unknown material kind"); }
        if (m.num_triangles && !m.tri_vertices) { delete sc; return fail(RBRT_E_INVALID, "null tri_vertices"); }
        sc->meshes.push_back(mesh_new(m.tri_vertices, m.num_triangles, Material{m.material.kind, from(m.material.albedo), m.material.param}, sc->lanes));
    }
    *out = reinterpret_cast<rbrt_scene*>(sc);
    return RBRT_OK;
}

int rbrt_ref_scene_create(const rbrt_sphere_desc* spheres, uint32_t ns, const rbrt_mesh_desc* meshes, uint32_t nm,
                          const rbrt_scene_opts* opts, rbrt_scene** out) {
    std::vector<rbrt_element_ref> order(ns);
    for (uint32_t i = 0; i < ns; ++i) order[i] = rbrt_element_ref{RBRT_ELEM_SPHERE, i};
    return rbrt_ref_scene_create_elements(order.data(), ns, spheres, ns, nullptr, 0, meshes, nm, opts, out);
}
int rbrt_ref_scene_destroy(rbrt_scene* s) { delete reinterpret_cast<Scene*>(s); return RBRT_OK; }

int rbrt_ref_render_hdr(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp,
                        const rbrt_render_opts* opts, float* out, rbrt_stats* stats) {
    if (!scene || !cam || !out) return fail(RBRT_E_INVALID, "null argument");
    std::vector<V3> sum;
    int rc = render_sum(*reinterpret_cast<const Scene*>(scene), *cam, spp, opts, sum, stats, g_threads);
    if (rc) return rc;
    float inv = 1.0f / (float)spp;                                    // lib.rs:101
    for (size_t i = 0; i < sum.size(); ++i) { V3 c = sum[i] * inv; out[3 * i] = c.x; out[3 * i + 1] = c.y; out[3 * i + 2] = c.z; }
    return RBRT_OK;
}

// per-pixel SUM over this shard's samples, W*H*4 f32 (rgb + 0), the multi-rank building block
int rbrt_ref_render_accum(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp,
                          const rbrt_render_opts* opts, float* out_rgba, rbrt_stats* stats) {
    if (!scene || !cam || !out_rgba) return fail(RBRT_E_INVALID, "null argument");
    std::vector<V3> sum;
    int rc = render_sum(*reinterpret_cast<const Scene*>(scene), *cam, spp, opts, sum, stats, g_threads);
    if (rc) return rc;
    for (size_t i = 0; i < sum.size(); ++i) { out_rgba[4 * i] = sum[i].x; out_rgba[4 * i + 1] = sum[i].y; out_rgba[4 * i + 2] = sum[i].z; out_rgba[4 * i + 3] = 0.0f; }
    return RBRT_OK;
}

// CPU-baseline helper for bench.py: the same render restricted to the pixel lattice (row % stride_y == 0,
// col % stride_x == 0) — a bounded, stratified sample of a workload too slow to render in full on the CPU.
// Pixels off the lattice stay zero.  Rays, paths and wall time are returned in stats.
int rbrt_ref_render_subset(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp, const rbrt_render_opts* opts,
                           uint32_t stride_x, uint32_t stride_y, float* out_rgba, rbrt_stats* stats) {
    if (!scene || !cam || !stride_x || !stride_y) return fail(RBRT_E_INVALID, "null argument or zero stride");
    std::vector<V3> sum;
    int rc = render_sum(*reinterpret_cast<const Scene*>(scene), *cam, spp, opts, sum, stats, g_threads, stride_x, stride_y);
    if (rc) return rc;
    if (out_rgba)
        for (size_t i = 0; i < sum.size(); ++i) { out_rgba[4 * i] = sum[i].x; out_rgba[4 * i + 1] = sum[i].y; out_rgba[4 * i + 2] = sum[i].z; out_rgba[4 * i + 3] = 0.0f; }
    return RBRT_OK;
}

// lib.rs:101 + 116-122 applied to a summed accumulation buffer
int rbrt_ref_finalize(const float* accum_rgba, uint32_t W, uint32_t H, uint32_t spp, uint8_t* rgb, float* hdr) {
    float inv = 1.0f / (float)spp;
    for (size_t i = 0; i < (size_t)W * H; ++i) {
        V3 c = v3(accum_rgba[4 * i], accum_rgba[4 * i + 1], accum_rgba[4 * i + 2]) * inv;
        if (hdr) { hdr[3 * i] = c.x; hdr[3 * i + 1] = c.y; hdr[3 * i + 2] = c.z; }
        if (rgb) { rgb[3 * i] = as_u8(sqrtf(c.x) * 256.0f); rgb[3 * i + 1] = as_u8(sqrtf(c.y) * 256.0f); rgb[3 * i + 2] = as_u8(sqrtf(c.z) * 256.0f); }
    }
    return RBRT_OK;
}

int rbrt_ref_render(const rbrt_scene* scene, const rbrt_camera* cam, uint32_t spp,
                    const rbrt_render_opts* opts, uint8_t* rgb, rbrt_stats* stats) {
    if (!scene || !cam || !rgb) return fail(RBRT_E_INVALID, "null argument");
    std::vector<float> acc((size_t)cam->img_width_pix * cam->img_height_pix * 4);
    int rc = rbrt_ref_render_accum(scene, cam, spp, opts, acc.data(), stats);
    if (rc) return rc;
    return rbrt_ref_finalize(acc.data(), cam->img_width_pix, cam->img_height_pix, spp, rgb, nullptr);
}

int rbrt_ref_trace_rays(const rbrt_scene* scene, const rbrt_ray* rays, uint64_t n, uint32_t /*mode*/,
                        rbrt_hit* hits, rbrt_stats* stats) {
    if (!scene || (n && (!rays || !hits))) return fail(RBRT_E_INVALID, "null argument");
    const Scene& sc = *reinterpret_cast<const Scene*>(scene);
    unsigned nthreads = g_threads ? g_threads : std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint64_t> next{0}, nans{0};
    auto t0 = std::chrono::steady_clock::now();
    auto worker = [&]() {
        std::vector<float> scratch;
        for (;;) {
            uint64_t b = next.fetch_add(64);
            if (b >= n) break;
            for (uint64_t i = b; i < std::min(n, b + 64); ++i) {
                Ray r{from(rays[i].origin), from(rays[i].direction)};
                HitInfo h; h.tri = 0;
                int rc = scene_hit(sc, r, 0.001f, 2000.0f, scratch, h);
                rbrt_hit& o = hits[i];
                memset(&o, 0, sizeof(o));
                if (rc == 1) { o.kind = h.kind; o.elem_idx = h.elem; o.tri_idx = h.tri; o.t = h.t; o.dist = h.dist; o.point = to(h.point); o.normal = to(h.normal); }
                else { o.kind = RBRT_HIT_NONE; if (rc < 0) nans++; }
            }
        }
    };
    std::vector<std::thread> pool;
    for (unsigned i = 1; i < nthreads; ++i) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rays = n; stats->nan_rays = nans; stats->launches = nthreads;
        stats->ms_total = stats->ms_device = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return RBRT_OK;
}

int rbrt_ref_primary_rays(const rbrt_camera* cam, uint64_t seed, uint32_t sample, rbrt_ray* out) {
    if (!cam || !out) return fail(RBRT_E_INVALID, "null argument");
    uint32_t W = cam->img_width_pix, H = cam->img_height_pix;
    for (uint32_t row = 0; row < H; ++row)
        for (uint32_t col = 0; col < W; ++col) {
            PathRng rng{{(uint32_t)seed, (uint32_t)(seed >> 32)}, row * W + col, sample, 0, 0};
            Ray r = get_ray_through_pixel(*cam, row, col, rng);
            out[(size_t)row * W + col] = rbrt_ray{to(r.origin), to(r.direction)};
        }
    return RBRT_OK;
}

// ---- known-answer-test hooks: thin wrappers so tests/ can pin each restated function ----
void rbrt_ref_kat_philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { philox4x32_10(ctr, key, out); }
rbrt_vec3 rbrt_ref_kat_reflect(rbrt_vec3 d, rbrt_vec3 n) { return to(reflect(from(d), from(n))); }
int rbrt_ref_kat_refract(rbrt_vec3 d, rbrt_vec3 n, float ni_over_nt, rbrt_vec3* out) {
    V3 o = v3(0, 0, 0); bool ok = refract(from(d), from(n), ni_over_nt, o); *out = to(o); return ok ? 1 : 0;
}
float rbrt_ref_kat_schlick(float cosine, float ref_idx) { return schlick(cosine, ref_idx); }
rbrt_vec3 rbrt_ref_kat_normalize(rbrt_vec3 v) { return to(normalize(from(v))); }
float rbrt_ref_kat_length(rbrt_vec3 v) { return length(from(v)); }
float rbrt_ref_kat_dot(rbrt_vec3 a, rbrt_vec3 b) { return dot(from(a), from(b)); }
rbrt_vec3 rbrt_ref_kat_cross(rbrt_vec3 a, rbrt_vec3 b) { return to(cross(from(a), from(b))); }
rbrt_vec3 rbrt_ref_kat_rotate_point(rbrt_vec3 p, rbrt_vec3 rot) { return to(rotate_point(from(p), from(rot))); }
rbrt_vec3 rbrt_ref_kat_triangle_normal(rbrt_vec3 a, rbrt_vec3 b, rbrt_vec3 c) { return to(triangle_normal(from(a), from(b), from(c))); }
void rbrt_ref_kat_min_max_3d(const float* tris, uint64_t n, rbrt_vec3* lo, rbrt_vec3* hi) {
    V3 l, h; compute_min_max_3d(tris, n, l, h); *lo = to(l); *hi = to(h);
}
int rbrt_ref_kat_bbox_hit(rbrt_vec3 lo, rbrt_vec3 hi, rbrt_ray r) { return bbox_hit(from(lo), from(hi), Ray{from(r.origin), from(r.direction)}) ? 1 : 0; }
int rbrt_ref_kat_sphere(rbrt_vec3 center, float radius, rbrt_ray r, float min_dist, float max_dist, rbrt_hit* out) {
    Sphere s{from(center), radius, Material{0, v3(0, 0, 0), 0}};
    HitInfo h; h.tri = 0;
    int rc = sphere_intersect(s, Ray{from(r.origin), from(r.direction)}, min_dist, max_dist, h);
    memset(out, 0, sizeof(*out));
    if (rc == 1) { out->kind = RBRT_HIT_SPHERE; out->t = h.t; out->dist = h.dist; out->point = to(h.point); out->normal = to(h.normal); }
    else out->kind = RBRT_HIT_NONE;
    return rc;
}
void rbrt_ref_kat_avx_dot(const float* a /*3x8*/, const float* b /*3x8*/, float* out /*8*/) {
    _mm256_storeu_ps(out, avx_dot(_mm256_loadu_ps(a), _mm256_loadu_ps(a + 8), _mm256_loadu_ps(a + 16),
                                  _mm256_loadu_ps(b), _mm256_loadu_ps(b + 8), _mm256_loadu_ps(b + 16)));
}
void rbrt_ref_kat_avx_cross(const float* a, const float* b, float* out /*3x8*/) {
    __m256 x, y, z;
    avx_cross(_mm256_loadu_ps(a), _mm256_loadu_ps(a + 8), _mm256_loadu_ps(a + 16),
              _mm256_loadu_ps(b), _mm256_loadu_ps(b + 8), _mm256_loadu_ps(b + 16), x, y, z);
    _mm256_storeu_ps(out, x); _mm256_storeu_ps(out + 8, y); _mm256_storeu_ps(out + 16, z);
}
void rbrt_ref_kat_sse_dot(const float* a /*3x4*/, const float* b, float* out /*4*/) {
    _mm_storeu_ps(out, sse_dot(_mm_loadu_ps(a), _mm_loadu_ps(a + 4), _mm_loadu_ps(a + 8),
                               _mm_loadu_ps(b), _mm_loadu_ps(b + 4), _mm_loadu_ps(b + 8)));
}
void rbrt_ref_kat_sse_cross(const float* a, const float* b, float* out /*3x4*/) {
    __m128 x, y, z;
    sse_cross(_mm_loadu_ps(a), _mm_loadu_ps(a + 4), _mm_loadu_ps(a + 8),
              _mm_loadu_ps(b), _mm_loadu_ps(b + 4), _mm_loadu_ps(b + 8), x, y, z);
    _mm_storeu_ps(out, x); _mm_storeu_ps(out + 4, y); _mm_storeu_ps(out + 8, z);
}
// one scatter step with an explicit RNG position, for material KATs / GPU-vs-oracle checks
int rbrt_ref_kat_scatter(rbrt_material mat, rbrt_ray in, rbrt_vec3 point, rbrt_vec3 normal, uint64_t seed,
                         uint32_t pixel, uint32_t sample, uint32_t bounce, rbrt_vec3* att, rbrt_ray* out) {
    Material m{mat.kind, from(mat.albedo), mat.param};
    HitInfo h; h.point = from(point); h.normal = from(normal); h.mat = &m; h.dist = 0; h.tri = 0;
    PathRng rng{{(uint32_t)seed, (uint32_t)(seed >> 32)}, pixel, sample, bounce, 0};
    V3 a = v3(0, 0, 0); Ray o{v3(0, 0, 0), v3(0, 0, 0)};
    bool ok = scatter(m, Ray{from(in.origin), from(in.direction)}, h, rng, a, o);
    *att = to(a); out->origin = to(o.origin); out->direction = to(o.direction);
    return ok ? 1 : 0;
}
uint8_t rbrt_ref_kat_as_u8(float v) { return as_u8(v); }

}  // extern "C"
