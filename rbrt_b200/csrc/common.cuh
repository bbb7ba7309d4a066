// common.cuh — device-side data layout, exact-rounding f32 vector algebra and Philox RNG.
//
// Parity rule (SURVEY.md Q5): the reference never contracts a*b+c into an FMA (Rust/LLVM does
// not, and vec3_avx.rs:18-21,40-42 uses separate mul/add/sub intrinsics).  Everything that
// reproduces reference arithmetic therefore goes through __fmul_rn/__fadd_rn/__fsub_rn/
// __fdiv_rn/__fsqrt_rn, which ptxas never fuses, independent of -fmad.  FMAs appear only in the
// BVH slab tests, which prune conservatively and never produce a reported value.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rbrt {

// ------------------------------------------------------------------ exact f32 algebra (vec3.rs)
struct f3 { float x, y, z; };
__host__ __device__ __forceinline__ f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }

#ifdef __CUDA_ARCH__
#define XMUL(a, b) __fmul_rn((a), (b))
#define XADD(a, b) __fadd_rn((a), (b))
#define XSUB(a, b) __fsub_rn((a), (b))
#define XDIV(a, b) __fdiv_rn((a), (b))
#define XSQRT(a) __fsqrt_rn((a))
#else
#define XMUL(a, b) ((a) * (b))
#define XADD(a, b) ((a) + (b))
#define XSUB(a, b) ((a) - (b))
#define XDIV(a, b) ((a) / (b))
#define XSQRT(a) sqrtf((a))
#endif

__device__ __forceinline__ f3 operator-(f3 a, f3 b) { return mk3(XSUB(a.x, b.x), XSUB(a.y, b.y), XSUB(a.z, b.z)); }  // vec3.rs:12-22
__device__ __forceinline__ f3 operator+(f3 a, f3 b) { return mk3(XADD(a.x, b.x), XADD(a.y, b.y), XADD(a.z, b.z)); }  // vec3.rs:23-34
__device__ __forceinline__ f3 operator*(f3 a, f3 b) { return mk3(XMUL(a.x, b.x), XMUL(a.y, b.y), XMUL(a.z, b.z)); }  // vec3.rs:57-67
__device__ __forceinline__ f3 operator*(float s, f3 a) { return mk3(XMUL(s, a.x), XMUL(s, a.y), XMUL(s, a.z)); }     // vec3.rs:68-78
__device__ __forceinline__ f3 operator*(f3 a, float s) { return mk3(XMUL(a.x, s), XMUL(a.y, s), XMUL(a.z, s)); }     // vec3.rs:80-90
// dot = (x*x' + y*y') + z*z'  (vec3.rs:115-117,157-159 and vec3_avx.rs:18-21)
__device__ __forceinline__ float dot3(f3 a, f3 b) { return XADD(XADD(XMUL(a.x, b.x), XMUL(a.y, b.y)), XMUL(a.z, b.z)); }
// length = sqrt((x*x + y*y) + z*z)  (vec3.rs:111-113)
__device__ __forceinline__ float len3(f3 a) { return XSQRT(XADD(XADD(XMUL(a.x, a.x), XMUL(a.y, a.y)), XMUL(a.z, a.z))); }
// normalize = three true divisions by the length (vec3.rs:119-126)
__device__ __forceinline__ f3 norm3(f3 a) { float l = len3(a); return mk3(XDIV(a.x, l), XDIV(a.y, l), XDIV(a.z, l)); }
// cross = (ay*bz - az*by, az*bx - ax*bz, ax*by - ay*bx), mul,mul,sub (vec3.rs:128-134, vec3_avx.rs:40-42)
__device__ __forceinline__ f3 cross3(f3 a, f3 b) {
    return mk3(XSUB(XMUL(a.y, b.z), XMUL(a.z, b.y)), XSUB(XMUL(a.z, b.x), XMUL(a.x, b.z)), XSUB(XMUL(a.x, b.y), XMUL(a.y, b.x)));
}

// ------------------------------------------------------------------ Philox4x32-10 (counter-based RNG)
// key = seed; counter = (pixel, sample, bounce, round).  One block per request site: camera
// jitter (2 words), one rejection round of random_point_in_unit_sphere (3), dielectric coin (1).
struct u4 { uint32_t x, y, z, w; };
__host__ __device__ __forceinline__ u4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
#endif
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3; return o;
}
// rand 0.8 `Standard` for f32: 24 random bits, [0,1)
__host__ __device__ __forceinline__ float u32_to_unit_f32(uint32_t u) { return (float)(u >> 8) * (1.0f / 16777216.0f); }

// ------------------------------------------------------------------ device scene layout (HBM)
// All arrays are 16-byte aligned float4 / uint records (north_star (1): flattened SoA buffers).
struct MeshDev {
    float lo[3], hi[3];        // exact mesh AABB (aabbox.rs:62-88), used by the reference's slab pre-test
    uint32_t tri_base;         // first triangle record of this mesh in SceneDev::tris (BVH order)
    uint32_t n_tris;           // N_eff triangles the reference actually tests (tail rule, mesh.rs:136-144)
    uint32_t node_base;        // first BVH node of this mesh in SceneDev::nodes
    int32_t  root_ref;         // >=0 node index (relative to node_base), <0 leaf reference
    uint32_t nrm_base;         // first normal of this mesh in SceneDev::normals (original order)
    uint32_t elem;             // element id = num_spheres + mesh index (material lookup)
    float qorg[3], qstep[3];   // 16-bit grid of this mesh's BVH node boxes: bound = qorg + q * qstep (bvh_build.cu); qstep NaN: see below
};

// Largest grid step the slab test of intersect.cuh (ray_slabs / bvh4_step) evaluates without overflow.  It forms -2^23 * qstep * (1/d) with
// |1/d| up to its clamp of 1e25 (a direction component of 0 or |d| <= 1e-25), and the node decode adds (2^23 + q) * qstep / d to that.
// Above ~4.05e6 (a padded extent of ~2.65e11 on the axis) the product overflows to inf, every t of the axis becomes -inf or +inf and the
// traversal rejects boxes the ray is inside: hits were lost.  2e6 keeps 2^23 * 2e6 * 1e25 = 1.68e38 below half of FLT_MAX, so nothing
// overflows for an origin anywhere in the grid.  On an axis whose step is larger (or inf / NaN), the mesh set-up stores qstep = NaN: every
// slab t of that axis is NaN, fminf / fmaxf ignore it, and the traversal culls on the other axes only (on none: every box is entered).
#define RBRT_QSTEP_MAX 2.0e6f

struct SceneDev {
    const float4* spheres;     // per ELEMENT of Scene.elements, in order: sphere {cx, cy, cz, r}; BasicTriangle {bits(index into etris), 0, 0, 0}
    const float4* etris;       // BasicTriangle elements: 4 x float4 {v0}, {e1}, {e2}, {unit normal} (triangle.rs:9-28)
    const uint32_t* elem_kind; // per element: RBRT_ELEM_*; only read when n_etris > 0
    const float4* tris;        // 3 x float4 per triangle: {v0.xyz, bits(orig idx)}, {e1.xyz, 0}, {e2.xyz, 0}
    const float4* nodes;       // 4 x 16 B per 4-wide BVH node: child boxes on the mesh's 16-bit grid + 4 child refs (intersect.cuh)
    const float4* normals;     // {n.xyz, 0} per triangle, original order
    const float4* mat;         // per element: {albedo.xyz, param}
    const uint32_t* mat_kind;  // per element: RBRT_MAT_*
    const MeshDev* meshes;
    uint32_t n_spheres, n_meshes;   // n_spheres = number of ELEMENTS (spheres + basic triangles)
    uint32_t n_etris;
};

#define RBRT_STACK 192            // traversal stack entries per lane: <= 3 per level of the 4-wide tree + sentinel (checked by the builder)

// leaf reference encoding: ~((first << 3) | (count - 1)), count in 1..8
__host__ __device__ __forceinline__ int32_t make_leaf_ref(uint32_t first, uint32_t count) { return ~(int32_t)((first << 3) | (count - 1)); }

// Camera as the kernels need it (subset of rbrt_camera, cam.rs:4-19)
struct CamDev {
    float pos[3], right[3], up[3], center[3];
    float mm_per_pix_hor, mm_per_pix_vert;
    uint32_t width, height;
};

// Division by a launch-invariant 32-bit divisor (Granlund-Montgomery round-up form, exact for every 32-bit dividend):
// the pixel mapping divides twice per path and bounce, and a run-time `/` is ~20 instructions.
struct FastDiv { uint32_t m, s1, s2; };
inline FastDiv make_fastdiv(uint32_t d) {
    uint32_t l = 0; while ((1ull << l) < d) ++l;                            // ceil(log2 d)
    FastDiv f;
    f.m = (uint32_t)((((1ull << 32) * ((1ull << l) - d)) / d) + 1);
    f.s1 = l < 1 ? l : 1; f.s2 = l - f.s1;
    return f;
}
__device__ __forceinline__ uint32_t fast_div(uint32_t n, FastDiv f) {
    const uint32_t t = __umulhi(f.m, n);
    return (t + ((n - t) >> f.s1)) >> f.s2;
}

// Pixel enumeration of one rank's shard: 8x4-pixel tiles (one warp = one tile), linear tile id
// T = tj * shard_count + shard_rank, row-major over ceil(W/8) x ceil(H/4) tiles.
struct ShardDev {
    uint32_t rank, count;      // tile striping (1 rank: 0,1)
    uint32_t tiles_x, tiles_total, tiles_mine;
    FastDiv fd_tiles_x;        // division by tiles_x
    uint32_t s0, s1;           // sample range rendered by this rank
};

__device__ __forceinline__ bool shard_pixel(const ShardDev& sh, const CamDev& cam, uint32_t j, uint32_t& row, uint32_t& col) {
    uint32_t tj = j >> 5, lane = j & 31;
    uint32_t T = tj * sh.count + sh.rank;
    if (T >= sh.tiles_total) return false;
    uint32_t ty = fast_div(T, sh.fd_tiles_x), tx = T - ty * sh.tiles_x;
    col = tx * 8 + (lane & 7);
    row = ty * 4 + (lane >> 3);
    return col < cam.width && row < cam.height;
}

}  // namespace rbrt
