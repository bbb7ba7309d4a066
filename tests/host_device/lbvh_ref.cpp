// lbvh_ref.cpp — a host restatement of the creation-time LBVH builder (rbrt_b200/csrc/bvh_build.cu), written from the algorithm and
// its formulas, sharing no code with the device file.  Built with g++ -ffp-contract=off: every float op is one IEEE-rounded op, as the
// device code (built with -fmad=false, IEEE division and sqrt, no FTZ) computes it.  Min and max are order-independent and every binary
// node is refit or rotated once, after its subtrees are final, so the device's tree is reproduced bit for bit; only the slot numbers
// the collapse hands out with atomicAdd differ, and this builder numbers the 4-wide nodes in breadth-first order (node j's internal
// children appended in slot order).
//
// Steps: exact AABB over all n_all triangles (NaN ignored) -> padding, grid and qstep -> 63-bit Morton keys of the triangle-box
// centres -> stable sort -> Karras 2012 radix tree (equal keys split by 64 + clz(i ^ j)) -> bottom-up boxes, with one pass of Kensler
// rotations where leaf_size == 1 and sah is set, at nodes whose (unrotated) range covers >= 16 triangles -> greedy collapse into 4-wide
// nodes (the internal child of largest half-area first, strict >; subtrees of <= leaf_size triangles are leaves) -> child boxes
// quantised outward, one step of margin, onto the 16-bit grid.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

const float QSTEP_MAX = 2.0e6f;            // RBRT_QSTEP_MAX (common.cuh)
const uint32_t STACK = 192;                // RBRT_STACK: a tree is refused when 3 * depth + 2 exceeds it
const int ROT_MIN = 16;                    // a node is rotated when it covers at least this many triangles

float bits2f(uint32_t b) { float f; std::memcpy(&f, &b, 4); return f; }
uint32_t f2bits(float f) { uint32_t b; std::memcpy(&b, &f, 4); return b; }
int32_t f2ord(float f) { int32_t i = (int32_t)f2bits(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
float ord2f(int32_t i) { return bits2f((uint32_t)(i >= 0 ? i : i ^ 0x7FFFFFFF)); }
// CUDA's fminf / fmaxf: a NaN operand is ignored unless both are NaN
float mn(float a, float b) { return std::isnan(a) ? b : std::isnan(b) ? a : (a < b ? a : b); }
float mx(float a, float b) { return std::isnan(a) ? b : std::isnan(b) ? a : (a > b ? a : b); }

uint64_t spread21(uint32_t v) {            // bit k of v -> bit 3k
    uint64_t r = 0;
    for (int k = 0; k < 21; ++k) r |= (uint64_t)((v >> k) & 1u) << (3 * k);
    return r;
}

struct Box { float lo[3], hi[3]; };
Box merge(const Box& a, const Box& b) {
    Box m;
    for (int k = 0; k < 3; ++k) { m.lo[k] = mn(a.lo[k], b.lo[k]); m.hi[k] = mx(a.hi[k], b.hi[k]); }
    return m;
}
float area(const Box& b) {                 // dx * dy + dy * dz + dz * dx, left to right
    const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    const float s = dx * dy + dy * dz;
    return s + dz * dx;
}

int delta(const std::vector<uint64_t>& key, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    if (key[i] == key[j]) { uint32_t x = (uint32_t)(i ^ j); return 64 + (x ? __builtin_clz(x) : 32); }
    return __builtin_clzll(key[i] ^ key[j]);
}

// child reference: >= 0 internal node, < 0 ~leaf position (as the device's build arrays)
void karras(const std::vector<uint64_t>& key, int n, int32_t* children, int32_t* range) {
    for (int i = 0; i < n - 1; ++i) {
        const int d = delta(key, n, i, i + 1) - delta(key, n, i, i - 1) >= 0 ? 1 : -1;
        const int dmin = delta(key, n, i, i - d);
        int lmax = 2;
        while (delta(key, n, i, i + lmax * d) > dmin) lmax *= 2;
        int l = 0;
        for (int t = lmax / 2; t >= 1; t /= 2)
            if (delta(key, n, i, i + (l + t) * d) > dmin) l += t;
        const int j = i + l * d;
        const int dnode = delta(key, n, i, j);
        int s = 0, t = l;
        do {                               // the split: the last position sharing more than dnode bits with i
            t = (t + 1) / 2;
            if (delta(key, n, i, i + (s + t) * d) > dnode) s += t;
        } while (t > 1);
        const int gamma = i + s * d + std::min(d, 0);
        const int first = std::min(i, j), last = std::max(i, j);
        children[2 * i] = first == gamma ? ~gamma : gamma;
        children[2 * i + 1] = last == gamma + 1 ? ~(gamma + 1) : gamma + 1;
        range[2 * i] = first; range[2 * i + 1] = last;
    }
}

uint32_t qlo(float v, float org, float step) {
    float q = std::floor((v - org) / step) - 1.0f;
    while (q > 0.0f && std::fmaf(q, step, org) > v) q -= 1.0f;
    return (uint32_t)mn(mx(q, 0.0f), 65535.0f);
}
uint32_t qhi(float v, float org, float step) {
    float q = std::ceil((v - org) / step) + 1.0f;
    while (q < 65535.0f && std::fmaf(q, step, org) < v) q += 1.0f;
    return (uint32_t)mn(mx(q, 0.0f), 65535.0f);
}
uint32_t leaf_ref(uint32_t first, uint32_t count) { return ~((first << 3) | (count - 1)); }

}  // namespace

extern "C" {

// The Karras topology alone (children / range: 2 x (n - 1) int32 each), for hand-derived checks.
void lbvh_ref_karras(const uint64_t* keys, int n, int32_t* children, int32_t* range) {
    std::vector<uint64_t> k(keys, keys + n);
    karras(k, n, children, range);
}

// One mesh.  raw: n_all x 9 floats.  Outputs:
//   grid[13]   lo[3] hi[3] qorg[3] qstep[3] pad  (the MeshDev fields and the padding; qorg / qstep are 0 when n == 0)
//   step_org[6] the grid's step[3] and org[3] (BuildParams.grid: step is not replaced by NaN)
//   perm[n]    sorted position -> original triangle
//   tris[12n]  {v0, orig bits} {e1, 0} {e2, 0}
//   normals[4n] unit normals, original order
//   nodes[16 * max(n - 1, 1)] 4-wide nodes, breadth-first
//   res[4]     live_nodes, depth, error, number of 4-wide nodes written (tail)
//   widths[cap_levels] nodes per level; returns the number of levels (may exceed cap_levels; only cap_levels are written)
int lbvh_ref_build(const float* raw, uint64_t n_all, uint32_t n, float pad_rel, uint32_t leaf_size, int sah, float* grid, float* step_org,
                   uint32_t* perm, float* tris, float* normals, uint32_t* nodes, uint32_t* res, uint32_t* widths, int cap_levels) {
    // ---- exact AABB over every coordinate of all n_all triangles, starting from +-FLT_MAX
    int32_t omin[3], omax[3];
    for (int k = 0; k < 3; ++k) { omin[k] = f2ord(3.40282347e+38f); omax[k] = f2ord(-3.40282347e+38f); }
    for (uint64_t v = 0; v < 3 * n_all; ++v)
        for (int k = 0; k < 3; ++k) {
            const float x = raw[3 * v + k];
            if (std::isnan(x)) continue;
            omin[k] = std::min(omin[k], f2ord(x)); omax[k] = std::max(omax[k], f2ord(x));
        }
    float lo[3], hi[3], m = 0.0f;
    for (int k = 0; k < 3; ++k) {
        lo[k] = ord2f(omin[k]); hi[k] = ord2f(omax[k]);
        m = mx(m, mx(std::fabs(lo[k]), std::fabs(hi[k])));
        m = mx(m, hi[k] - lo[k]);
    }
    // ---- padding (relative, with a floor of 2^-21 * (mx + 1000)), the 16-bit grid with 8 steps of slack, qstep
    const float pad = pad_rel > 0.0f ? mx(pad_rel * m, 4.7683716e-7f * (m + 1000.0f)) : 0.0f;
    float step[3], org[3], inv_ext[3];
    for (int k = 0; k < 3; ++k) {
        const float ext = (hi[k] + pad) - (lo[k] - pad);
        float s = ext / 65500.0f;
        if (!(s > 1e-30f)) s = 1e-30f;
        step[k] = s; org[k] = (lo[k] - pad) - 8.0f * s;
        inv_ext[k] = hi[k] > lo[k] ? 1.0f / (hi[k] - lo[k]) : 0.0f;
        grid[k] = lo[k]; grid[3 + k] = hi[k];
        grid[6 + k] = n ? org[k] : 0.0f;
        grid[9 + k] = n ? (s <= QSTEP_MAX ? s : bits2f(0x7FFFFFFFu)) : 0.0f;
        step_org[k] = s; step_org[3 + k] = org[k];
    }
    grid[12] = pad;
    for (int k = 0; k < 4; ++k) res[k] = 0;
    if (!n) return 0;
    // ---- normals and Morton keys
    std::vector<uint64_t> key(n);
    for (uint32_t i = 0; i < n; ++i) {
        const float* t = raw + 9 * (size_t)i;
        float e1[3], e2[3], c[3];
        for (int k = 0; k < 3; ++k) { e1[k] = t[3 + k] - t[k]; e2[k] = t[6 + k] - t[k]; }
        c[0] = e1[1] * e2[2] - e1[2] * e2[1];
        c[1] = e1[2] * e2[0] - e1[0] * e2[2];
        c[2] = e1[0] * e2[1] - e1[1] * e2[0];
        const float l = std::sqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
        for (int k = 0; k < 3; ++k) normals[4 * (size_t)i + k] = c[k] / l;
        normals[4 * (size_t)i + 3] = 0.0f;
        uint32_t q[3];
        for (int k = 0; k < 3; ++k) {
            const float cen = 0.5f * (mn(t[k], mn(t[3 + k], t[6 + k])) + mx(t[k], mx(t[3 + k], t[6 + k])));
            const float f = mn(mx((cen - lo[k]) * inv_ext[k], 0.0f), 1.0f);
            q[k] = std::min((uint32_t)(f * 2097152.0f), 2097151u);
        }
        key[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    }
    // ---- stable sort by key
    for (uint32_t i = 0; i < n; ++i) perm[i] = i;
    std::stable_sort(perm, perm + n, [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
    std::vector<uint64_t> skey(n);
    std::vector<Box> leaf(n);
    for (uint32_t p = 0; p < n; ++p) {
        const uint32_t o = perm[p];
        skey[p] = key[o];
        const float* t = raw + 9 * (size_t)o;
        for (int k = 0; k < 3; ++k) {
            tris[12 * (size_t)p + k] = t[k];
            tris[12 * (size_t)p + 4 + k] = t[3 + k] - t[k];
            tris[12 * (size_t)p + 8 + k] = t[6 + k] - t[k];
            leaf[p].lo[k] = mn(t[k], mn(t[3 + k], t[6 + k])) - pad;
            leaf[p].hi[k] = mx(t[k], mx(t[3 + k], t[6 + k])) + pad;
        }
        tris[12 * (size_t)p + 3] = bits2f(o);
        tris[12 * (size_t)p + 7] = 0.0f;
        tris[12 * (size_t)p + 11] = 0.0f;
    }
    if (n <= leaf_size || n == 1) return 0;           // the whole mesh is one leaf: no nodes
    // ---- radix tree
    const int ni = (int)n - 1;
    std::vector<int32_t> ch(2 * (size_t)ni), rg(2 * (size_t)ni), par(ni, -1), parl(n, -1);
    karras(skey, (int)n, ch.data(), rg.data());
    for (int i = 0; i < ni; ++i)
        for (int s = 0; s < 2; ++s) { const int c = ch[2 * i + s]; if (c >= 0) par[c] = i; else parl[~c] = i; }
    // ---- bottom-up boxes (+ rotations): leaves in order, the second arrival at a node handles it; any order in which a node
    // comes after both of its subtrees gives the same tree
    std::vector<Box> nb(ni);
    std::vector<uint8_t> seen(ni, 0);
    const bool rot = sah && leaf_size == 1;
    auto box_of = [&](int c) -> Box { return c >= 0 ? nb[c] : leaf[~c]; };
    for (uint32_t p = 0; p < n; ++p) {
        for (int cur = parl[p]; cur >= 0; cur = par[cur]) {
            if (!seen[cur]++) break;
            int c0 = ch[2 * cur], c1 = ch[2 * cur + 1];
            Box b0 = box_of(c0), b1 = box_of(c1);
            if (rot && rg[2 * cur + 1] - rg[2 * cur] + 1 >= ROT_MIN) {
                float best = 0.0f; int bside = -1, bwhich = 0; Box bnew = b0;
                for (int side = 0; side < 2; ++side) {         // X: the child rebuilt, Y: the other child, moved down into X
                    const int X = side ? c1 : c0;
                    if (X < 0) continue;
                    const Box& bx = side ? b1 : b0; const Box& by = side ? b0 : b1;
                    const Box g0 = box_of(ch[2 * X]), g1 = box_of(ch[2 * X + 1]);
                    const float ax = area(bx);
                    const Box m0 = merge(by, g1), m1 = merge(g0, by);   // Y takes g0's place / g1's place
                    const float d0 = area(m0) - ax, d1 = area(m1) - ax;
                    if (d0 < best) { best = d0; bside = side; bwhich = 0; bnew = m0; }
                    if (d1 < best) { best = d1; bside = side; bwhich = 1; bnew = m1; }
                }
                if (bside >= 0) {
                    const int X = bside ? c1 : c0, Y = bside ? c0 : c1;
                    const int up = ch[2 * X + bwhich];
                    ch[2 * X + bwhich] = Y;
                    nb[X] = bnew;
                    const Box bup = box_of(up);
                    if (bside) { c0 = up; b0 = bup; b1 = bnew; } else { c1 = up; b1 = bup; b0 = bnew; }
                    ch[2 * cur] = c0; ch[2 * cur + 1] = c1;
                    if (Y >= 0) par[Y] = X; else parl[~Y] = X;
                    if (up >= 0) par[up] = cur; else parl[~up] = cur;
                }
            }
            nb[cur] = merge(b0, b1);
        }
    }
    // ---- collapse into 4-wide nodes, breadth-first
    std::vector<int32_t> queue(1, 0);
    size_t begin = 0;
    int levels = 0;
    while (begin < queue.size()) {
        const size_t end = queue.size();
        if (levels < cap_levels) widths[levels] = (uint32_t)(end - begin);
        ++levels;
        for (size_t j = begin; j < end; ++j) {
            int src[4]; int64_t ref[4]; int nc = 2;           // ref >= 0: internal (expandable), < 0: a leaf (its 32-bit ref)
            auto eff = [&](int c, int k) {
                src[k] = c;
                if (c < 0) { ref[k] = -1 - (int64_t)leaf_ref((uint32_t)~c, 1); return; }
                const uint32_t cnt = (uint32_t)(rg[2 * c + 1] - rg[2 * c] + 1);
                ref[k] = cnt <= leaf_size ? -1 - (int64_t)leaf_ref((uint32_t)rg[2 * c], cnt) : c;
            };
            const int i = queue[j];
            eff(ch[2 * i], 0); eff(ch[2 * i + 1], 1);
            for (int round = 0; round < 2; ++round) {
                int best = -1; float best_a = -1.0f;
                for (int k = 0; k < nc; ++k)
                    if (ref[k] >= 0) { const float a = area(nb[src[k]]); if (a > best_a) { best_a = a; best = k; } }
                if (best < 0) break;
                const int c = src[best];
                eff(ch[2 * c], best); eff(ch[2 * c + 1], nc); ++nc;
            }
            uint32_t* w = nodes + 16 * j;
            for (int k = 0; k < 4; ++k) {
                if (k < nc) {
                    const Box b = box_of(src[k]);
                    for (int a = 0; a < 3; ++a) w[3 * k + a] = qlo(b.lo[a], org[a], step[a]) | (qhi(b.hi[a], org[a], step[a]) << 16);
                    if (ref[k] >= 0) { w[12 + k] = (uint32_t)queue.size(); queue.push_back(src[k]); }
                    else w[12 + k] = (uint32_t)(-1 - ref[k]);
                } else {
                    w[3 * k] = w[3 * k + 1] = w[3 * k + 2] = 0x0000FFFFu;
                    w[12 + k] = leaf_ref(0, 1);
                }
            }
        }
        begin = end;
    }
    const bool bad = 3u * (uint32_t)levels + 2u > STACK;
    res[0] = bad ? 0u : (uint32_t)queue.size(); res[1] = (uint32_t)levels; res[2] = bad ? 1u : 0u; res[3] = (uint32_t)queue.size();
    return levels;
}

}  // extern "C"
