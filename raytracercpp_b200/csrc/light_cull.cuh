// light_cull.cuh -- per-light masks of the shadow packets (kernels.cuh: packet_trace<true, ...>, SceneView::tri_occ / blk_occ).
//
// tri_test is the reference's Moeller-Trumbore with back-face culling (triangle.cpp:37-40): it accepts a triangle only when
// dot(n, -d) > 0, i.e. when the ray crosses the triangle's plane from the front side to the back side.  Every shadow ray of a
// frame aims at one point light L.  When L lies strictly on the front side of a triangle's plane, a ray that crosses that
// plane before it reaches L crosses it towards the front side and is rejected: the triangle can never occlude, and a subtree
// that holds only such triangles can be skipped without changing any answer.
//
// The rule, per triangle (a, b, c, cached un-normalised normal n; |n|_1 = |n.x| + |n.y| + |n.z| >= |n|):
//     prune  iff  n . (L - v) > margin  for v = a, b and c,   margin = |n|_1 * (2.5e-4 + 2^-16 * (max_v |v|_1 + |L|_1 + span))
// written with '>' so that NaN and degenerate triangles are kept.  Derivation: the shadow ray of a hit point p starts at
// o = p + 1e-4 nrm (nrm the normalised shading normal, renderer.cpp:344) and has the direction d of L - p, so it passes
// |delta| = 1e-4 off L.  With h = n . (L - a) the plane function g(t) = n . (o + t d - a) is >= h - |n| |delta| at t_L = |L - p|.
// A front-facing crossing has n . d < 0, |n . d| <= |n|, so it lies at t >= t_L + (h - |n| |delta|) / |n|, and then
// |p - q| >= t - |delta| >= t_L = |p - L| as soon as h >= 2 |n| |delta|: the reference's distance test (renderer.cpp:354)
// rejects the hit.  The absolute term 2.5e-4 covers 2 |delta| with 25 % to spare.  The relative term covers the rounding of
// tri_test's det, plane distance and t, of the hit point and of the distance test, and of the mask's own dot products: a few
// ulps of |n| times the lengths involved, |v|, |L|, |L - v| <= span and the ray length t_L <= span (2^-16 = 256 ulps).  A
// near-parallel ray whose det rounds to > 0 although n . d >= 0 has det within a few ulps of |n|; its t = n . (o - a) / det
// is then far beyond t_L and fails the distance test as well.  span bounds every shadow ray: 1.01 x the largest distance from
// L to a corner of the root box or of an analytic sphere's box, + 1e-3 (hit points lie in those boxes up to rounding).  A
// scene with an analytic plane has unbounded hit points: its masks have every bit set.  tests/test_light_cull.py restates
// tri_test and the rule in float32 and checks that no pruned triangle is ever accepted.
//
// The masks are built over the array the packets traverse (wrecs[], or recs[] with RT_OPT_LEAF_SPLIT 0):
//   tri_occ[]  one bit per triangle in tris[] order: the triangle may occlude (k_lc_tris);
//   blk_occ[]  one byte per child block; blocks start at even record indices (k_ob_place, build_wide_tree: the root's block at
//              2), so byte link >> 1 belongs to the block at `link` alone; bit k = child record k's subtree holds a triangle
//              that may occlude.  Byte 0 (no block starts at record 0 or 1) holds the root's own bit.
// Bottom-up without the builders' level lists: every record learns its parent (k_lc_parents), then every leaf with a
// triangle that may occlude sets its bit and walks up setting its ancestors' bits (k_lc_leaves); a walk stops at the first bit
// that was already set, because whoever set it walks on from there.  Each record's bit is set once.
#pragma once

#include "rt_device.h"

namespace rtb {
namespace lightcull {

constexpr float kAbsMargin = 2.5e-4f;
constexpr float kRelMargin = 1.52587890625e-5f;      // 2^-16

__device__ __forceinline__ float norm1(V3 v) { return fabsf(v.x) + fabsf(v.y) + fabsf(v.z); }

// false only when the light is strictly in front of the triangle by more than the margin (the rule above)
__device__ __forceinline__ bool may_occlude(float4 p0, float4 p1, float4 p2, V3 L, float span)
{
    const V3 a = v3(p0.x, p0.y, p0.z), b = v3(p1.x, p1.y, p1.z), c = v3(p2.x, p2.y, p2.z);
    const V3 n = v3(p0.w, p1.w, p2.w);
    const float ha = dot(n, L - a), hb = dot(n, L - b), hc = dot(n, L - c);
    const float ext = fmaxf(norm1(a), fmaxf(norm1(b), norm1(c))) + norm1(L) + span;
    const float margin = norm1(n) * (kAbsMargin + kRelMargin * ext);
    return !(ha > margin && hb > margin && hc > margin);
}

// one warp per 32 consecutive triangles, one word each; words beyond the triangles are 0
__global__ void __launch_bounds__(256)
k_lc_tris(const float4* tris, uint32_t n, uint32_t n_words, V3 L, float span, uint32_t* tri_occ)
{
    const uint64_t total = 32ull * n_words;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        bool may = false;
        if (i < n) may = may_occlude(tris[3 * i], tris[3 * i + 1], tris[3 * i + 2], L, span);
        const uint32_t w = __ballot_sync(0xffffffffu, may);
        if ((threadIdx.x & 31u) == 0u) tri_occ[i >> 5] = w;
    }
}

__device__ __forceinline__ bool lc_interior(uint32_t meta) { return !(meta & RT_LEAF_BIT) && (meta & RT_META_COUNT_MASK) != 0u; }

__global__ void __launch_bounds__(256)
k_lc_parents(const float4* recs, uint32_t n_recs, uint32_t* parent)
{
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_recs; r += gridDim.x * blockDim.x) {
        const float4 q3 = recs[4 * (size_t)r + 3];
        const uint32_t link = __float_as_uint(q3.z), meta = __float_as_uint(q3.w);
        if (!lc_interior(meta)) continue;
        for (uint32_t k = 0; k < (meta & RT_META_COUNT_MASK); k++) parent[link + k] = r;
    }
}

// blk_words: blk_occ as 32-bit words (zeroed before), so that bits can be set with atomicOr
__global__ void __launch_bounds__(256)
k_lc_leaves(const float4* recs, uint32_t n_recs, const uint32_t* parent, const uint32_t* tri_occ, uint32_t* blk_words)
{
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_recs; r += gridDim.x * blockDim.x) {
        const float4 q3 = recs[4 * (size_t)r + 3];
        const uint32_t meta = __float_as_uint(q3.w);
        if (!(meta & RT_LEAF_BIT)) continue;
        const uint32_t b = __float_as_uint(q3.z), e = b + (meta & ~RT_LEAF_BIT);
        bool any = false;
        for (uint32_t w = b >> 5; w <= ((e - 1u) >> 5) && b < e && !any; w++) {
            uint32_t bits = tri_occ[w];
            if (w == (b >> 5)) bits &= ~0u << (b & 31u);
            if (w == ((e - 1u) >> 5)) bits &= ~0u >> (31u - ((e - 1u) & 31u));
            any = bits != 0u;
        }
        if (!any) continue;
        uint32_t c = r;
        for (; c != 0u; c = parent[c]) {
            const uint32_t blk = __float_as_uint(recs[4 * (size_t)parent[c] + 3].z);
            const uint32_t bit = 1u << (8u * ((blk >> 1) & 3u) + (c - blk));
            if (atomicOr(&blk_words[blk >> 3], bit) & bit) break;
        }
        if (c == 0u) atomicOr(&blk_words[0], 1u);
    }
}

} // namespace lightcull
} // namespace rtb
