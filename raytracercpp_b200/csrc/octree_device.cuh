// octree_device.cuh -- the reference's octree (BVH::BVH, bvh.cpp:19-66; OctreeNode::insert / create_children /
// compute_volume, bvh.h:141-210) built ON THE GPU, into the flattened layout of scene_layout.h.  SURVEY.md section 8(f)1:
// the reference rebuilds the whole tree on every set_object_transform (renderer/renderer.cpp:214-224); here a rebuild of a
// 10 M-triangle scene is a few milliseconds of device work on arrays that never leave HBM.
//
// The reference inserts triangles one by one, but the tree it ends up with does not depend on the order (octree_build.cpp):
// a cell splits iff more than leaf_max triangles are routed to it and it is shallower than max_depth, and a triangle is
// routed by comparing its bbox centroid with the cell's midpoint.  So, per triangle and independently of all others:
//
//   1. k_ob_keys     the PATH of the triangle through the (unbounded) subdivision: at every level the octant
//                    (c.x > mid.x) | (c.y > mid.y) << 1 | (c.z > mid.z) << 2 of bvh.h:203-207, with the cell corners
//                    computed exactly as bvh.h:155-166 does in float -- including the lower corners `lo + (0, mid.y, 0)` of
//                    children 2, 4 and 6, which make those cells' own midpoints differ from a regular grid's.  3 bits per
//                    level, max_depth levels of the reference plus kExtraLevels more for the device-side refinement of
//                    oversized leaves, one 64-bit key.
//   2. radix sort    (key, triangle index), stable, least significant byte first: triangles that share a cell at any depth
//                    are now one contiguous range, in the input order inside it -- the leaf order of the reference.
//   3. k_ob_split    level by level from the root: a cell is a range of the sorted array; it splits by the reference's rule,
//                    its <= 8 non-empty children are found by binary search on the next 3 key bits.  Below a reference
//                    leaf with more than leaf_split triangles (device-side refinement, not part of the reference tree)
//                    k_ob_refine makes the host builder's median cuts: up to 8 groups per cell, repeatedly, until a group
//                    holds <= leaf_split.  k_ob_leaf_order then puts every leaf in input order.
//   4. k_ob_bounds   bottom-up: 7-slab extents (bvh.h:33-46 per leaf, :147-149 per interior cell), subtree sizes;
//      k_ob_place    top-down: record positions in depth-first order, child blocks contiguous and 128-byte aligned;
//      k_ob_records  the 64-byte child records;  k_ob_triangles  tris[] / shade[] / orig[] / leaf_of[] in leaf order.
//
// Cells, leaf contents, leaf order, slab extents and the statistics of rt_bvh_info are those of the host builder, hence the
// reference's, and so are the groups of the refinement below oversized leaves (tests/test_gpu_parity.py::test_device_build_*:
// statistics, record counts, closest hits and the tallies of the traversal are compared with the host builder's).
#pragma once

#include "scene_layout.h"

namespace rtb {
namespace devbuild {

constexpr int kExtraLevels = 0;          // key levels below the reference's max_depth (none: the refinement orders its ranges itself)
constexpr int kMaxKeyLevels = 21;        // 3 bits each in a 64-bit key
constexpr int kSortRounds = 64;          // keys per lane of a radix-sort unit: a warp owns 32 * kSortRounds consecutive keys
constexpr int kSortUnit = 32 * kSortRounds;
constexpr int kScanItems = 4;            // items per thread of the scan kernels
constexpr int kScanBlock = 1024 * kScanItems;

struct Params {
    int32_t max_depth, leaf_max, leaf_split, total_depth;
    float s3;                            // sqrt(3) / 3, computed once on the host (bvh.cpp:12)
};

struct Stats {                           // of the reference-shaped tree
    unsigned long long interior, nonempty_children;
    unsigned int max_depth, max_leaf;
    unsigned int root_lo[3], root_hi[3]; // ordered-integer images of the root cell's corners (atomicMin / atomicMax)
    unsigned int top_n;
};

// cell flags
constexpr uint32_t kCellLeaf = 0u, kCellRefInterior = 1u, kCellDevInterior = 2u;
struct Cells {
    uint32_t* begin;                     // range [begin, end) of the sorted triangle array
    uint32_t* end;
    uint32_t* first_child;               // index of the first child cell (children are consecutive, in octant order)
    uint32_t* info;                      // nchild | kind << 8 | is_reference_cell << 10
    float* nr;                           // 7 per cell
    float* fr;
    uint32_t* size;                      // records below this cell's own record (depth-first span)
    uint32_t* rec;                       // where the cell's record goes
    uint32_t* block;                     // where its children's block starts
};

__device__ __forceinline__ unsigned int float_order(float f)      // monotonic float -> unsigned
{
    const unsigned int b = __float_as_uint(f);
    return b ^ ((b & 0x80000000u) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float order_float(unsigned int k)
{
    return __uint_as_float(k ^ ((k & 0x80000000u) ? 0x80000000u : 0xffffffffu));
}

__global__ void k_ob_init(Stats* st)
{
    st->interior = 0ull; st->nonempty_children = 0ull; st->max_depth = 0u; st->max_leaf = 0u; st->top_n = 0u;
    for (int k = 0; k < 3; k++) { st->root_lo[k] = 0xffffffffu; st->root_hi[k] = 0u; }
}

// Triangle::bbox_centroid (triangle.cpp:162-165) and the bounds of all vertices (bvh.cpp:25-36).
__global__ void __launch_bounds__(256)
k_ob_centroids(const float* xyz9, uint32_t n, float* centroid, Stats* st)
{
    __shared__ unsigned int s_lo[3], s_hi[3];
    if (threadIdx.x < 3) { s_lo[threadIdx.x] = 0xffffffffu; s_hi[threadIdx.x] = 0u; }
    __syncthreads();
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float* p = xyz9 + 9 * (size_t)i;
        for (int k = 0; k < 3; k++) {
            const float a = p[k], b = p[3 + k], c = p[6 + k];
            const float mn = fminf(a, fminf(b, c)), mx = fmaxf(a, fmaxf(b, c));
            centroid[3 * (size_t)i + k] = 0.5f * (mn + mx);                        // kk * (pmin + pmax), kk = 1.f / 2
            lo[k] = fminf(lo[k], mn); hi[k] = fmaxf(hi[k], mx);
        }
    }
    for (int k = 0; k < 3; k++) {
        unsigned int l = float_order(lo[k]), h = float_order(hi[k]);
        l = __reduce_min_sync(0xffffffffu, l); h = __reduce_max_sync(0xffffffffu, h);
        if ((threadIdx.x & 31u) == 0) { atomicMin(&s_lo[k], l); atomicMax(&s_hi[k], h); }
    }
    __syncthreads();
    if (threadIdx.x < 3) { atomicMin(&st->root_lo[threadIdx.x], s_lo[threadIdx.x]); atomicMax(&st->root_hi[threadIdx.x], s_hi[threadIdx.x]); }
}

// One level of OctreeNode::create_children (bvh.h:155-166) for the child the centroid is routed to (bvh.h:203-207).
__device__ __forceinline__ int descend(V3& lo, V3& hi, V3 c)
{
    const V3 mid = v3((lo.x + hi.x) / 2, (lo.y + hi.y) / 2, (lo.z + hi.z) / 2);
    const int o = (c.x > mid.x ? 1 : 0) + (c.y > mid.y ? 2 : 0) + (c.z > mid.z ? 4 : 0);
    V3 clo, chi;
    switch (o) {
    case 0: clo = lo;                          chi = v3(mid.x, mid.y, mid.z); break;
    case 1: clo = v3(mid.x, lo.y, lo.z);       chi = v3(hi.x, mid.y, mid.z); break;
    case 2: clo = lo + v3(0, mid.y, 0);        chi = v3(mid.x, hi.y, mid.z); break;     // as written at bvh.h:161
    case 3: clo = v3(mid.x, mid.y, lo.z);      chi = v3(hi.x, hi.y, mid.z); break;
    case 4: clo = lo + v3(0, 0, mid.z);        chi = v3(mid.x, mid.y, hi.z); break;     // bvh.h:163
    case 5: clo = v3(mid.x, lo.y, mid.z);      chi = v3(hi.x, mid.y, hi.z); break;
    case 6: clo = lo + v3(0, mid.y, mid.z);    chi = v3(mid.x, hi.y, hi.z); break;     // bvh.h:165
    default: clo = v3(mid.x, mid.y, mid.z);    chi = v3(hi.x, hi.y, hi.z); break;
    }
    lo = clo; hi = chi;
    return o;
}

__global__ void __launch_bounds__(256)
k_ob_keys(const float* centroid, uint32_t n, const Stats* st, Params P, unsigned long long* keys, uint32_t* idx)
{
    const V3 rlo = v3(order_float(st->root_lo[0]), order_float(st->root_lo[1]), order_float(st->root_lo[2]));
    const V3 rhi = v3(order_float(st->root_hi[0]), order_float(st->root_hi[1]), order_float(st->root_hi[2]));
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const V3 c = v3(centroid[3 * (size_t)i], centroid[3 * (size_t)i + 1], centroid[3 * (size_t)i + 2]);
        V3 lo = rlo, hi = rhi;
        unsigned long long key = 0ull;
        for (int level = 0; level < P.total_depth; level++) key = (key << 3) | (unsigned long long)descend(lo, hi, c);
        keys[i] = key;
        idx[i] = i;
    }
}

// ---- stable LSD radix sort of (64-bit key, 32-bit value), 8 bits per pass.  A warp owns kSortUnit consecutive keys: it
// counts their digits (k_rs_count), an exclusive scan over [digit][unit] turns the counts into positions, and the same warp
// then places its keys in input order (k_rs_scatter) -- lanes that hold the same digit in one round are ranked with
// match.any, so no two warps ever need to agree on anything and the order inside a digit is the input order.
__global__ void __launch_bounds__(128)
k_rs_count(const unsigned long long* keys, uint32_t n, int shift, uint32_t n_units, uint32_t* hist)
{
    __shared__ uint32_t cnt[4][256];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t unit = blockIdx.x * 4u + warp;
    for (int d = lane; d < 256; d += 32) cnt[warp][d] = 0u;
    __syncwarp();
    if (unit < n_units) {
        const uint32_t base = unit * (uint32_t)kSortUnit;
        for (int r = 0; r < kSortRounds; r++) {
            const uint32_t i = base + (uint32_t)r * 32u + lane;
            const bool ok = i < n;
            const uint32_t digit = ok ? (uint32_t)(keys[i] >> shift) & 255u : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, digit);
            if (ok && lane == (unsigned)(__ffs(peers) - 1)) cnt[warp][digit] += (uint32_t)__popc(peers);
            __syncwarp();
        }
        for (int d = lane; d < 256; d += 32) hist[(size_t)d * n_units + unit] = cnt[warp][d];
    }
}

__global__ void __launch_bounds__(128)
k_rs_scatter(const unsigned long long* keys, const uint32_t* vals, uint32_t n, int shift, uint32_t n_units, const uint32_t* hist,
             unsigned long long* keys_out, uint32_t* vals_out)
{
    __shared__ uint32_t pos[4][256];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t unit = blockIdx.x * 4u + warp;
    if (unit >= n_units) return;
    for (int d = lane; d < 256; d += 32) pos[warp][d] = hist[(size_t)d * n_units + unit];
    __syncwarp();
    const uint32_t base = unit * (uint32_t)kSortUnit;
    for (int r = 0; r < kSortRounds; r++) {
        const uint32_t i = base + (uint32_t)r * 32u + lane;
        const bool ok = i < n;
        const unsigned long long key = ok ? keys[i] : 0ull;
        const uint32_t digit = ok ? (uint32_t)(key >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, digit);
        const uint32_t rank = (uint32_t)__popc(peers & ((1u << lane) - 1u));
        uint32_t at = 0u;
        if (ok) at = pos[warp][digit] + rank;
        __syncwarp();
        if (ok && lane == (unsigned)(__ffs(peers) - 1)) pos[warp][digit] += (uint32_t)__popc(peers);
        __syncwarp();
        if (ok) { keys_out[at] = key; vals_out[at] = vals[i]; }
    }
}

// ---- exclusive scan of n 32-bit counters, in place: block sums, one block scans the sums, blocks add their offset.
__device__ __forceinline__ uint32_t block_exclusive_1024(uint32_t v, uint32_t* warp_part, uint32_t& total)
{
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, inc, o);
        if ((int)lane >= o) inc += a;
    }
    __syncthreads();
    if (lane == 31) warp_part[warp] = inc;
    __syncthreads();
    uint32_t w = warp_part[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, w, o);
        if ((int)lane >= o) w += a;
    }
    total = __shfl_sync(0xffffffffu, w, 31);
    const uint32_t before = __shfl_sync(0xffffffffu, w - warp_part[lane], warp);
    return before + inc - v;
}

__global__ void __launch_bounds__(1024)
k_scan_sums(const uint32_t* data, size_t n, uint32_t* sums)
{
    __shared__ uint32_t warp_part[32];
    const size_t first = (size_t)blockIdx.x * kScanBlock + (size_t)threadIdx.x * kScanItems;
    uint32_t v = 0;
    for (int j = 0; j < kScanItems; j++) if (first + j < n) v += data[first + j];
    uint32_t total;
    block_exclusive_1024(v, warp_part, total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024)
k_scan_top(uint32_t* sums, uint32_t n_blocks, uint32_t* grand_total)      // one block; n_blocks may exceed 1024
{
    __shared__ uint32_t warp_part[32];
    uint32_t carry = 0;
    for (uint32_t b = 0; b < n_blocks; b += 1024u) {
        const uint32_t i = b + threadIdx.x;
        const uint32_t v = i < n_blocks ? sums[i] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_1024(v, warp_part, total);
        if (i < n_blocks) sums[i] = carry + ex;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && grand_total) *grand_total = carry;
}

__global__ void __launch_bounds__(1024)
k_scan_apply(uint32_t* data, size_t n, const uint32_t* sums)
{
    __shared__ uint32_t warp_part[32];
    const size_t first = (size_t)blockIdx.x * kScanBlock + (size_t)threadIdx.x * kScanItems;
    uint32_t x[kScanItems], v = 0;
    for (int j = 0; j < kScanItems; j++) { x[j] = first + j < n ? data[first + j] : 0u; v += x[j]; }
    uint32_t total;
    uint32_t at = sums[blockIdx.x] + block_exclusive_1024(v, warp_part, total);
    for (int j = 0; j < kScanItems; j++) {
        if (first + j < n) data[first + j] = at;
        at += x[j];
    }
}

// ---- the tree, level by level.  Children of a cell at `depth`: the next octant is bits [shift, shift + 3) of the key.
__device__ __forceinline__ uint32_t octant_of(unsigned long long key, int shift) { return (uint32_t)(key >> shift) & 7u; }

// first position in [b, e) whose octant is >= o
__device__ __forceinline__ uint32_t octant_lower_bound(const unsigned long long* keys, uint32_t b, uint32_t e, int shift, uint32_t o)
{
    while (b < e) {
        const uint32_t m = b + ((e - b) >> 1);
        if (octant_of(keys[m], shift) < o) b = m + 1; else e = m;
    }
    return b;
}

// The groups the host builder's refinement (octree_build.cpp: emit_group) cuts a leaf of n triangles into: three rounds of
// halving every group that still holds more than leaf_split.  bounds[0..groups] are offsets into the leaf's range.
__device__ __forceinline__ int refine_groups(uint32_t n, uint32_t leaf_split, uint32_t bounds[9])
{
    int ng = 1;
    bounds[0] = 0u; bounds[1] = n;
    for (int round = 0; round < 3; round++) {
        uint32_t next[9];
        int nn = 0;
        next[0] = 0u;
        for (int g = 0; g < ng; g++) {
            const uint32_t b = bounds[g], e = bounds[g + 1];
            if (e - b > leaf_split) next[++nn] = b + (e - b) / 2u;
            next[++nn] = e;
        }
        ng = nn;
        for (int g = 0; g <= ng; g++) bounds[g] = next[g];
    }
    return ng;
}

// Between pass A and pass B: the ranges of the cells that are refined below the reference's leaves are put in the order of
// the host builder's median cuts -- per group the axis of largest centroid extent, the lower half by (centroid[axis], index)
// first -- so that pass B's groups are consecutive sub-ranges.  One warp per cell; a cut is a rank sort (leaves hold tens of
// triangles; the two 1 937-triangle pole leaves of the 10 M-triangle sphere cost a warp 0.2 ms each).
__global__ void __launch_bounds__(256)
k_ob_refine(Cells C, uint32_t level_first, uint32_t level_count, Params P, const float* centroid, uint32_t* idx, uint32_t* tmp)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < level_count; j += warps) {
        const uint32_t cell = level_first + j;
        if (((C.info[cell] >> 8) & 3u) != kCellDevInterior) continue;
        const uint32_t base = C.begin[cell], n = C.end[cell] - base;
        uint32_t bounds[9];
        int ng = 1;
        bounds[0] = 0u; bounds[1] = n;
        for (int round = 0; round < 3; round++) {
            uint32_t next[9];
            int nn = 0;
            next[0] = 0u;
            for (int g = 0; g < ng; g++) {
                const uint32_t b = base + bounds[g], e = base + bounds[g + 1];
                if (e - b > (uint32_t)P.leaf_split) {
                    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
                    for (uint32_t i = b + lane; i < e; i += 32u) {
                        const float* c = centroid + 3 * (size_t)idx[i];
                        for (int k = 0; k < 3; k++) { lo[k] = fminf(lo[k], c[k]); hi[k] = fmaxf(hi[k], c[k]); }
                    }
                    for (int k = 0; k < 3; k++)
                        for (int o = 16; o > 0; o >>= 1) {
                            lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
                            hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
                        }
                    const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
                    const int axis = (ex >= ey && ex >= ez) ? 0 : (ey >= ez ? 1 : 2);
                    for (uint32_t i = b + lane; i < e; i += 32u) {
                        const uint32_t a = idx[i];
                        const float ca = centroid[3 * (size_t)a + axis];
                        uint32_t rank = 0;
                        for (uint32_t k = b; k < e; k++) {
                            const uint32_t o = idx[k];
                            const float co = centroid[3 * (size_t)o + axis];
                            rank += (co < ca || (co == ca && o < a)) ? 1u : 0u;
                        }
                        tmp[b + rank] = a;
                    }
                    __syncwarp();
                    for (uint32_t i = b + lane; i < e; i += 32u) idx[i] = tmp[i];
                    __syncwarp();
                    next[++nn] = bounds[g] + (bounds[g + 1] - bounds[g]) / 2u;
                }
                next[++nn] = bounds[g + 1];
            }
            ng = nn;
            for (int g = 0; g <= ng; g++) bounds[g] = next[g];
        }
    }
}

// Pass A: does the cell split, and into how many non-empty children?  counts[cell - level_first] = children.
__global__ void __launch_bounds__(256)
k_ob_split(const unsigned long long* keys, Cells C, uint32_t level_first, uint32_t level_count, int depth, Params P, uint32_t* counts, Stats* st)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= level_count) return;
    const uint32_t cell = level_first + j;
    const uint32_t b = C.begin[cell], e = C.end[cell], n = e - b;
    const bool is_ref = ((C.info[cell] >> 10) & 1u) != 0u;
    const bool ref_split = is_ref && n > (uint32_t)P.leaf_max && depth != P.max_depth;              // bvh.h:171-177
    // below the reference's leaves: the host builder's refinement (median cuts into up to 8 groups, k_ob_refine), again and
    // again until a group holds <= leaf_split
    const bool dev_split = !ref_split && P.leaf_split > 0 && n > (uint32_t)P.leaf_split;
    uint32_t kids = 0;
    if (dev_split) { uint32_t gb[9]; kids = (uint32_t)refine_groups(n, (uint32_t)P.leaf_split, gb); }
    if (ref_split) {
        const int shift = 3 * (P.total_depth - 1 - depth);
        uint32_t prev = b;
        for (uint32_t o = 1; o <= 8; o++) {
            const uint32_t at = o < 8 ? octant_lower_bound(keys, prev, e, shift, o) : e;
            if (at > prev) kids++;
            prev = at;
        }
    }
    counts[j] = kids;
    C.info[cell] = kids | ((ref_split ? kCellRefInterior : dev_split ? kCellDevInterior : kCellLeaf) << 8) | ((is_ref ? 1u : 0u) << 10);
    if (ref_split) {
        atomicAdd(&st->interior, 1ull);
        atomicAdd(&st->nonempty_children, (unsigned long long)kids);
        atomicMax(&st->max_depth, (unsigned int)(depth + 1));           // all 8 children exist in the reference tree
    } else if (is_ref) {
        atomicMax(&st->max_leaf, n);
        atomicMax(&st->max_depth, (unsigned int)depth);
    }
}

// Pass B: the children.  counts[] now holds the exclusive scan of pass A's counts.
__global__ void __launch_bounds__(256)
k_ob_children(const unsigned long long* keys, Cells C, uint32_t level_first, uint32_t level_count, int depth, Params P, const uint32_t* counts,
              uint32_t next_first)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= level_count) return;
    const uint32_t cell = level_first + j;
    const uint32_t kind = (C.info[cell] >> 8) & 3u;
    if (kind == kCellLeaf) { C.first_child[cell] = 0u; return; }
    const uint32_t b = C.begin[cell], e = C.end[cell];
    const int shift = 3 * (P.total_depth - 1 - depth);
    uint32_t child = next_first + counts[j];
    C.first_child[cell] = child;
    if (kind == kCellDevInterior) {
        uint32_t gb[9];
        const int kids = refine_groups(e - b, (uint32_t)P.leaf_split, gb);
        for (int k = 0; k < kids; k++) {
            C.begin[child + k] = b + gb[k];
            C.end[child + k] = b + gb[k + 1];
            C.info[child + k] = 0u;
        }
        return;
    }
    uint32_t prev = b;
    for (uint32_t o = 1; o <= 8; o++) {
        const uint32_t at = o < 8 ? octant_lower_bound(keys, prev, e, shift, o) : e;
        if (at > prev) {
            C.begin[child] = prev; C.end[child] = at;
            C.info[child] = (kind == kCellRefInterior ? 1u : 0u) << 10;
            child++;
        }
        prev = at;
    }
}

// Inside a leaf the reference keeps the triangles in the order of the caller's array (sequential insertion; the host builder
// sorts the groups of a refined leaf the same way).  The radix sort ordered a leaf's range by the deeper key bits, so every
// leaf's indices are ranked here: one warp per leaf, rank = number of smaller indices.
__global__ void __launch_bounds__(256)
k_ob_leaf_order(Cells C, uint32_t n_cells, const uint32_t* idx_in, uint32_t* idx_out)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t cell = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; cell < n_cells; cell += warps) {
        if (((C.info[cell] >> 8) & 3u) != kCellLeaf) continue;
        const uint32_t b = C.begin[cell], n = C.end[cell] - b;
        for (uint32_t i = lane; i < n; i += 32u) {
            const uint32_t v = idx_in[b + i];
            uint32_t rank = 0;
            for (uint32_t k = 0; k < n; k++) rank += idx_in[b + k] < v ? 1u : 0u;
            idx_out[b + rank] = v;
        }
    }
}

// tris[] / shade[] / orig[] / leaf_of[] in leaf order (= sorted order): Triangle::Triangle caches cross(b - a, c - a)
// (triangle.cpp:9-10); texture coordinates default to -1 and the material index to -1 (triangle.h:48).
__global__ void __launch_bounds__(256)
k_ob_triangles(const float* xyz9, const float* uv6, const int32_t* mat, const uint32_t* idx, uint32_t n, float4* tris, float4* shade, int32_t* orig,
               int32_t* leaf_of)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t t = idx[i];
        const float* p = xyz9 + 9 * (size_t)t;
        const V3 a = v3(p[0], p[1], p[2]), b = v3(p[3], p[4], p[5]), c = v3(p[6], p[7], p[8]);
        const V3 nrm = cross(b - a, c - a);
        tris[3 * (size_t)i] = make_float4(a.x, a.y, a.z, nrm.x);
        tris[3 * (size_t)i + 1] = make_float4(b.x, b.y, b.z, nrm.y);
        tris[3 * (size_t)i + 2] = make_float4(c.x, c.y, c.z, nrm.z);
        float u[6] = {-1, -1, -1, -1, -1, -1};
        if (uv6) for (int k = 0; k < 6; k++) u[k] = uv6[6 * (size_t)t + k];
        const int32_t m = mat ? mat[t] : -1;
        shade[2 * (size_t)i] = make_float4(u[0], u[1], u[2], u[3]);
        shade[2 * (size_t)i + 1] = make_float4(u[4], u[5], __uint_as_float((uint32_t)m), __uint_as_float(t));
        orig[i] = (int32_t)t;
        leaf_of[t] = (int32_t)i;
    }
}

// Bottom-up, one level per launch: slab extents and the number of records below each cell.
__global__ void __launch_bounds__(128)
k_ob_bounds(const float4* tris, Cells C, uint32_t level_first, uint32_t level_count, Params P)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= level_count) return;
    const uint32_t cell = level_first + j;
    const uint32_t info = C.info[cell], kind = (info >> 8) & 3u, kids = info & 0xffu;
    float nr[7], fr[7];
    for (int pl = 0; pl < 7; pl++) { nr[pl] = INFINITY; fr[pl] = -INFINITY; }
    uint32_t size = 0;
    if (kind == kCellLeaf) {
        const float s = P.s3;
        const V3 planes[7] = {v3(1, 0, 0), v3(0, 1, 0), v3(0, 0, 1), v3(s, s, s), v3(-s, s, s), v3(-s, -s, s), v3(s, -s, s)};   // bvh.cpp:8-16
        const uint32_t b = C.begin[cell], e = C.end[cell];
        for (uint32_t i = b; i < e; i++) {                                      // bvh.h:33-46,143-145
            for (int k = 0; k < 3; k++) {
                const float4 q = tris[3 * (size_t)i + k];
                const V3 p = v3(q.x, q.y, q.z);
                for (int pl = 0; pl < 7; pl++) {
                    const float d = dot(planes[pl], p);
                    nr[pl] = d < nr[pl] ? d : nr[pl];                           // std::min / std::max
                    fr[pl] = fr[pl] < d ? d : fr[pl];
                }
            }
        }
    } else {
        const uint32_t first = C.first_child[cell];
        for (uint32_t k = 0; k < kids; k++) {                                   // bvh.h:147-149
            for (int pl = 0; pl < 7; pl++) {
                const float a = C.nr[7 * (size_t)(first + k) + pl], b = C.fr[7 * (size_t)(first + k) + pl];
                nr[pl] = a < nr[pl] ? a : nr[pl];
                fr[pl] = fr[pl] < b ? b : fr[pl];
            }
            size += C.size[first + k];
        }
        // a cell with one non-empty child has that child's volume: the level is skipped (as the host builder does when it
        // refines), so it adds no block of its own
        if (!(kids == 1u && P.leaf_split > 0)) size += (kids + 1u) & ~1u;
    }
    for (int pl = 0; pl < 7; pl++) { C.nr[7 * (size_t)cell + pl] = nr[pl]; C.fr[7 * (size_t)cell + pl] = fr[pl]; }
    C.size[cell] = size;
}

// Top-down: record positions, depth-first.  The block of a cell's children follows ... its record's subtree start.
__global__ void __launch_bounds__(256)
k_ob_place(Cells C, uint32_t level_first, uint32_t level_count, Params P)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= level_count) return;
    const uint32_t cell = level_first + j;
    const uint32_t info = C.info[cell], kind = (info >> 8) & 3u, kids = info & 0xffu;
    if (kind == kCellLeaf) return;
    const uint32_t first = C.first_child[cell];
    if (kids == 1u && P.leaf_split > 0) { C.rec[first] = C.rec[cell]; C.block[first] = C.block[cell]; return; }
    const uint32_t blk = C.block[cell];
    uint32_t at = blk + ((kids + 1u) & ~1u);
    for (uint32_t k = 0; k < kids; k++) {
        C.rec[first + k] = blk + k;
        C.block[first + k] = at;
        at += C.size[first + k];
    }
}

// nextafterf applied RT_SLAB_PAD_ULPS times towards -inf / +inf, on the bits (octree_build.cpp: pad)
__device__ __forceinline__ float pad_ulps(float f, int ulps)
{
    if (f != f) return f;
    const int32_t i = __float_as_int(f);
    long long ord = i >= 0 ? (long long)i : -(long long)(i & 0x7fffffff);
    ord += ulps;
    const long long inf = 0x7f800000;
    if (ord >= inf) return INFINITY;
    if (ord <= -inf) return -INFINITY;
    const uint32_t o = ord > 0 ? (uint32_t)ord : ord < 0 ? (0x80000000u | (uint32_t)(-ord)) : ((uint32_t)i & 0x80000000u);
    return __uint_as_float(o);
}

__global__ void __launch_bounds__(256)
k_ob_records(Cells C, uint32_t n_cells, Params P, float4* recs)
{
    const uint32_t cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const uint32_t info = C.info[cell], kind = (info >> 8) & 3u, kids = info & 0xffu;
    if (kind != kCellLeaf && kids == 1u && P.leaf_split > 0) return;            // skipped level: the child writes this record
    float nr[7], fr[7];
    for (int pl = 0; pl < 7; pl++) {
        nr[pl] = pad_ulps(C.nr[7 * (size_t)cell + pl], -RT_SLAB_PAD_ULPS);
        fr[pl] = pad_ulps(C.fr[7 * (size_t)cell + pl], RT_SLAB_PAD_ULPS);
    }
    const uint32_t link = kind == kCellLeaf ? C.begin[cell] : C.block[cell];
    const uint32_t meta = kind == kCellLeaf ? (RT_META_LEAF | (C.end[cell] - C.begin[cell])) : kids;
    float4* q = recs + 4 * (size_t)C.rec[cell];
    q[0] = make_float4(nr[0], fr[0], nr[1], fr[1]);
    q[1] = make_float4(nr[2], fr[2], nr[3], fr[3]);
    q[2] = make_float4(nr[4], fr[4], nr[5], fr[5]);
    q[3] = make_float4(nr[6], fr[6], __uint_as_float(link), __uint_as_float(meta));
}

// The top table (octree_build.cpp: build_top_table): breadth-first from the root, whole child blocks while they fit.
__global__ void k_ob_top_table(float4* recs, float4* top, Stats* st)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t q_rec[RT_TOP_RECORDS + 1];
    int q_top[RT_TOP_RECORDS + 1];
    int qn = 0, used = 0;
    q_rec[qn] = 0u; q_top[qn] = -1; qn++;
    for (int qi = 0; qi < qn; qi++) {
        float4* q3 = recs + 4 * (size_t)q_rec[qi] + 3;
        const uint32_t link = __float_as_uint(q3->z), meta = __float_as_uint(q3->w);
        if ((meta & RT_META_LEAF) || meta == 0u) continue;
        const uint32_t count = meta & RT_META_COUNT_MASK;
        if (used + (int)count > RT_TOP_RECORDS) continue;
        for (uint32_t k = 0; k < count; k++) {
            for (int j = 0; j < 4; j++) top[4 * (size_t)(used + k) + j] = recs[4 * (size_t)(link + k) + j];
            q_rec[qn] = link + k; q_top[qn] = used + (int)k; qn++;
        }
        const uint32_t tagged = meta | RT_META_TOP | ((uint32_t)used << RT_META_TOP_SHIFT);
        q3->w = __uint_as_float(tagged);
        if (q_top[qi] >= 0) top[4 * (size_t)q_top[qi] + 3].w = __uint_as_float(tagged);
        used += (int)count;
    }
    st->top_n = (unsigned int)used;
}

// ---- wrecs[]: the wide copy of the tree that the packet kernels traverse.  A packet's cell round (pop, fetch, stage,
// pyramid cull, slab tests, insertion) has a fixed cost sized for kWideBlock (16) children, and a cell of the reference's
// octree has 2.6 on average (10 M-triangle sphere): one round per level.  Every block of wrecs[] is a collapse of the tree
// below one owner record instead.  Collapse rule: the block starts as the owner's children; repeatedly, the interior member
// with the largest surface area of its axis box (first three slabs) among those whose children still fit (members - 1 + its
// count <= limit, limit = kWideBlock) is replaced IN PLACE by its children, ties to the lower position; it stops when no
// member fits.  Members spliced in can be absorbed in turn, so a block may reach several levels down.
// A node of the wide tree is a record of recs[] (`src`): leaves are copied unchanged (same triangles), interior records
// get their wide block and member count.  Same pattern as the narrow build: nodes frontier by frontier (k_wb_collapse,
// scan, k_wb_children), sizes bottom-up (k_wb_size), positions top-down (k_ob_place), then the records (k_wb_records).
// Packet stack: a cell round pops one entry and pushes at most the block's members, so a packet never holds more than
// 1 + max over root-to-leaf paths of the sum of (members - 1) of the blocks on the path.  Wider blocks can raise that sum
// above the narrow tree's (a block may absorb a sibling of the path and still advance it by one level), so k_wb_size
// computes it (`need`) and build_wide_tree lowers the limit until 1 + need fits RT_STACK_SIZE; with limit 1 nothing is
// absorbed and the bound is the narrow tree's.
__device__ __forceinline__ bool wb_interior(uint32_t meta) { return !(meta & RT_META_LEAF) && (meta & RT_META_COUNT_MASK) != 0u; }

__device__ __forceinline__ float wb_axis_area(const float4* recs, uint32_t r)      // half the surface area of the axis box
{
    const float4 q0 = recs[4 * (size_t)r], q1 = recs[4 * (size_t)r + 1];
    const float dx = q0.y - q0.x, dy = q0.w - q0.z, dz = q1.y - q1.x;
    return dx * dy + dy * dz + dz * dx;
}

// members[kWideBlock j ..] = the block of node lf + j (a record of recs[] that is interior), counts[j] = its size (0: leaf)
__global__ void __launch_bounds__(256)
k_wb_collapse(const float4* recs, const uint32_t* src, uint32_t lf, uint32_t lc, uint32_t limit, uint32_t* info, uint32_t* counts, uint32_t* members)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= lc) return;
    const float4 own = recs[4 * (size_t)src[lf + j] + 3];
    const uint32_t meta = __float_as_uint(own.w);
    if (!wb_interior(meta)) { counts[j] = 0u; info[lf + j] = 0u; return; }
    uint32_t m[kWideBlock], kids[kWideBlock], link[kWideBlock];
    float area[kWideBlock];
    int n = 0;
    auto put = [&](int at, uint32_t r) {
        const float4 q3 = recs[4 * (size_t)r + 3];
        const uint32_t mm = __float_as_uint(q3.w);
        m[at] = r;
        kids[at] = wb_interior(mm) ? (mm & RT_META_COUNT_MASK) : 0u;
        link[at] = __float_as_uint(q3.z);
        area[at] = kids[at] ? wb_axis_area(recs, r) : 0.0f;
    };
    const uint32_t first = __float_as_uint(own.z), count = meta & RT_META_COUNT_MASK;
    for (uint32_t k = 0; k < count; k++) put(n++, first + k);
    for (;;) {
        int best = -1;
        for (int k = 0; k < n; k++)
            if (kids[k] && n - 1 + (int)kids[k] <= (int)limit && (best < 0 || area[k] > area[best])) best = k;
        if (best < 0) break;
        const int c = (int)kids[best];
        const uint32_t l = link[best];
        for (int k = n - 1; k > best; k--) {                                   // the members behind it move c - 1 places up
            m[k + c - 1] = m[k]; kids[k + c - 1] = kids[k]; link[k + c - 1] = link[k]; area[k + c - 1] = area[k];
        }
        for (int k = 0; k < c; k++) put(best + k, l + (uint32_t)k);
        n += c - 1;
    }
    for (int k = 0; k < n; k++) members[kWideBlock * (size_t)j + k] = m[k];
    counts[j] = (uint32_t)n;
    info[lf + j] = (uint32_t)n | (kCellRefInterior << 8);
}

// the members of the frontier's blocks become the next frontier; counts[] now holds the exclusive scan
__global__ void __launch_bounds__(256)
k_wb_children(Cells C, uint32_t* src, uint32_t lf, uint32_t lc, const uint32_t* counts, const uint32_t* members, uint32_t next_first)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= lc) return;
    const uint32_t kids = C.info[lf + j] & 0xffu;
    const uint32_t child = next_first + counts[j];
    C.first_child[lf + j] = kids ? child : 0u;
    for (uint32_t k = 0; k < kids; k++) src[child + k] = members[kWideBlock * (size_t)j + k];
}

// bottom-up: records below each node (its block, padded to an even count, and the blocks below) and the stack need of its
// subtree (max over paths of the sum of members - 1)
__global__ void __launch_bounds__(256)
k_wb_size(Cells C, uint32_t* need, uint32_t lf, uint32_t lc)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= lc) return;
    const uint32_t node = lf + j, kids = C.info[node] & 0xffu, first = C.first_child[node];
    uint32_t size = kids ? (kids + 1u) & ~1u : 0u, below = 0u;
    for (uint32_t k = 0; k < kids; k++) { size += C.size[first + k]; below = max(below, need[first + k]); }
    C.size[node] = size;
    need[node] = kids ? kids - 1u + below : 0u;
}

__global__ void __launch_bounds__(256)
k_wb_records(const float4* recs, const uint32_t* src, Cells C, uint32_t n_nodes, float4* wrecs)
{
    const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n_nodes) return;
    const float4* s = recs + 4 * (size_t)src[node];
    float4* q = wrecs + 4 * (size_t)C.rec[node];
    float4 q3 = s[3];
    const uint32_t kids = C.info[node] & 0xffu;
    if (kids) { q3.z = __uint_as_float(C.block[node]); q3.w = __uint_as_float(kids); }
    q[0] = s[0]; q[1] = s[1]; q[2] = s[2]; q[3] = q3;
}

// The box set of the screen coverage (rtb200.cu: screen_coverage): the axis box (padded first three slabs) of every wide node
// in [0, n) that lies on a level at or below `first_kept` or is a leaf; the others get an empty box.  Every triangle lies in
// a leaf, and every leaf either lies above that level or below a node of it, so the union of the kept boxes holds them all.
__global__ void __launch_bounds__(256)
k_wb_boxes(const float4* recs, const uint32_t* src, const uint32_t* info, uint32_t n, uint32_t first_kept, float* boxes)
{
    const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= n) return;
    const float4 q0 = recs[4 * (size_t)src[node]], q1 = recs[4 * (size_t)src[node] + 1];
    const bool keep = node >= first_kept || (info[node] & 0xffu) == 0u;
    float* b = boxes + 6 * (size_t)node;
    b[0] = keep ? q0.x : INFINITY; b[1] = keep ? q0.z : INFINITY; b[2] = keep ? q1.x : INFINITY;
    b[3] = keep ? q0.y : -INFINITY; b[4] = keep ? q0.w : -INFINITY; b[5] = keep ? q1.y : -INFINITY;
}

// Transform::operator()(Triangle) on the device copy of the caller's vertices (mat.cpp:133-140), renderer.cpp:214-224
__global__ void __launch_bounds__(256)
k_ob_transform(float* xyz, size_t n_vertices, M4 t)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vertices; i += (size_t)gridDim.x * blockDim.x) {
        const V3 p = xform_point(t, v3(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        xyz[3 * i] = p.x; xyz[3 * i + 1] = p.y; xyz[3 * i + 2] = p.z;
    }
}

} // namespace devbuild
} // namespace rtb
