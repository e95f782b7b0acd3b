// scene_layout.h -- the flattened, HBM-resident form of the reference's pointer octree (bvh.h:108-289).
//
// Reference layout (per node, 176 B + heap): 8 child pointers, std::vector<Triangle*>, AABB, 7 near + 7 far floats.
// B200 layout (SoA, read with 128-bit loads):
//
//   recs[]  : one 64-byte "child record" per NON-EMPTY octree cell = 4 x float4, the 7 slabs as (near, far) pairs:
//               q0 = near[0], far[0], near[1], far[1]      q1 = near[2], far[2], near[3], far[3]
//               q2 = near[4], far[4], near[5], far[5]      q3 = near[6], far[6], bits(link), bits(meta)
//             (pairs, so that the lane that stages a float4 for a 32-ray packet whose rays agree on the sign of a slab's
//             denominator can swap that pair in place: the packet's slab test then needs no min/max per slab, kernels.cuh;
//             the three axis slabs are q0 and half of q1)
//             meta bit 31 = leaf; low 8 bits = number of child records (interior, 1..8; 1..16 in wrecs[]); leaf: low 31 bits = triangle count
//             meta bit 30 (interior only) = the children block is also in the TOP TABLE, at record offset (meta >> 8) & 0xff
//             link        = first triangle (leaf) or first child record (interior)
//             The (<= 8) records of one interior cell are contiguous and start on a 128-byte boundary, so a cell
//             is 1..4 full cache lines.  Record 0 is the root cell itself.  Cells are laid out depth-first, so a
//             subtree is one contiguous span.  Empty cells (the reference allocates all 8 children, bvh.h:159-166)
//             have near=+inf/far=-inf, can never pass the slab test (bvh.h:101) and are dropped.
//             Bounds are widened by RT_SLAB_PAD_ULPS ulps: the slab test multiplies by a reciprocal where the
//             reference divides (bvh.h:92-93), so the widening keeps it conservative; it can only add visits.
//   top[]   : copies of the child blocks of the first levels, breadth-first from the root, at most RT_TOP_RECORDS records
//             (root's block + its children's blocks: 8 + 64 when all are full) = 4.6 KB that every CTA of the packet kernels
//             loads into shared memory once, with one bulk asynchronous copy (cp.async.bulk), and traverses from there.
//   tris[]  : 48 bytes per triangle in LEAF order = 3 x float4: (a.xyz, n.x) (b.xyz, n.y) (c.xyz, n.z) with
//             n = cross(b-a, c-a), the un-normalised normal the reference caches (triangle.cpp:9-10).
//   shade[] : 32 bytes per triangle in leaf order, read by shading only = 2 x float4:
//             (u_a, u_b, u_c, v_a) (v_b, v_c, bits(material), bits(original index))
#pragma once

#include <stdint.h>
#include <memory>
#include <new>
#include <utility>
#include <vector>

#include "rt_math.h"

#define RT_SLAB_PAD_ULPS 4
#define RT_MAX_TREE_DEPTH 20
#define RT_META_LEAF 0x80000000u
#ifndef RT_META_TOP
#define RT_META_TOP 0x40000000u
#define RT_META_TOP_SHIFT 8
#define RT_META_COUNT_MASK 0xffu       /* interior records */
#ifndef RT_TOP_RECORDS
#define RT_TOP_RECORDS 72
#endif
#endif

namespace rtb {

struct alignas(16) F4 {
    float x, y, z, w;
};

// std::allocator whose value-less construct() leaves trivial types uninitialised: resize(n) of a gigabyte array does not
// write it once on one thread before the parallel copy fills it.
template <class T>
struct DefaultInitAllocator : std::allocator<T> {
    template <class U> struct rebind { typedef DefaultInitAllocator<U> other; };
    template <class U> void construct(U* p) { ::new ((void*)p) U; }
    template <class U, class... A> void construct(U* p, A&&... a) { ::new ((void*)p) U(std::forward<A>(a)...); }
};
template <class T> using RawVector = std::vector<T, DefaultInitAllocator<T>>;

struct FlatScene {
    RawVector<F4> recs;          // 4 per record
    RawVector<F4> tris;          // 3 per triangle, leaf order
    RawVector<F4> shade;         // 2 per triangle, leaf order
    RawVector<int32_t> orig;     // leaf order -> index in the caller's array
    RawVector<F4> top;           // 4 per record of the top table (<= RT_TOP_RECORDS records)
    // statistics of the (reference-shaped) octree
    uint64_t nodes = 0, leaves = 0, empty_leaves = 0, interior = 0;
    uint32_t max_depth_reached = 0, max_leaf_size = 0;
    uint64_t n_records = 0;
};

// Builds the reference's octree (same cells, same leaf contents in the same order as sequential insertion,
// bvh.cpp:19-66 / bvh.h:141-210) top-down and flattens it.  uv6 / mat may be null (defaults of triangle.h:48).
// leaf_split > 0 additionally refines, on the B200 side only, every reference leaf that holds more than leaf_split
// triangles into a small median-split hierarchy of groups of <= leaf_split triangles (octree_build.cpp:emit_group) and
// skips levels with a single non-empty child; leaf_split = 0 keeps exactly the reference's cells and leaves.  The
// statistics below always describe the reference-shaped octree.
void build_flat_scene(const float* xyz9, const float* uv6, const int32_t* mat, size_t n, int max_depth,
                      int leaf_max, int leaf_split, FlatScene& out);

inline uint32_t f2u(float f) { uint32_t u; __builtin_memcpy(&u, &f, 4); return u; }
inline float u2f(uint32_t u) { float f; __builtin_memcpy(&f, &u, 4); return f; }

} // namespace rtb
