// rt_device.h -- per-ray device functions of the hot path: 7-slab octree traversal (closest hit and any hit),
// Moeller-Trumbore, shading, texture taps, the rough-reflection fan.  Included by kernels.cu (nvcc, sm_100a).
// The functions are plain inline code over pointer-based views so that tests/hostsim can compile the very same
// source with g++ and run it single-threaded against the oracle before any GPU time is spent; that build lives
// under tests/ only and is never part of librtb200.so.
//
// Build contract: no FMA contraction (nvcc --fmad=false / g++ -ffp-contract=off), IEEE div/sqrt.
#pragma once

#include "rt_math.h"
#include "../../include/rtb200.h"

#if defined(__CUDACC__)
#define RT_LDG4(p) __ldg(reinterpret_cast<const float4*>(p))
#define RT_DEV __device__ __forceinline__
#define RT_DEV_NOINLINE __device__ __noinline__
#define RT_FMA(a, b, c) __fmaf_rn((a), (b), (c))
typedef float4 rt_f4;
#else
#include "scene_layout.h"
#define RT_LDG4(p) (*(p))
#define RT_DEV inline
#define RT_DEV_NOINLINE inline
#define RT_FMA(a, b, c) fmaf((a), (b), (c))
typedef rtb::F4 rt_f4;
#endif

/* 7 * RT_MAX_TREE_DEPTH + root, rounded up.  Also bounds the packet stacks on the wide tree (octree_device.cuh, k_wb_*):
   a root-to-leaf path there visits a subset of the records of the same path in recs[], so it is never deeper. */
#define RT_STACK_SIZE 160
#define RT_LEAF_BIT 0x80000000u
#ifndef RT_META_TOP                    /* the meta word of an interior record, see scene_layout.h */
#define RT_META_TOP 0x40000000u
#define RT_META_TOP_SHIFT 8
#define RT_META_COUNT_MASK 0xffu
#ifndef RT_TOP_RECORDS
#define RT_TOP_RECORDS 72
#endif
#endif

namespace rtb {

#if defined(__CUDACC__)
RT_DEV uint32_t f4_bits(float f) { return __float_as_uint(f); }
#else
inline uint32_t f4_bits(float f) { uint32_t u; __builtin_memcpy(&u, &f, 4); return u; }
#endif

struct TexView {
    const void* data;   // RGBA texels, row 0 first
    int32_t w, h;
    int32_t format;     // 0 = none, 1 = u8 (decoded as u8 * (1/255.f)), 2 = f32
    int32_t pad;
};

// Everything a ray needs, by value in kernel parameter space.
struct SceneView {
    const rt_f4* recs;      // 4 per child record (scene_layout.h)
    const rt_f4* top;       // the top table: copies of the first levels' child blocks, top_n records (<= RT_TOP_RECORDS)
    int32_t top_n;
    const rt_f4* tris;      // 3 per triangle, leaf order
    const rt_f4* shade;     // 2 per triangle, leaf order
    const rt_f4* mats;      // 4 per material (RtMaterial = 16 floats)
    const int32_t* orig;    // leaf order -> index in the caller's array (tie-break + reported ids)
    const int32_t* leaf_of; // the inverse: index in the caller's array -> leaf order (split primary packets)
    const rt_f4* shapes;    // 2 per analytic shape, in the order they were added: (a.xyz, radius^2) (n.xyz, bits(mat | kind << 31))
    int32_t n_shapes;       // kind 0 = Sphere (a = centre), 1 = Plane (a = point, n = normal)
    int32_t n_mats;
    uint32_t n_tris;
    const rt_f4* frag_shade; // hybrid raster path only (raster_device.h): shading records of the clipped pieces being shaded, one per
                             // thread; triangle index n_tris + i means record i here (their texture coordinates are the clipped ones)
    // Any-hit packet traversal only (light_cull.cuh): which triangles and subtrees may occlude the point light.  tri_occ: bit i
    // = triangle i; blk_occ[link >> 1]: bit k = child record k of the block that starts at record `link`; byte 0, bit 0 = the root.
    const uint32_t* tri_occ;
    const uint8_t* blk_occ;
    TexView tex[RT_TEX_COUNT];
};

struct FrameView {
    M4 proj_inv;            // Camera::_perspective_proj_mat_inv
    M4 cam_to_world;        // Camera::_camera_to_world_mat
    V3 cam_pos;             // Camera::_position
    V3 light;               // PointLight::_position
    int32_t rw, rh;         // supersampled frame (renderer.cpp:116-120)
    int32_t factor;         // ssaa factor or 1
    RtSettings s;
};

struct HitRec {             // what a closest-hit query returns; tri is a LEAF-ORDER index
    int32_t tri;
    float t, u, v;
};

struct Hit {                // HitInfo, hitInfo.h:8-29 (triangle pointer -> leaf-order index)
    int32_t tri;
    float t, u, v;
    int32_t mat;
    V3 normal;
    V3 tangent;
};

RT_DEV Hit fresh_hit()
{
    Hit h;
    h.tri = -1; h.t = -1.0f; h.u = 1.0f; h.v = 0.0f; h.mat = -1;
    h.normal = v3(0, 0, 0); h.tangent = v3(0, 0, 0);
    return h;
}

struct TraceCounters {      // per-thread tallies, reduced by the kernels
    uint32_t refl_rays, refl_shadow_rays, stack_overflow;
    // work actually done by the traversal (only maintained by the COUNT instantiations): 7-slab volume tests and
    // ray/triangle tests, the V and T of the bytes-per-ray metric (56 V + 36 T, DESIGN.md)
    unsigned long long vol_tests, tri_tests;
    // what the kernel FETCHED for those tests (COUNT only): 64-byte child records and 48-byte triangles.  A single ray
    // fetches one per test; a 32-ray packet fetches one per warp and tests it in every lane (counted by lane 0).
    unsigned long long rec_fetch, tri_fetch;
};

RT_DEV TraceCounters zero_counters()
{
    TraceCounters tc;
    tc.refl_rays = 0; tc.refl_shadow_rays = 0; tc.stack_overflow = 0; tc.vol_tests = 0; tc.tri_tests = 0; tc.rec_fetch = 0; tc.tri_fetch = 0;
    return tc;
}

// ------------------------------------------------------------------------------------------------------------
// Per-ray constants of the slab test.  The reference computes, per plane i, denom = N_i.d and numer = N_i.o
// (bvh.h:216-223) and then (d_near - numer) / denom, (d_far - numer) / denom (bvh.h:92-93).  Here the two quotients
// are one fused multiply-add each: bound * inv_i - c_i with inv_i = 1/denom_i and c_i = numer_i * inv_i.  That form
// is NOT bit-identical to the reference's (it does not have to be: slab distances only prune and order, they never
// reach a result) and it can cancel when |c_i| is large, so the interval is widened by `slack` = 2^-22 * max_i |c_i|
// on top of the ulp padding of the stored bounds (scene_layout.h): the test can only accept more than the exact one.
// A plane with denom == 0 is skipped by the reference (bvh.h:86-87); here its c is NaN so both distances are NaN and
// the NaN-dropping fminf / fmaxf leave the running interval untouched.
struct SlabRay {
    float inv[7];
    float c[7];
    float slack;
};

RT_DEV void slab_setup(V3 o, V3 d, SlabRay& sr)
{
    const float s = 0.57735026f;                     // sqrt(3.f)/3, bvh.cpp:12-15 (same float)
    float den[7], num[7];
    den[0] = d.x; den[1] = d.y; den[2] = d.z;
    num[0] = o.x; num[1] = o.y; num[2] = o.z;
    den[3] = s * d.x + s * d.y + s * d.z;      num[3] = s * o.x + s * o.y + s * o.z;
    den[4] = -s * d.x + s * d.y + s * d.z;     num[4] = -s * o.x + s * o.y + s * o.z;
    den[5] = -s * d.x + -s * d.y + s * d.z;    num[5] = -s * o.x + -s * o.y + s * o.z;
    den[6] = s * d.x + -s * d.y + s * d.z;     num[6] = s * o.x + -s * o.y + s * o.z;
    float cmax = 0.0f;
#pragma unroll
    for (int i = 0; i < 7; i++) {
        if (den[i] == 0.0f) { sr.inv[i] = 0.0f; sr.c[i] = NAN; }
        else {
            sr.inv[i] = 1.0f / den[i];
            sr.c[i] = num[i] * sr.inv[i];
            cmax = fmaxf(cmax, fabsf(sr.c[i]));
        }
    }
    sr.slack = cmax * 2.3841858e-7f;                 // 2^-22
}

// 7-slab interval of one 64-byte record.  Returns the entry distance, or +inf when the record is missed / lies
// behind the ray / starts beyond t_limit.  (The reference has no t_far<0 / t_near>best cull, bvh.h:79-105; both
// are pure pruning: a triangle needs t >= 0 and must beat the best hit strictly, bvh.h:241.)  The three axis slabs
// are tested first: most children of a visited cell are already missed there (measured on the 10 M-triangle scene:
// 65 % of the child tests end at the axis slabs).  The diagonal slabs are not optional: skipping them on interior
// records made the shadow pass 12x slower.
RT_DEV float slab_entry(const rt_f4& q0, const rt_f4& q1, const rt_f4& q2, const rt_f4& q3, const SlabRay& sr, float t_limit)
{
    float tn = -INFINITY, tf = INFINITY;
#define RT_SLAB(i, NEAR, FAR)                                   \
    {                                                           \
        float a = RT_FMA((NEAR), sr.inv[i], -sr.c[i]);          \
        float b = RT_FMA((FAR), sr.inv[i], -sr.c[i]);           \
        tn = fmaxf(tn, fminf(a, b));                            \
        tf = fminf(tf, fmaxf(a, b));                            \
    }
    RT_SLAB(0, q0.x, q0.y)
    RT_SLAB(1, q0.z, q0.w)
    RT_SLAB(2, q1.x, q1.y)
    const float lim = fminf(t_limit, tf) + 2.0f * sr.slack;
    if (!(tn <= lim) || tf + sr.slack < 0.0f) return INFINITY;
    RT_SLAB(3, q1.z, q1.w)
    RT_SLAB(4, q2.x, q2.y)
    RT_SLAB(5, q2.z, q2.w)
    RT_SLAB(6, q3.x, q3.y)
#undef RT_SLAB
    bool ok = (tn <= tf + 2.0f * sr.slack) && (tf + sr.slack >= 0.0f) && (tn - sr.slack <= t_limit);
    return ok ? tn - sr.slack : INFINITY;
}

// Triangle::intersect with MOLLER_TRUMBORE 1 / BACKFACE_CULLING 1 -- triangle.cpp:25-91.  p0..p2 are the three
// float4 of a triangle (a|n.x, b|n.y, c|n.z).  Returns true and (t,u,v) when the reference would.
RT_DEV bool tri_test(const rt_f4& p0, const rt_f4& p1, const rt_f4& p2, V3 o, V3 md, float& t, float& u, float& v)
{
    V3 a = v3(p0.x, p0.y, p0.z);
    V3 n = v3(p0.w, p1.w, p2.w);
    float det = dot(n, md);
    if (!(det > 0.0f)) return false;                      // Mdet <= 0 (or NaN): back-facing or parallel, :38-39
    V3 ab = v3(p1.x, p1.y, p1.z) - a;
    V3 ac = v3(p2.x, p2.y, p2.z) - a;
    V3 oa = o - a;
    V3 mdxoa = cross(md, oa);
    det = 1.0f / det;
    u = dot(mdxoa, ac) * det;
    if (u < 0.0f || u > 1.0f) return false;
    v = dot(mdxoa, -ab) * det;
    if (v < 0.0f || u + v > 1.0f) return false;
    t = dot(n, oa) * det;
    if (t < 0.0f) return false;
    return true;
}

// ------------------------------------------------------------------------------------------------------------
// Traversal as a resumable state machine with ONE TEST PER STEP: a step is either one 7-slab test of one child
// record (mode CHILDREN) or one ray/triangle test (mode TRIANGLES).  The run-to-completion functions below loop over
// the steps; the persistent kernels (kernels.cuh) interleave the steps of 32 rays, so every lane of a warp does the
// same amount of work per iteration whatever the arity of its cell or the size of its leaf, and lanes whose ray has
// ended are refilled.
//
// Closest hit (ANY = false): BVH::intersect (bvh.cpp:68-71 -> bvh.h:212-287).  The reference descends children in
// order of slab entry distance through a heap-allocated priority queue and stops when the best hit beats the next
// entry; the result is the exact closest front-facing hit, first-found on ties.  Here the hit children of a cell go
// far-to-near onto an explicit per-thread stack of (entry distance, link, meta) triples, the nearest is popped first,
// and entries whose distance exceeds the best hit are dropped at pop time.  Leaf triangles are visited in array order
// with the reference's strict `<` (bvh.h:241); a tie on t goes to the lower original index (the same rule inside a
// leaf).
//
// Any hit (ANY = true): Renderer::is_shadowed (renderer.cpp:340-402).  The reference runs a CLOSEST-hit query from
// p + n*EPSILON towards the light and then compares |p - hitpoint|^2 with |p - light|^2.  Beyond 2e-4 from the origin
// that predicate is monotone in t, so "some front-facing hit with t > 0 satisfies it" is the same statement as "the
// closest one does": the same near-first traversal stops at the first such hit and drops cells that start beyond the
// light.  (Near-first matters: a point that faces away from the light is occluded by its own neighbourhood, which an
// unordered walk may reach last -- measured 1.5x on the lower half of the 10 M-triangle sphere.)
#define RT_MODE_DONE 0u
#define RT_MODE_CHILDREN 1u
#define RT_MODE_TRIANGLES 2u

struct RayState {
    SlabRay sr;
    V3 o, md;                       // origin, -direction
    float t_max;                    // closest: best t so far; any: distance limit of the light
    HitRec best;                    // closest: best.tri = LEAF-ORDER index or -1
    V3 p;                           // any: the shaded point (renderer.cpp:344)
    float dist2;                    // any: |p - light|^2
    bool occluded;                  // any: result
    uint32_t mode;                  // RT_MODE_*
    uint32_t next, left;            // next child record / triangle to test and how many remain in the range
    int sp, base;                   // stack top; first entry pushed by the current cell
};

// The per-thread traversal stack lives apart from the scalar state so that the state stays in registers.
struct RayStack {
    float t[RT_STACK_SIZE];
    uint32_t link[RT_STACK_SIZE];
    uint32_t meta[RT_STACK_SIZE];
};

RT_DEV void ray_enter(RayState& S, uint32_t link, uint32_t meta)
{
    S.next = link;
    S.base = S.sp;
    if (meta & RT_LEAF_BIT) { S.mode = RT_MODE_TRIANGLES; S.left = meta & ~RT_LEAF_BIT; }
    else { S.mode = RT_MODE_CHILDREN; S.left = meta & RT_META_COUNT_MASK; }
}

RT_DEV void ray_pop(RayState& S, const RayStack& K)
{
    S.mode = RT_MODE_DONE;
    while (S.sp > 0) {
        --S.sp;
        if (K.t[S.sp] > S.t_max) continue;                  // a closer hit was found since this cell was pushed
        ray_enter(S, K.link[S.sp], K.meta[S.sp]);
        break;
    }
}

// Root cell (bvh.h:232-233) + per-ray constants.
template <bool COUNT>
RT_DEV void ray_begin(const SceneView& sc, V3 o, V3 d, float t_max, RayState& S, TraceCounters* tc)
{
    slab_setup(o, d, S.sr);
    S.o = o; S.md = -d;
    S.t_max = t_max;
    S.best.tri = -1; S.best.t = -1.0f; S.best.u = 1.0f; S.best.v = 0.0f;
    S.occluded = false;
    S.sp = 0;
    S.mode = RT_MODE_DONE;
    const rt_f4* r = sc.recs;
    rt_f4 q0 = RT_LDG4(r), q1 = RT_LDG4(r + 1), q2 = RT_LDG4(r + 2), q3 = RT_LDG4(r + 3);
    if (COUNT) { tc->vol_tests++; tc->rec_fetch++; }
    const uint32_t meta = f4_bits(q3.w);
    if (slab_entry(q0, q1, q2, q3, S.sr, S.t_max) != INFINITY && (meta & ~(RT_LEAF_BIT | RT_META_TOP)) != 0u) ray_enter(S, f4_bits(q3.z), meta);
}

template <bool COUNT>
RT_DEV void closest_begin(const SceneView& sc, V3 o, V3 d, RayState& S, TraceCounters* tc)
{
    ray_begin<COUNT>(sc, o, d, INFINITY, S, tc);
}

template <bool COUNT>
RT_DEV void any_begin(const SceneView& sc, V3 p, V3 n, V3 light, RayState& S, TraceCounters* tc)
{
    const V3 o = p + 1.0e-4f * n;                            // Renderer::EPSILON, renderer.h:23
    const V3 d = normalize(light - p);
    const float dist2 = length2(p - light);
    ray_begin<COUNT>(sc, o, d, (sqrtf(dist2) + 4.0e-4f) * 1.0001f, S, tc);
    S.p = p;
    S.dist2 = dist2;
}

template <bool COUNT>
RT_DEV void ray_child_step(const SceneView& sc, RayState& S, RayStack& K, TraceCounters* tc)
{
    const rt_f4* r = sc.recs + 4 * (size_t)S.next;
    rt_f4 c0 = RT_LDG4(r), c1 = RT_LDG4(r + 1), c2 = RT_LDG4(r + 2), c3 = RT_LDG4(r + 3);
    if (COUNT) { tc->vol_tests++; tc->rec_fetch++; }
    const float tn = slab_entry(c0, c1, c2, c3, S.sr, S.t_max);
    if (tn != INFINITY) {
        if (S.sp >= RT_STACK_SIZE) { tc->stack_overflow = 1; S.mode = RT_MODE_DONE; return; }
        int j = S.sp;                                       // keep [base, sp) sorted by descending entry distance
        while (j > S.base && K.t[j - 1] < tn) {
            K.t[j] = K.t[j - 1];
            K.link[j] = K.link[j - 1];
            K.meta[j] = K.meta[j - 1];
            --j;
        }
        K.t[j] = tn;
        K.link[j] = f4_bits(c3.z);
        K.meta[j] = f4_bits(c3.w);
        ++S.sp;
    }
    ++S.next;
    if (--S.left == 0u) ray_pop(S, K);
}

template <bool ANY, bool COUNT>
RT_DEV void ray_triangle_step(const SceneView& sc, RayState& S, const RayStack& K, TraceCounters* tc)
{
    const rt_f4* tp = sc.tris + 3 * (size_t)S.next;
    rt_f4 p0 = RT_LDG4(tp), p1 = RT_LDG4(tp + 1), p2 = RT_LDG4(tp + 2);
    if (COUNT) { tc->tri_tests++; tc->tri_fetch++; }
    float t, u, v;
    if (tri_test(p0, p1, p2, S.o, S.md, t, u, v)) {
        if (ANY) {
            if (t > 0.0f) {
                V3 q = S.o + t * (-S.md);                    // renderer.cpp:351
                if (length2(S.p - q) < S.dist2) {            // renderer.cpp:354
                    S.occluded = true;
                    S.mode = RT_MODE_DONE;
                    return;
                }
            }
        } else if (t < S.t_max || (t == S.t_max && sc.orig[S.next] < sc.orig[S.best.tri])) {
            S.t_max = t;
            S.best.tri = (int32_t)S.next; S.best.t = t; S.best.u = u; S.best.v = v;
        }
    }
    ++S.next;
    if (--S.left == 0u) ray_pop(S, K);
}

// Returns the reference's bool (a hit with t > 0: the leaf returns t_near > 0, bvh.h:245-247).
RT_DEV bool closest_found(const RayState& S) { return S.best.tri >= 0 && S.best.t > 0.0f; }

template <bool COUNT>
RT_DEV bool trace_closest(const SceneView& sc, V3 o, V3 d, HitRec& best, TraceCounters* tc)
{
    RayState S;
    RayStack K;
    closest_begin<COUNT>(sc, o, d, S, tc);
    while (S.mode != RT_MODE_DONE) {
        if (S.mode == RT_MODE_CHILDREN) ray_child_step<COUNT>(sc, S, K, tc);
        else ray_triangle_step<false, COUNT>(sc, S, K, tc);
    }
    best = S.best;
    return closest_found(S);
}

template <bool COUNT>
RT_DEV bool trace_occluded(const SceneView& sc, V3 p, V3 n, V3 light, TraceCounters* tc)
{
    RayState S;
    RayStack K;
    any_begin<COUNT>(sc, p, n, light, S, tc);
    while (S.mode != RT_MODE_DONE) {
        if (S.mode == RT_MODE_CHILDREN) ray_child_step<COUNT>(sc, S, K, tc);
        else ray_triangle_step<true, COUNT>(sc, S, K, tc);
    }
    return S.occluded;
}

// ------------------------------------------------------------------------------------------------------------
// Textures: Image::texture_floor -> sample_floor -> offset (image.h:79-97,122-134): nearest texel, clamp to edge.
// float -> int as the reference's host does it (x86 cvttss2si): truncation, and INT_MIN for NaN and for values outside
// the int range -- where CUDA's conversion would saturate (NaN -> 0, +big -> INT_MAX).  Texture coordinates can get
// there (parallax interpolation weight with a zero denominator); the clamp that follows then picks the same texel.
RT_DEV int f2i_x86(float x)
{
#if defined(__CUDACC__)
    return (x >= -2147483648.0f && x < 2147483648.0f) ? (int)x : (int)0x80000000;
#else
    return (int)x;
#endif
}

// Image::operator()(int, int) -> offset (image.h:40-49,122-134): the texel with clamp-to-edge addressing.
RT_DEV Col tex_texel(const TexView& tx, int px, int py)
{
    if (px < 0) px = 0;
    if (px > tx.w - 1) px = tx.w - 1;
    if (py < 0) py = 0;
    if (py > tx.h - 1) py = tx.h - 1;
    size_t idx = (size_t)py * (size_t)tx.w + (size_t)px;
    if (tx.format == 1) {
#if defined(__CUDACC__)
        uchar4 c = __ldg(reinterpret_cast<const uchar4*>(tx.data) + idx);
        const float kk = 1.0f / 255.0f;                      // Color / 255 -> kk = 1 / k; kk * c (color.cpp:87-91)
        return col((float)c.x * kk, (float)c.y * kk, (float)c.z * kk);
#else
        const uint8_t* c = reinterpret_cast<const uint8_t*>(tx.data) + 4 * idx;
        const float kk = 1.0f / 255.0f;
        return col((float)c[0] * kk, (float)c[1] * kk, (float)c[2] * kk);
#endif
    }
    rt_f4 c = RT_LDG4(reinterpret_cast<const rt_f4*>(tx.data) + idx);
    return col(c.x, c.y, c.z);
}

RT_DEV Col tex_floor(const TexView& tx, float x, float y)
{
    float fu = floorf(x * (float)tx.w);
    float fv = floorf(y * (float)tx.h);
    return tex_texel(tx, f2i_x86(fu), f2i_x86(fv));
}

// Image::texture_bilinear -> sample_bilinear (image.h:66-77,89-92): weights from the fractional part, texel indices by
// truncation, the four products summed left to right.
RT_DEV Col tex_bilinear(const TexView& tx, float x, float y)
{
    float sx = x * (float)tx.w, sy = y * (float)tx.h;
    float u = sx - floorf(sx);
    float v = sy - floorf(sy);
    int ix = f2i_x86(sx), iy = f2i_x86(sy);
    return tex_texel(tx, ix, iy) * ((1 - u) * (1 - v)) + tex_texel(tx, ix + 1, iy) * (u * (1 - v)) + tex_texel(tx, ix, iy + 1) * ((1 - u) * v) +
           tex_texel(tx, ix + 1, iy + 1) * (u * v);
}

struct MatView {
    Col ambient_coeff, diffuse, specular, emission;
    float reflection, roughness, ns, specular_threshold;
};

RT_DEV MatView load_material(const SceneView& sc, int32_t index)
{
    const rt_f4* m = sc.mats + 4 * (size_t)index;
    rt_f4 a = RT_LDG4(m), b = RT_LDG4(m + 1), c = RT_LDG4(m + 2), d = RT_LDG4(m + 3);
    MatView mv;
    mv.ambient_coeff = col(a.x, a.y, a.z);
    mv.diffuse = col(a.w, b.x, b.y);
    mv.specular = col(b.z, b.w, c.x);
    mv.emission = col(c.y, c.z, c.w);
    mv.reflection = d.x; mv.roughness = d.y; mv.ns = d.z; mv.specular_threshold = d.w;
    return mv;
}

struct TriShade {       // shading-side triangle data
    V3 tu, tv;          // Triangle::_tex_coords_u / _v (triangle.h:99-103)
    int32_t mat;
    int32_t orig;
};

RT_DEV TriShade load_tri_shade(const SceneView& sc, int32_t tri)
{
    rt_f4 a, b;
    if ((uint32_t)tri >= sc.n_tris) {
        // a clipped piece of raster_trace: written by this very thread a moment ago, so an ordinary (coherent) load
        const rt_f4* s = sc.frag_shade + 2 * (size_t)((uint32_t)tri - sc.n_tris);
        a = s[0]; b = s[1];
    } else {
        const rt_f4* s = sc.shade + 2 * (size_t)tri;
        a = RT_LDG4(s); b = RT_LDG4(s + 1);
    }
    TriShade ts;
    ts.tu = v3(a.x, a.y, a.z);
    ts.tv = v3(a.w, b.x, b.y);
    ts.mat = (int32_t)f4_bits(b.z);
    ts.orig = (int32_t)f4_bits(b.w);
    return ts;
}

// Triangle::interpolate_texcoords -- triangle.cpp:155-160
RT_DEV void tri_texcoords(const TriShade& ts, float u, float v, float& tex_u, float& tex_v)
{
    tex_u = (1 - u - v) * ts.tu.x + u * ts.tu.y + v * ts.tu.z;
    tex_v = (1 - u - v) * ts.tv.x + u * ts.tv.y + v * ts.tv.z;
}

// ------------------------------------------------------------------------------------------------------------
// Analytic shapes: Sphere::intersect / Plane::intersect -- analyticShape.cpp:9-76, every operation as written there
// (a sphere assumes a unit direction: a = 1, also for the un-normalised rays of rough reflections).  A hit record names
// shape i as tri = -2 - i.  Only t, normal and material of a shape hit are ever read: frames with shapes refuse the
// switches that would read the rest of the reference's HitInfo (host_common.h).
RT_DEV bool shape_intersect(const SceneView& sc, int i, V3 o, V3 d, float& t_out, V3& n_out, int32_t& mat_out)
{
    const rt_f4 s0 = RT_LDG4(sc.shapes + 2 * (size_t)i), s1 = RT_LDG4(sc.shapes + 2 * (size_t)i + 1);
    const uint32_t bits = f4_bits(s1.w);
    const V3 a = v3(s0.x, s0.y, s0.z);
    float t;
    if (!(bits & 0x80000000u)) {
        V3 L = o - a;
        float b = 2 * dot(d, L);
        float c = dot(L, L) - s0.w;
        float delta = b * b - 4 * c;                             // a = 1: 4 * a * c
        if (delta < 0) return false;
        if (delta == 0.0f) t = -b / 2;
        else {
            float sq = sqrtf(delta);
            float t1 = (-b - sq) / 2;
            float t2 = (-b + sq) / 2;
            if (!(t1 < t2)) return false;                        // only with NaN / inf input; the reference then reads a stale t
            t = t1;
            if (t < 0) t = t2;
        }
        if (t < 0) return false;
        n_out = normalize((o + t * d) - a);
    } else {
        const V3 n = v3(s1.x, s1.y, s1.z);
        t = dot(a - o, n) / dot(d, n);
        if (t < 0) return false;
        n_out = n;
    }
    t_out = t;
    mat_out = (int32_t)(bits & 0x7fffffffu);
    return true;
}

RT_DEV int32_t shape_material(const SceneView& sc, int i) { return (int32_t)(f4_bits(RT_LDG4(sc.shapes + 2 * (size_t)i + 1).w) & 0x7fffffffu); }

// The shapes half of Renderer::is_shadowed -- renderer.cpp:376-397, for the shadow ray (o, d) of the shaded point p.
RT_DEV bool shapes_occlude_ray(const SceneView& sc, V3 o, V3 d, V3 p, float dist2)
{
    for (int i = 0; i < sc.n_shapes; i++) {
        float t;
        V3 sn;
        int32_t sm;
        if (shape_intersect(sc, i, o, d, t, sn, sm)) {
            V3 q = o + t * d;
            if (length2(p - q) < dist2) return true;
        }
    }
    return false;
}

RT_DEV bool shapes_occlude(const SceneView& sc, V3 p, V3 n, V3 light)
{
    // ray origin p + n * EPSILON (renderer.h:23), direction normalize(light - p) -- renderer.cpp:344
    return shapes_occlude_ray(sc, p + 1.0e-4f * n, normalize(light - p), p, length2(p - light));
}

// Fills the HitInfo fields Triangle::intersect sets on a hit (triangle.cpp:81-88): material, normalised normal,
// tangent (Triangle::get_tangent, triangle.cpp:134-153).
RT_DEV Hit complete_hit(const SceneView& sc, const HitRec& hr)
{
    Hit h;
    h.tri = hr.tri; h.t = hr.t; h.u = hr.u; h.v = hr.v;
    const rt_f4* tp = sc.tris + 3 * (size_t)hr.tri;
    rt_f4 p0 = RT_LDG4(tp), p1 = RT_LDG4(tp + 1), p2 = RT_LDG4(tp + 2);
    V3 a = v3(p0.x, p0.y, p0.z);
    V3 ab = v3(p1.x, p1.y, p1.z) - a;
    V3 ac = v3(p2.x, p2.y, p2.z) - a;
    TriShade ts = load_tri_shade(sc, hr.tri);
    float du1 = ts.tu.y - ts.tu.x, dv1 = ts.tv.y - ts.tv.x;
    float du2 = ts.tu.z - ts.tu.x, dv2 = ts.tv.z - ts.tv.x;
    float f = 1.0f / (du1 * dv2 - du2 * dv1);
    h.tangent = v3(f * (dv2 * ab.x - dv1 * ac.x), f * (dv2 * ab.y - dv1 * ac.y), f * (dv2 * ab.z - dv1 * ac.z));
    h.mat = ts.mat;
    h.normal = normalize(v3(p0.w, p1.w, p2.w));
    return h;
}

// The hit record of a ray (origin o, direction d) as a Hit: a triangle (complete_hit) or analytic shape -2 - tri, whose
// normal is recomputed from the ray exactly as Sphere::intersect / Plane::intersect computed it.
RT_DEV Hit make_hit(const SceneView& sc, const HitRec& hr, V3 o, V3 d)
{
    if (hr.tri >= 0) return complete_hit(sc, hr);
    Hit h = fresh_hit();
    h.tri = hr.tri; h.t = hr.t;
    float t;
    shape_intersect(sc, -2 - hr.tri, o, d, t, h.normal, h.mat);
    return h;
}

RT_DEV void hit_texcoords(const SceneView& sc, const Hit& h, float u, float v, float& tu, float& tv)
{
    TriShade ts = load_tri_shade(sc, h.tri);            // Renderer::get_tex_coords, renderer.cpp:436-445
    tri_texcoords(ts, u, v, tu, tv);
}

// Renderer::normal_mapping -- renderer.cpp:464-478
RT_DEV V3 normal_mapping(const SceneView& sc, const Hit& h, float u, float v)
{
    float tu, tv;
    hit_texcoords(sc, h, u, v, tu, tv);
    V3 tg = h.tangent;
    V3 bt = cross(tg, h.normal);
    Col nc = tex_floor(sc.tex[RT_TEX_NORMAL], tu, tv);
    V3 nm = 2.0f * v3(nc.r, nc.g, nc.b) - v3(1, 1, 1);
    V3 q = normalize(nm);
    V3 pn = v3(tg.x * q.x + bt.x * q.y + h.normal.x * q.z,      // Transform(T,B,N)(Vector), mat.cpp:69-75,103-115
               tg.y * q.x + bt.y * q.y + h.normal.y * q.z,
               tg.z * q.x + bt.z * q.y + h.normal.z * q.z);
    return normalize(pn);
}

// Renderer::parallax_occlusion_mapping -- renderer.cpp:518-554.  Marches the displacement map along the view
// direction's (x, y) in `parallax_mapping_steps` layers, then interpolates between the last two layers.  As in the
// reference, (new_u, new_v) are TEXTURE coordinates that the caller nevertheless hands to the mapping functions as if
// they were barycentrics (renderer.cpp:567-585); parity keeps that.
RT_DEV void parallax_occlusion_mapping(const SceneView& sc, const FrameView& fr, const Hit& h, float u, float v, V3 view_dir, float& new_u,
                                       float& new_v)
{
    const TexView& dm = sc.tex[RT_TEX_DISPLACEMENT];
    float tu, tv;
    hit_texcoords(sc, h, u, v, tu, tv);
    float current_depth;
    float depth_step = 1.0f / fr.s.parallax_mapping_steps;
    float sampled_depth = tex_floor(dm, tu, tv).r;
    V3 search_direction = fr.s.displacement_mapping_strength * (-view_dir);       // -view_dir * strength (Vector * float, vec.cpp:98-101)
    float delta_u = search_direction.x / fr.s.parallax_mapping_steps;
    float delta_v = search_direction.y / fr.s.parallax_mapping_steps;
    current_depth = 0.0f;
    new_u = tu;
    new_v = tv;
    while (current_depth < sampled_depth) {
        new_u += delta_u;
        new_v += delta_v;
        sampled_depth = tex_floor(dm, new_u, new_v).r;
        current_depth += depth_step;
    }
    float previous_u = new_u - delta_u;
    float previous_v = new_v - delta_v;
    float after_depth = sampled_depth - current_depth;
    float before_depth = tex_floor(dm, previous_u, previous_v).r - (current_depth - depth_step);
    float w = after_depth / (after_depth - before_depth);
    new_u = (1 - w) * new_u + w * previous_u;
    new_v = (1 - w) * new_v + w * previous_v;
}

// Renderer::compute_specular -- renderer.cpp:270-280
RT_DEV Col compute_specular(const MatView& m, V3 ray_dir, V3 n, V3 to_light)
{
    V3 half = normalize(to_light - ray_dir);
    float angle = dot(half, n);
    if (angle <= m.specular_threshold) return col(0.0f);
    float p = powf(fmaxf(0.0f, angle), m.ns);
    return m.specular * col(p);
}

// The part of Renderer::shade_ray_inter_point (renderer.cpp:556-617) that needs no further rays:
// diffuse * ao * enable_diffuse + specular * enable_specular, evaluated after the normal-map update of hit.normal.
RT_DEV Col shade_direct(const SceneView& sc, const FrameView& fr, V3 ro, V3 rd, Hit& hit, V3& p_out, MatView& m_out)
{
    const RtSettings& s = fr.s;
    float u = hit.u, v = hit.v;
    V3 p = ro + hit.t * rd;
    if (s.enable_displacement_mapping) parallax_occlusion_mapping(sc, fr, hit, hit.u, hit.v, normalize(fr.cam_pos - p), u, v);
    V3 to_light = normalize(fr.light - p);
    if (s.enable_normal_mapping) hit.normal = normal_mapping(sc, hit, u, v);
    MatView m = load_material(sc, hit.mat);
    float ao = 1.0f;
    if (s.enable_ao_mapping) {
        float tu, tv;
        hit_texcoords(sc, hit, u, v, tu, tv);
        ao = tex_floor(sc.tex[RT_TEX_AO], tu, tv).r;
    }
    Col diffuse;
    if (s.enable_diffuse_mapping) {
        float tu, tv;
        hit_texcoords(sc, hit, u, v, tu, tv);
        diffuse = tex_floor(sc.tex[RT_TEX_DIFFUSE], tu, tv);
        diffuse = diffuse * col(fmaxf(0.5f, dot(hit.normal, normalize(fr.cam_pos - p))));
    } else
        diffuse = m.diffuse * col(fmaxf(0.0f, dot(hit.normal, to_light)));          // compute_diffuse :263-266
    Col c = col(0.0f);
    c = c + diffuse * ao * (s.enable_diffuse ? 1.0f : 0.0f);
    c = c + compute_specular(m, rd, hit.normal, to_light) * (s.enable_specular ? 1.0f : 0.0f);
    p_out = p;
    m_out = m;
    return c;
}

// The rest of shade_ray_inter_point once the shadow flag and the reflection colour are known (renderer.cpp:591-597,
// 612-616) and the second clamp of trace_ray (renderer.cpp:1045-1047, idempotent).
RT_DEV Col shade_compose(const FrameView& fr, const MatView& m, Col direct, bool shadowed, Col reflection)
{
    const RtSettings& s = fr.s;
    Col c = direct;
    if (shadowed) c = c * col(0.5f);                                                // SHADOW_INTENSITY, renderer.h:24
    c = c + m.emission * (s.enable_emissive ? 1.0f : 0.0f);
    if (m.reflection > 0.0f) c = c + reflection * m.reflection;
    c = c + col(0.1f) * m.ambient_coeff * (1 - m.reflection) * (s.enable_ambient ? 1.0f : 0.0f); // AMBIENT_COLOR :18
    return col(clamp01(c.r), clamp01(c.g), clamp01(c.b));
}

// The debug shading modes of shade_ray_inter_point (renderer.cpp:599-609, 404-434).
RT_DEV Col shade_debug(const SceneView& sc, const FrameView& fr, const Hit& hit)
{
    Col c = col(0.0f);
    int mode = fr.s.shading_method;
    if (mode == RT_ABS_NORMALS_SHADING)
        c = col(fabsf(hit.normal.x), fabsf(hit.normal.y), fabsf(hit.normal.z));
    else if (mode == RT_PASTEL_NORMALS_SHADING)
        c = (col(hit.normal.x, hit.normal.y, hit.normal.z) + col(1.0f)) * 0.5f;
    else if (mode == RT_BARYCENTRIC_COORDINATES_SHADING)
        c = col(1, 0, 0) * hit.u + col(0, 1, 0) * hit.v + col(0, 0, 1) * (1 - hit.u - hit.v);
    else if (mode == RT_VISUALIZE_AO) {
        c = col(0.9f);
        if (fr.s.enable_ao_mapping) {
            float tu, tv;
            hit_texcoords(sc, hit, hit.u, hit.v, tu, tv);
            c = c * col(tex_floor(sc.tex[RT_TEX_AO], tu, tv).r);
        }
    }
    return col(clamp01(c.r), clamp01(c.g), clamp01(c.b));
}

// Skybox::sample -- renderer/skybox.cpp:12-51: the face the direction (z flipped) points at, the face coordinates, one
// bilinear tap.  The reference's `0.5` literals are doubles: norm_factor = float(0.5 / double(|axis|)) and
// u = float(double(u * norm_factor) + 0.5); so here.
RT_DEV Col skybox_sample(const SceneView& sc, V3 dir)
{
    const V3 d2 = v3(dir.x, dir.y, -dir.z);
    const V3 a = v3(fabsf(d2.x), fabsf(d2.y), fabsf(d2.z));
    int face;
    float nf, u, v;
    if (a.z >= a.x && a.z >= a.y) {
        face = d2.z < 0.0f ? 4 : 5;
        nf = (float)(0.5 / (double)a.z);
        u = d2.z < 0.0f ? -d2.x : d2.x;
        v = -d2.y;
    } else if (a.y >= a.x) {
        face = d2.y < 0.0f ? 3 : 2;
        nf = (float)(0.5 / (double)a.y);
        u = d2.x;
        v = d2.y < 0.0f ? -d2.z : d2.z;
    } else {
        face = d2.x < 0.0f ? 1 : 0;
        nf = (float)(0.5 / (double)a.x);
        u = d2.x < 0.0f ? d2.z : -d2.z;
        v = -d2.y;
    }
    u = (float)((double)(u * nf) + 0.5);
    v = (float)((double)(v * nf) + 0.5);
    return tex_bilinear(sc.tex[RT_TEX_SKYBOX_RIGHT + face], u, v);
}

// Miss shader of trace_ray -- renderer.cpp:1052-1065: skysphere, else cube-map skybox, else BACKGROUND_COLOR.  The
// reference mixes float libm calls with double constants; so does this.
RT_DEV Col shade_miss(const SceneView& sc, const FrameView& fr, V3 rd)
{
    if (fr.s.enable_skysphere) {
        float u = (float)(0.5 + (double)atan2f(-rd.z, -rd.x) / (2 * 3.14159265358979323846));
        float v = (float)(0.5 + (double)asinf(-rd.y) / 3.14159265358979323846);
        return tex_floor(sc.tex[RT_TEX_SKYSPHERE], u, v);
    }
    if (fr.s.enable_skybox) return skybox_sample(sc, rd);                           // renderer.cpp:1061-1062
    return col(135.0f / 255.0f, 206.0f / 255.0f, 235.0f / 255.0f);                  // renderer.cpp:19
}

// Does the miss colour depend on the ray (else it is the constant background)?
RT_DEV bool miss_needs_ray(const FrameView& fr) { return fr.s.enable_skysphere || fr.s.enable_skybox; }

template <bool COUNT>
RT_DEV_NOINLINE Col trace_ray_secondary(const SceneView& sc, const FrameView& fr, V3 ro, V3 rd, Hit& final_hit,
                                       int depth, XorShift32& rng, TraceCounters* tc);

// Renderer::compute_reflection -- renderer.cpp:283-338.  One thread walks the whole fan in order: the reference's
// random stream (3 draws per rough sample, consumed also by nested fans that are cut off by the recursion limit)
// and its reflection_hit_info (declared OUTSIDE the sample loop, :286, so sample k is shaded with the closest hit
// seen by samples 1..k) are both sequential by construction.  Returns colour already multiplied by
// material.reflection once (:337); the caller multiplies again (:595).
template <bool COUNT>
RT_DEV Col compute_reflection(const SceneView& sc, const FrameView& fr, V3 rd, V3 p, const Hit& hit, const MatView& m,
                             int depth, XorShift32& rng, TraceCounters* tc)
{
    const RtSettings& s = fr.s;
    Hit rh = fresh_hit();
    V3 n = hit.normal;
    V3 origin = p + 0.01f * n;
    V3 mirror = rd - (2 * dot(rd, n)) * n;
    int samples = 0;
    Col total = col(0.0f);
    for (int i = 0; i < s.rough_reflections_sample_count; i++) {
        float roughness;
        if (s.enable_roughness_mapping) {
            float tu, tv;
            hit_texcoords(sc, hit, hit.u, hit.v, tu, tv);
            roughness = tex_floor(sc.tex[RT_TEX_ROUGHNESS], tu, tv).r;
        } else
            roughness = m.roughness;
        if (roughness > 0) {
            // Vector(rand, rand, rand), renderer.cpp:313: the compiled reference (g++) evaluates right to left.
            float rz = rng.bilateral();
            float ry = rng.bilateral();
            float rx = rng.bilateral();
            V3 r = normalize(v3(rx, ry, rz));
            if (dot(r, hit.normal) < 0) r = -r;
            V3 dir = roughness * r + (1 - roughness) * mirror;
            total = total + trace_ray_secondary<COUNT>(sc, fr, origin, dir, rh, depth + 1, rng, tc);
            samples++;
        } else {
            total = total + trace_ray_secondary<COUNT>(sc, fr, origin, mirror, rh, depth + 1, rng, tc);
            samples = 1;
            break;
        }
    }
    return total / col((float)samples) * col(m.reflection);
}

// Renderer::trace_ray for depth >= 1 (renderer.cpp:1008-1066) with shade_ray_inter_point inlined; recursion as in
// the reference, bounded by max_recursion_depth (the C ABI caps it so the device stack can be sized).
template <bool COUNT>
RT_DEV_NOINLINE Col trace_ray_secondary(const SceneView& sc, const FrameView& fr, V3 ro, V3 rd, Hit& final_hit, int depth,
                                       XorShift32& rng, TraceCounters* tc)
{
    if (depth > fr.s.max_recursion_depth) return col(0.0f);
    if (tc) tc->refl_rays++;
    HitRec hr;
    if (trace_closest<COUNT>(sc, ro, rd, hr, tc)) {
        if (hr.t < final_hit.t || final_hit.t == -1.0f) final_hit = complete_hit(sc, hr);
    }
    for (int i = 0; i < sc.n_shapes; i++) {                                          // renderer.cpp:1029-1037
        float t;
        V3 sn;
        int32_t sm;
        if (shape_intersect(sc, i, ro, rd, t, sn, sm) && (t < final_hit.t || final_hit.t == -1.0f)) {
            final_hit.tri = -2 - i; final_hit.t = t; final_hit.normal = sn; final_hit.mat = sm;
        }
    }
    if (final_hit.t > 0.1f) {                                                        // min_t, renderer.cpp:1039
        if (fr.s.shading_method != RT_SHADING) return shade_debug(sc, fr, final_hit);
        V3 p;
        MatView m;
        Col direct = shade_direct(sc, fr, ro, rd, final_hit, p, m);
        bool shadowed = false;
        if (fr.s.compute_shadows) {
            if (tc) tc->refl_shadow_rays++;
            shadowed = trace_occluded<COUNT>(sc, p, final_hit.normal, fr.light, tc) || (sc.n_shapes > 0 && shapes_occlude(sc, p, final_hit.normal, fr.light));
        }
        Col refl = col(0.0f);
        if (m.reflection > 0.0f) refl = compute_reflection<COUNT>(sc, fr, rd, p, final_hit, m, depth, rng, tc);
        return shade_compose(fr, m, direct, shadowed, refl);
    }
    return shade_miss(sc, fr, rd);
}

// Primary ray of pixel (px, py) of the supersampled frame -- renderer.cpp:1083-1098.
RT_DEV void primary_ray(const FrameView& fr, int px, int py, V3& o, V3& d)
{
    float yw = ((float)py + 0.5f) / (float)fr.rh * 2 - 1;
    float xw = ((float)px + 0.5f) / (float)fr.rw * 2 - 1;
    V3 vs = xform_point(fr.proj_inv, v3(xw, yw, -1));
    V3 ws = xform_point(fr.cam_to_world, vs);
    o = fr.cam_pos;
    d = normalize(ws - fr.cam_pos);
}

} // namespace rtb
