// kernels.cuh -- the wavefront pipeline's __global__ kernels (sm_100a).  One frame (rt_render_device_begin, rtb200.cu):
//
//   host               tiles outside the screen-space bound of the scene's root box are set aside: they get no ray slots
//   k_fill_miss        ... only the miss colour (background / skysphere / cube-map skybox)
//   per chunk of the other tiles (two chunks in flight on two streams, RT_OPT_LANES):
//     k_primary_packet ray generation + closest hit, 32 rays (an 8x4 pixel block) per warp in ONE traversal with a
//                      shared-memory stack; misses are shaded and stored at once, hit records go to dense per-slot arrays
//     k_primary_items  x6, k_primary_finish: the packets that ran out of rounds, split into work items (short launches)
//     k_compact        turns the per-slot hit records into the hit queue, block by block in slot order, so that 32
//                      consecutive queue entries are 32 neighbouring pixels (coherent shadow packets); also the
//                      reflection queue
//     k_reflect        (only if a material reflects) one thread per reflective hit walks its rough-reflection fan
//     k_shade_packet   32 queued hits per warp: textures / Blinn-Phong, any-hit shadow packet, compose, quantise, store
//     k_shade_items    x6, k_shade_finish: the shadow packets that ran out of rounds, split into work items
//   k_resolve          integer SSAA box filter of the quantised samples (imageUtils.h:98-147)
//
// plus the single-ray kernels k_primary / k_shade (RT_OPT_PACKETS 0: one traversal state machine per lane with lane
// refill; they count the reference-shaped work for the roofline), the batch kernels behind rt_intersect / rt_occluded /
// rt_generate_primary_rays and the tile pack / unpack of the framebuffer gather.
// Nothing here is a dense contraction, so no tensor-core path; the kernels are bound by fp32 issue and L2 latency on
// node/triangle fetches (DESIGN.md section 5).
#pragma once

#include <cuda_runtime.h>
#include "rt_device.h"

namespace rtb {

constexpr int kPatch = 8;            // a warp's work item is a kPatch x kPatch block of supersampled pixels (2 passes of 8x4)
constexpr int kPrimaryThreads = 128;
constexpr int kQueueThreads = 128;
constexpr int kPrimaryFetch = 1;     // 32-ray packets a warp of k_primary_packet takes per atomic (4: -4 %, coarser load balance)
constexpr int kStepsPerCheck = 4;    // single-test steps between two refill / completion checks of a persistent single-ray warp
constexpr unsigned kParkCtas = 296;  // fused item scheduling: the warps of this many CTAs (the first waves: about two CTAs per SM) stay to serve late items
constexpr unsigned kFusedGenerations = 12;   // ... an item of this generation is traced to the end (no round budget)
constexpr int kItemPasses = 6;       // generations of work items of a split packet = launches of k_*_items; the last has no round
                                     // budget (3 left a straggler in the unlimited pass: k_shade 8.9 ms against 8.0 with 6; 10: same)
#ifndef RTB_SHADE_MINB
#define RTB_SHADE_MINB 7   /* resident CTAs per SM the compiler must allow for k_shade_packet; measured on cfg4: 7 -> 8.9 ms, 6: 9.4, 8: 9.6 */
#endif

// Fused item scheduling: the item queue of a stage is kSubQueues independent ticket queues, each with its counters on a
// 128-byte line of its own (= an L2 slice of its own).  One queue polled and compare-and-swapped by every warp of the grid
// after every packet is a single hot address: the L2 serves a few hundred million operations per second on one line, the
// grid asks for billions, and the launch slows down tenfold (measured).  A warp emits into and polls its HOME queue;
// only a warp that has run out of packets looks at all of them (one load per lane, in parallel).
constexpr int kSubQueues = 32;
struct alignas(128) SubQueue {
    unsigned int n;                  // tickets reserved in this sub-queue
    unsigned int next;               // tickets handed out
    unsigned int pad[30];
};
struct alignas(16) FusedTotals {     // termination: read packets_done, then done, then reserved
    unsigned int reserved;           // real items published, all sub-queues
    unsigned int done;               // items completed
    unsigned int packets_done;       // packets completed (reported per warp when it runs out of packets)
    unsigned int pad;
};

struct ChunkCounters {               // one per chunk, zeroed before the frame
    unsigned int next_patch;         // next ray slot of k_primary
    unsigned int next_shade;         // next hit-queue entry of k_shade
    unsigned int n_hits;
    unsigned int n_refl;
    unsigned int stack_overflow;
    unsigned int n_split;            // shadow packets that ran out of rounds and were split into work items
    unsigned int items_n[kItemPasses];    // work items written for item pass p (each: one unvisited cell of a split packet)
    unsigned int items_next[kItemPasses]; // next item of pass p to take
    unsigned int p_split, p_items_n[kItemPasses], p_items_next[kItemPasses];   // the same for split PRIMARY packets
    // fused item scheduling (Tuning::fused): [0] primary stage, [1] shade stage
    SubQueue sq[2][kSubQueues];
    FusedTotals ft[2];
    unsigned long long refl_rays;
    unsigned long long refl_shadow_rays;
    // COUNT instantiations only: volume / triangle tests done by the traversal, per ray class
    unsigned long long primary_vol, primary_tri, shadow_vol, shadow_tri, refl_vol, refl_tri;
    unsigned long long primary_fetch, shadow_fetch, refl_fetch;   // bytes fetched for those tests: 64 per child record, 48 per triangle
    unsigned long long traced_primary;                            // primary rays that really were traced (always maintained)
    // COUNT instantiations of the packet kernels only: cell/leaf rounds per packet, [0] primary, [1] shadow
    unsigned int rounds_hist[2][16]; // bucket b: packets with 2^b <= rounds < 2^(b+1) (bucket 0 also holds 0 rounds)
    unsigned int max_rounds[2];
    unsigned long long max_packet_ns[2], sum_packet_ns[2];
};

RT_DEV unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// one lane per warp: tallies of one traced packet (diagnostics of the COUNT instantiations)
RT_DEV void note_packet(ChunkCounters* cnt, int which, unsigned rounds, unsigned long long ns)
{
    const int b = rounds ? min(31 - __clz(rounds), 15) : 0;
    atomicAdd(&cnt->rounds_hist[which][b], 1u);
    atomicMax(&cnt->max_rounds[which], rounds);
    atomicMax(&cnt->max_packet_ns[which], ns);
    atomicAdd(&cnt->sum_packet_ns[which], ns);
}

RT_DEV void flush_work(TraceCounters& tc, unsigned long long* vol, unsigned long long* tri, unsigned long long* fetch)
{
    // warp-aggregated: one atomic triple per warp
    unsigned long long v = tc.vol_tests, t = tc.tri_tests, f = 64ull * tc.rec_fetch + 48ull * tc.tri_fetch;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v += __shfl_xor_sync(0xffffffffu, v, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
        f += __shfl_xor_sync(0xffffffffu, f, o);
    }
    if ((threadIdx.x & 31u) == 0) {
        if (v) atomicAdd(vol, v);
        if (t) atomicAdd(tri, t);
        if (f) atomicAdd(fetch, f);
    }
}

// Which part of the frame a launch covers: owned tiles [tile_begin, tile_end) of the shard's tile list.
struct WorkView {
    const uint32_t* tiles;           // indices into the tiles_x * tiles_y grid of final-resolution tiles
    uint32_t tile_begin, tile_end;
    int32_t tiles_x;
    int32_t tile_px;                 // tile side in supersampled pixels (tile_size * factor)
    int32_t patches_per_side;        // ceil(tile_px / kPatch)
    // The scene's screen coverage (host side, screen_coverage): bit bx % 32 of word by * cover_words + bx / 32 is set when the
    // rays of the 8x4 block (bx, by) of supersampled pixels can hit the scene.  Null when no bound exists: every block can.
    const uint32_t* cover;
    int32_t cover_words;
};

struct QueueView {
    // dense, one per ray slot of the chunk (slot = position in patch order, see slot_pixel)
    int32_t* slot_tri;               // leaf-order triangle of the closest hit, -1 = miss / no ray
    float* slot_t;                   // valid where slot_tri >= 0
    float* slot_u;
    float* slot_v;
    // compacted by k_compact
    uint32_t* hit_slot;              // hit queue: ray slots of the hits
    // light-space order of the hit queue (k_sort_*): sort_mode 0 = off, 1 = always, 2 = when fewer than a quarter of the
    // chunk's sort_slots ray slots are hits (sparse hits = hits at unrelated depths); the shade stage reads hit_sorted then
    uint32_t* hit_sorted;
    uint32_t sort_mode, sort_slots;
    // G-buffers of the SSAO post-process (ssao.cuh), one entry per supersampled pixel; null when SSAO is off
    float* g_z;
    V3* g_n;
    // split shadow packets (k_shade_packet -> k_shade_items -> k_shade_finish)
    uint32_t* split_base;            // first hit-queue entry of the packet
    uint32_t* split_active;          // lanes that had no answer when the packet was split
    uint32_t* split_occ;             // lanes found occluded since (atomicOr by the items)
    uint4* items;                    // kItemPasses regions of item_capacity: (split index, link, meta, -)
    uint32_t split_capacity, item_capacity;
    // fused item scheduling: items[] is one queue of kItemPasses * item_capacity slots; slot i is valid once item_ready[i] == tag
    // (tag differs per frame and stage, so the flags never need clearing); split_pending[sidx] counts the record's items that
    // have not completed yet -- the warp that brings it to zero stores the record's pixels / slot records
    uint32_t* item_ready;
    uint32_t* split_pending;
    uint32_t tag;
    // split primary packets (k_primary_packet -> k_primary_items -> k_primary_finish); item regions are shared with the
    // shadow packets (the two never run at the same time), split_base / split_active too
    unsigned long long* split_best;  // 32 per split record: bits(t) << 32 | original triangle index of the closest hit so far (atomicMin)
    uint32_t* refl_idx;              // reflection queue: indices into the hit queue
    float* refl_rgb;                 // 3 floats per hit-queue entry, written by k_reflect
    unsigned long long* refl_cnt;    // 3 words per hit-queue entry, written by k_reflect: rays | shadow rays << 32, V, T
    uint32_t capacity;
};

// Ray slot -> pixel of the supersampled frame.  Slots enumerate the chunk's tiles, inside a tile its 8x8 patches
// row-major, inside a patch its pixels row-major, so 32 consecutive slots are an 8x4 pixel block.  Returns false for
// slots that hang over the tile or frame edge.
RT_DEV bool slot_pixel(const WorkView& wk, const FrameView& fr, uint32_t slot, int& px, int& py)
{
    const uint32_t pps = (uint32_t)wk.patches_per_side;
    const uint32_t per_tile = pps * pps * (uint32_t)(kPatch * kPatch);
    const uint32_t tile = wk.tiles[wk.tile_begin + slot / per_tile];
    const uint32_t in_tile = slot % per_tile;
    const uint32_t patch = in_tile / (uint32_t)(kPatch * kPatch), in_patch = in_tile % (uint32_t)(kPatch * kPatch);
    const int lx = (int)(patch % pps) * kPatch + (int)(in_patch & 7u);
    const int ly = (int)(patch / pps) * kPatch + (int)(in_patch >> 3);
    px = (int)(tile % (uint32_t)wk.tiles_x) * wk.tile_px + lx;
    py = (int)(tile / (uint32_t)wk.tiles_x) * wk.tile_px + ly;
    return lx < wk.tile_px && ly < wk.tile_px && px < fr.rw && py < fr.rh;
}

// The 8x4 block of supersampled pixel (px, py) may hold a hit (WorkView::cover).  The 32 lanes of a packet whose block is
// aligned to the 8x4 grid read one word.
RT_DEV bool covered(const WorkView& wk, int px, int py)
{
    if (wk.cover == nullptr) return true;
    const uint32_t w = __ldg(wk.cover + ((uint32_t)py >> 2) * (uint32_t)wk.cover_words + ((uint32_t)px >> 8));
    return ((w >> (((uint32_t)px >> 3) & 31u)) & 1u) != 0u;
}

// Refill thresholds of the persistent kernels: a warp fetches new rays when at least this many of its lanes are idle
// (and always when all are).  Low = lanes never idle long but the per-ray set-up code runs with few lanes; high = the
// opposite.  Set through rt_set_option for experiments.
struct Tuning {
    int32_t primary_refill;
    int32_t shade_refill;
    int32_t tri_batch;        // run the triangle phase once this many lanes wait for it (or nothing else can run)
    int32_t packets;          // 1: primary and shadow rays are traced as 32-ray packets (k_primary_packet / k_shade_packet)
    int32_t packet_rounds;    // a shadow packet that needs more cell/leaf rounds than this is split into work items (0: never)
    int32_t item_rounds;      // the same for the items of all passes but the last
    int32_t primary_rounds;   // round budget of a primary packet (0: never split)
    int32_t fused;            // 1: the packet kernels consume the work items of their split packets themselves (one launch per stage);
                              // 0: item passes and a finish kernel are separate launches (k_*_items x kItemPasses, k_*_finish)
    // adaptive budgets (the defaults): a packet / item that has done at least *_min rounds is also split as soon as its
    // launch's work queue has been handed out completely -- from then on it would only lengthen the launch's tail, whereas its
    // unvisited cells can be traced by the warps that have nothing left to do.  0: the budgets above are all there is.
    int32_t packet_min, item_min, primary_min;
    int32_t item_passes;      // generations of work items actually launched (<= kItemPasses); the last has no budget
    int32_t cull;             // bounding-pyramid cull of a cell's children (packet_set_cull): bit 0 primary packets, bit 1 shadow packets
};

// When a packet should give up before its round budget: the launch's queue (`counter` = tickets handed out, `total` =
// tickets there are) is drained and the packet has done `min_rounds` rounds.  Looked at every 16th round.
struct Drain {
    const unsigned int* counter;
    uint32_t total;
    int min_rounds;
};
RT_DEV Drain no_drain() { Drain d; d.counter = nullptr; d.total = 0u; d.min_rounds = 0; return d; }
RT_DEV Drain make_drain(const unsigned int* counter, uint32_t total, int min_rounds)
{
    Drain d; d.counter = min_rounds > 0 ? counter : nullptr; d.total = total; d.min_rounds = min_rounds; return d;
}

// One scheduling round of a persistent warp: either every lane that sits in a cell tests one child record, or every
// lane that sits in a leaf tests one triangle.  Triangle tests are postponed until `tri_batch` lanes want one.
template <bool ANY, bool COUNT>
RT_DEV void warp_step(const SceneView& sc, RayState& S, RayStack& K, TraceCounters* tc, bool alive, const Tuning& tune)
{
    const unsigned want_c = __ballot_sync(0xffffffffu, alive && S.mode == RT_MODE_CHILDREN);
    const unsigned want_t = __ballot_sync(0xffffffffu, alive && S.mode == RT_MODE_TRIANGLES);
    if (want_c != 0u && __popc(want_t) < tune.tri_batch) {
        if (alive && S.mode == RT_MODE_CHILDREN) ray_child_step<COUNT>(sc, S, K, tc);
    } else if (want_t != 0u) {
        if (alive && S.mode == RT_MODE_TRIANGLES) ray_triangle_step<ANY, COUNT>(sc, S, K, tc);
    }
}

// Ray generation + closest hit.  Persistent warps; every lane owns one ray at a time and steps it through the
// traversal state machine (rt_device.h); lanes whose ray has ended are refilled from an atomic ray-slot counter with
// the next slots in patch order, so a warp starts on 32 adjacent pixels and stays on nearby ones.  Misses are shaded
// and stored at once; the hit record of every slot goes to the dense slot arrays (k_compact makes the queue).
template <bool COUNT>
__global__ void __launch_bounds__(kPrimaryThreads)
k_primary(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t pps = (uint32_t)wk.patches_per_side;
    const uint32_t total = (wk.tile_end - wk.tile_begin) * pps * pps * (uint32_t)(kPatch * kPatch);   // ray slots of the chunk
    TraceCounters tc = zero_counters();
    RayState S;
    RayStack K;
    S.mode = RT_MODE_DONE;
    bool alive = false, exhausted = false;
    int px = 0, py = 0;
    uint32_t slot = 0, traced = 0;
    V3 dir = v3(0, 0, 0);
    for (;;) {
        // ---- refill the idle lanes
        const unsigned idle = __ballot_sync(0xffffffffu, !alive);
        const int n_idle = __popc(idle);
        if (!exhausted && (n_idle >= tune.primary_refill || n_idle == 32)) {
            uint32_t base = 0;
            const int leader = __ffs(idle) - 1;
            if ((int)lane == leader) base = atomicAdd(&cnt->next_patch, (unsigned)n_idle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + (uint32_t)n_idle >= total) exhausted = true;
            const uint32_t r = base + (uint32_t)__popc(idle & lt_mask);
            if (!alive && r < total) {
                slot = r;
                if (slot_pixel(wk, fr, slot, px, py)) {
                    V3 o;
                    primary_ray(fr, px, py, o, dir);
                    closest_begin<COUNT>(sc, o, dir, S, &tc);
                    alive = true;
                    ++traced;
                } else
                    q.slot_tri[slot] = -1;
            }
        }
        if (__ballot_sync(0xffffffffu, alive) == 0u) {
            if (exhausted) break;
            continue;
        }
        // ---- a few single-test steps: slab tests for the lanes inside a cell, triangle tests for those inside a leaf
#pragma unroll 1
        for (int it = 0; it < kStepsPerCheck; it++) warp_step<false, COUNT>(sc, S, K, &tc, alive, tune);
        // ---- rays that have ended
        if (alive && S.mode == RT_MODE_DONE) {
            alive = false;
            const bool hit = closest_found(S) && S.best.t > 0.1f;          // min_t, renderer.cpp:1039-1040
            if (hit) {
                q.slot_tri[slot] = S.best.tri; q.slot_t[slot] = S.best.t; q.slot_u[slot] = S.best.u; q.slot_v[slot] = S.best.v;
            } else {
                q.slot_tri[slot] = -1;
                if (sc.n_shapes > 0) q.slot_t[slot] = closest_found(S) ? S.best.t : -1.0f;   // see k_primary_shapes
                super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, dir));
            }
        }
    }
    if (tc.stack_overflow) atomicOr(&cnt->stack_overflow, 1u);
    traced = __reduce_add_sync(0xffffffffu, traced);
    if (lane == 0 && traced) atomicAdd(&cnt->traced_primary, (unsigned long long)traced);
    if (COUNT) flush_work(tc, &cnt->primary_vol, &cnt->primary_tri, &cnt->primary_fetch);
}

// ---------------------------------------------------------------------------------------------------------------------
// 32-ray packets.  Primary rays of an 8x4 pixel block (2x1 final pixels at 16 spp) and the shadow rays of 32 neighbouring
// hits walk almost the same cells, so the warp traverses ONCE for all of them: one shared stack per warp (shared
// memory), every lane tests the same record / triangle for its own ray, a cell is entered if ANY lane hits it (ballot),
// ordered by the smallest entry distance of the warp (shuffle-min), and dropped at pop time when no lane can still beat
// its own best hit there.  Control flow is warp-uniform: no divergence inside the tests, one broadcast fetch per record.
// Per ray the result is the same exact closest hit (or occlusion flag): a lane only ever sees extra candidates.
// Incoherent rays (reflection fans, arbitrary batches) keep the per-ray state machine above.
struct PacketStack {
    int saved;                      // entries [0, saved) are the unvisited cells of a packet that ran out of rounds
    float4 plane[4];                // the packet's bounding pyramid (packet_set_cull): inside = x * n.x + y * n.y + z * n.z - w >= 0
    float4 stage[32];               // the cell (<= 8 records) or leaf chunk (<= 10 triangles) being tested, 512 bytes
    float t[RT_STACK_SIZE];
    uint32_t link[RT_STACK_SIZE];
    uint32_t meta[RT_STACK_SIZE];
};

// Minimum over the warp (no NaNs on this path): floats map to unsigned keys that sort the same way, so ONE redux.sync
// replaces five dependent shuffle + min steps.
RT_DEV float warp_min(float x)
{
    const uint32_t b = __float_as_uint(x);
    const uint32_t key = b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);
    const uint32_t m = __reduce_min_sync(0xffffffffu, key);
    return __uint_as_float(m ^ ((m & 0x80000000u) ? 0x80000000u : 0xffffffffu));
}

// The bounding pyramid of a packet whose rays all leave from (or arrive at) one point: the primary rays of a pixel block
// from the camera, the shadow rays of neighbouring hits towards the point light.  Axis = the first active lane's direction
// from the apex; every lane's direction in the tangent plane of that axis; the warp's min / max give a rectangle there,
// its four sides four planes through the apex.  A cell's child whose axis-aligned box (its first three slabs) lies outside
// one of them cannot be hit by any ray of the packet: packet_trace drops such children with ONE pass in which lane
// 4 * child + plane tests the box's farthest corner -- all <= 8 children at once, before any per-ray slab arithmetic.
// Pure pruning with margins on every rounding (the rectangle is widened, the plane test has a relative and an absolute
// slack), so results cannot change.  Returns false (warp-uniform) when the packet has no pyramid: no active lane, or a
// direction more than ~84 degrees off the axis.  `slack`: how far a ray may leave the segment (point -> apex); 0 for primary
// rays, 2e-4 for shadow rays, which start EPSILON = 1e-4 off the hit point but aim from the hit point itself (renderer.cpp:344).
RT_DEV bool packet_set_cull(PacketStack& K, bool active, V3 apex, V3 point, float slack)
{
    const unsigned lane = threadIdx.x & 31u;
    const unsigned am = __ballot_sync(0xffffffffu, active);
    if (am == 0u) return false;
    const int lead = __ffs(am) - 1;
    const V3 v = point - apex;
    V3 ez = v3(__shfl_sync(0xffffffffu, v.x, lead), __shfl_sync(0xffffffffu, v.y, lead), __shfl_sync(0xffffffffu, v.z, lead));
    const float len2 = length2(ez);
    if (!(len2 > 1e-30f)) return false;
    ez = normalize(ez);
    const V3 helper = fabsf(ez.x) < 0.5f ? v3(1, 0, 0) : v3(0, 1, 0);
    const V3 ex = normalize(cross(helper, ez));
    const V3 ey = cross(ez, ex);
    const float vz = dot(v, ez), vx = dot(v, ex), vy = dot(v, ey);
    const bool good = !active || (vz > 0.0f && vz * vz > 0.01f * length2(v));
    if (__ballot_sync(0xffffffffu, !good) != 0u) return false;
    const float tx = active ? vx / vz : 0.0f, ty = active ? vy / vz : 0.0f;
    float x0 = warp_min(active ? tx : INFINITY), x1 = -warp_min(active ? -tx : INFINITY);
    float y0 = warp_min(active ? ty : INFINITY), y1 = -warp_min(active ? -ty : INFINITY);
    const float wx = 1.0e-5f * (1.0f + fmaxf(fabsf(x0), fabsf(x1))), wy = 1.0e-5f * (1.0f + fmaxf(fabsf(y0), fabsf(y1)));
    x0 -= wx; x1 += wx; y0 -= wy; y1 += wy;
    if (lane < 4u) {
        V3 n;
        if (lane == 0u) n = ex - x0 * ez;
        else if (lane == 1u) n = x1 * ez - ex;
        else if (lane == 2u) n = ey - y0 * ez;
        else n = y1 * ez - ey;
        const float inv = 1.0f / sqrtf(length2(n));
        n = inv * n;
        K.plane[lane] = make_float4(n.x, n.y, n.z, dot(n, apex) - slack);
    }
    __syncwarp();
    return true;
}

// planes no box is outside of
RT_DEV void packet_no_cull(PacketStack& K)
{
    if ((threadIdx.x & 31u) < 4u) K.plane[threadIdx.x & 31u] = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
    __syncwarp();
}

// slab_entry (rt_device.h) for packets, with a warp-uniform exit between the axis slabs and the diagonal slabs: the
// rays of a packet mostly agree, so when NO lane survives the three axis slabs the record is dropped without the
// divergent region a per-lane early return costs.  Same arithmetic, same conservative acceptance.
// ORDERED: the staged record holds, per slab, (entry bound, exit bound) for THIS packet -- the lane that staged the
// float4 swapped the (near, far) pairs of the slabs whose denominator is negative for every ray of the packet -- so the
// per-slab min/max of the two quotients is not needed: 14 FMA + 2 x 7 running max/min instead of + 14 more min/max.
template <bool ORDERED>
RT_DEV float slab_entry_packet(const float4* rec, const SlabRay& sr, float t_limit, bool active, uint32_t& link, uint32_t& meta)
{
    float tn = -INFINITY, tf = INFINITY;
#define RT_SLAB(i, NEAR, FAR)                                   \
    {                                                           \
        float a = RT_FMA((NEAR), sr.inv[i], -sr.c[i]);          \
        float b = RT_FMA((FAR), sr.inv[i], -sr.c[i]);           \
        if (ORDERED) { tn = fmaxf(tn, a); tf = fminf(tf, b); }  \
        else { tn = fmaxf(tn, fminf(a, b)); tf = fminf(tf, fmaxf(a, b)); } \
    }
    const float4 q0 = rec[0];
    const float2 q1a = *reinterpret_cast<const float2*>(rec + 1);
    RT_SLAB(0, q0.x, q0.y)
    RT_SLAB(1, q0.z, q0.w)
    RT_SLAB(2, q1a.x, q1a.y)
    const float lim = fminf(t_limit, tf) + 2.0f * sr.slack;
    const bool pass = active && (tn <= lim) && !(tf + sr.slack < 0.0f);
    if (__ballot_sync(0xffffffffu, pass) == 0u) return INFINITY;
    const float2 q1b = *(reinterpret_cast<const float2*>(rec + 1) + 1);
    const float4 q2 = rec[2], q3 = rec[3];
    RT_SLAB(3, q1b.x, q1b.y)
    RT_SLAB(4, q2.x, q2.y)
    RT_SLAB(5, q2.z, q2.w)
    RT_SLAB(6, q3.x, q3.y)
#undef RT_SLAB
    link = f4_bits(q3.z); meta = f4_bits(q3.w);
    const bool ok = pass && (tn <= tf + 2.0f * sr.slack) && (tf + sr.slack >= 0.0f) && (tn - sr.slack <= t_limit);
    return ok ? tn - sr.slack : INFINITY;
}

RT_DEV uint32_t ld_vol(const unsigned int* p) { return *((const volatile unsigned int*)p); }

// One cell round of a packet: the (<= 8) staged or top-table records at `rec` are tested by every lane for its own ray; a
// child is entered if ANY lane hits it, with the smallest entry distance of the warp as its sort key (one redux.sync);
// lane 0 keeps the cell's entries [base, sp) of the shared-memory stack sorted by descending distance, so the nearest is
// popped first.  (Tried instead: the accepted children kept in registers, one per lane, ranked with a shuffle sweep, stored
// in parallel and the nearest entered without going through the stack -- +6 % frame time on cfg4: the sweep runs on every
// cell whereas the insertion costs one short loop per ACCEPTED child, mostly 1-3 per cell.)
template <bool ORDERED, bool COUNT>
RT_DEV bool packet_cell(const float4* rec, uint32_t count, const SlabRay& sr, float t_max, bool active, PacketStack& K, int& sp, TraceCounters& tc,
                        uint32_t keep)
{
    const unsigned lane = threadIdx.x & 31u;
    const int base = sp;
    // keep: bit k set = child k is to be tested (all `count` children, or those the bounding pyramid has not dropped)
    for (uint32_t m = keep; m != 0u; m &= m - 1u) {
        const uint32_t k = (uint32_t)__ffs((int)m) - 1u;
        if (COUNT && active) tc.vol_tests++;
        uint32_t cl = 0u, cm = 0u;
        const float tn = slab_entry_packet<ORDERED>(rec + 4 * k, sr, t_max, active, cl, cm);
        if (__ballot_sync(0xffffffffu, tn != INFINITY) == 0u) continue;
        const float tmin = warp_min(tn);
        if (sp >= RT_STACK_SIZE) return false;
        if (lane == 0) {                                     // keep [base, sp) sorted by descending entry distance
            int j = sp;
            while (j > base && K.t[j - 1] < tmin) {
                K.t[j] = K.t[j - 1]; K.link[j] = K.link[j - 1]; K.meta[j] = K.meta[j - 1];
                --j;
            }
            K.t[j] = tmin; K.link[j] = cl; K.meta[j] = cm;
        }
        ++sp;
    }
    return true;
}

// The top table in shared memory: loaded once per CTA at kernel start with ONE bulk asynchronous copy (cp.async.bulk, the
// 1-D form of TMA) that completes on an mbarrier; every thread of the CTA waits for it before its first packet.
struct TopTable {
    float4 rec[4 * RT_TOP_RECORDS];
    unsigned long long bar;
};
struct NoTopTable {                     // what a kernel instantiated without the top table keeps in shared memory instead
    unsigned long long bar;
};
template <bool TOP> struct TopStorage { typedef TopTable type; };
template <> struct TopStorage<false> { typedef NoTopTable type; };
RT_DEV const float4* top_pointer(TopTable& T) { return T.rec; }
RT_DEV const float4* top_pointer(NoTopTable&) { return nullptr; }
RT_DEV void load_top_table(const SceneView&, NoTopTable&) {}

RT_DEV void load_top_table(const SceneView& sc, TopTable& T)
{
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&T.bar), dst = (uint32_t)__cvta_generic_to_shared(&T.rec[0]);
    const uint32_t bytes = (uint32_t)sc.top_n * 64u;
    if (bytes == 0u) return;                                 // warp-uniform: a kernel argument
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(sc.top), "r"(bytes), "r"(bar)
                     : "memory");
    }
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TOP_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
        "@!p bra TOP_WAIT;\n"
        "}\n" ::"r"(bar)
        : "memory");
}

// Per-lane inputs: `active`, ray (o, d), t_max (closest: INFINITY; any: light limit).  Outputs: best (closest) or
// occluded (any).  For ANY: p / dist2 of the reference predicate; subtrees and triangles whose bit in the per-light masks is
// clear (sc.blk_occ / sc.tri_occ, light_cull.cuh) cannot occlude and are skipped.  K points to this warp's stack in shared memory, `top`
// to the CTA's copy of the top table (null: none).
// The traversal starts at the root cell, or (start_meta != 0) at the cell / leaf (start_link, start_meta).
// Returns false when the packet used up `max_rounds` cell/leaf rounds without finishing (max_rounds 0: no limit); the
// lanes whose `active` is still set then have no result yet, and K.link/meta[0, K.saved) are the cells the packet has
// not visited.  A packet's rounds are one dependent chain (pop -> fetch -> test -> push), 1-2 us each, so a packet that
// needs thousands of them (measured: one shadow packet through the pole of the 10 M-triangle sphere, 8 000 rounds =
// 11 ms of a 17 ms kernel) is SPLIT: each unvisited cell becomes a work item that another warp traces for the same 32
// rays (k_shade_items), and the answers are merged (any-hit: OR).
template <bool ANY, bool COUNT, bool CULL = false>
RT_DEV bool packet_trace(const SceneView& sc, PacketStack& K, const float4* top, bool& active, V3 o, V3 d, float t_max, V3 p, float dist2,
                         HitRec& best, bool& occluded, TraceCounters& tc, unsigned& overflow, int max_rounds, unsigned& rounds,
                         uint32_t start_link = 0u, uint32_t start_meta = 0u, int32_t best_orig = 0x7fffffff,
                         const unsigned int* poll_occ = nullptr, const unsigned long long* poll_best = nullptr, Drain drain = no_drain())
{
    const unsigned lane = threadIdx.x & 31u;
    SlabRay sr;
    slab_setup(o, d, sr);
    const V3 md = -d;
    best.tri = -1; best.t = -1.0f; best.u = 1.0f; best.v = 0.0f;
    occluded = false;
    // Do the packet's rays agree, slab by slab, on the sign of the denominator?  (A zero denominator agrees with both: its
    // quotients are NaN and drop out of the running max / min.)  If so the staged records are swapped into (entry, exit)
    // order for this packet and the ordered slab test is used; a packet that disagrees on any slab uses the general one.
    unsigned neg_mask = 0u;
#ifdef RTB_NO_ORDERED
    bool ordered = false;
#else
    bool ordered = true;
#endif
#pragma unroll
    for (int i = 0; i < 7; i++) {
        const bool nz = active && sr.inv[i] != 0.0f;
        const unsigned bn = __ballot_sync(0xffffffffu, nz && sr.inv[i] < 0.0f), bp = __ballot_sync(0xffffffffu, nz && sr.inv[i] > 0.0f);
        if (bn != 0u && bp != 0u) ordered = false;
        if (bn != 0u) neg_mask |= 1u << i;
    }
    // the pair(s) this lane swaps when it stages float4 number (lane & 3) of a record: slabs 2f and 2f + 1 (float4 3: slab 6 only)
    const unsigned f = lane & 3u;
    const bool swap_lo = ordered && ((neg_mask >> (2u * f)) & 1u) != 0u;
    const bool swap_hi = ordered && f < 3u && ((neg_mask >> (2u * f + 1u)) & 1u) != 0u;
    uint32_t link = start_link, meta = start_meta;
    if (start_meta == 0u) {
        const rt_f4* r = sc.recs;
        rt_f4 q0 = RT_LDG4(r), q1 = RT_LDG4(r + 1), q2 = RT_LDG4(r + 2), q3 = RT_LDG4(r + 3);
        if (COUNT && active) tc.vol_tests++;
        if (COUNT && lane == 0) tc.rec_fetch++;
        const float tn = active ? slab_entry(q0, q1, q2, q3, sr, t_max) : INFINITY;
        link = f4_bits(q3.z); meta = f4_bits(q3.w);
        if (__ballot_sync(0xffffffffu, tn != INFINITY) == 0u || (meta & ~(RT_LEAF_BIT | RT_META_TOP)) == 0u) return true;
        if (ANY && (__ldg(sc.blk_occ) & 1u) == 0u) return true;             // nothing in the scene can occlude the light
    }
    int sp = 0;
    for (;;) {
        if (max_rounds > 0 && sp < RT_STACK_SIZE) {
            bool stop = (int)rounds >= max_rounds;
            if (!stop && drain.counter != nullptr && (int)rounds >= drain.min_rounds && (rounds & 15u) == 0u) {
                uint32_t handed = 0;
                if (lane == 0) handed = ld_vol(drain.counter);
                stop = __shfl_sync(0xffffffffu, handed, 0) >= drain.total;     // nothing left to fetch: the other warps are idle or about to be
            }
            if (stop) {
                if (lane == 0) { K.t[sp] = 0.0f; K.link[sp] = link; K.meta[sp] = meta; K.saved = sp + 1; }
                __syncwarp();
                return false;
            }
        }
        ++rounds;
        // An item of a split packet that runs concurrently with the record's other items (fused scheduling) looks at what
        // they have found every fourth round: an answered shadow ray is dropped (and the item ends when all are), a closer
        // primary hit lowers this lane's limit.  Pure pruning: the merged answer is an OR / a minimum either way.
        if ((rounds & 3u) == 0u) {
            if (ANY && poll_occ != nullptr) {
                uint32_t w = 0;
                if (lane == 0) w = ld_vol(poll_occ);
                w = __shfl_sync(0xffffffffu, w, 0);
                if ((w >> lane) & 1u) active = false;
                if (__ballot_sync(0xffffffffu, active) == 0u) return true;
            }
            if (!ANY && poll_best != nullptr) {
                const unsigned long long key = *((const volatile unsigned long long*)(poll_best + lane));
                if (key != ~0ull) {
                    const float te = __uint_as_float((uint32_t)(key >> 32));
                    const int32_t oe = (int32_t)(uint32_t)key;
                    if (te < t_max || (te == t_max && oe < best_orig)) { t_max = te; best_orig = oe; }
                }
            }
        }
        if (!(meta & RT_LEAF_BIT)) {
            // ---- one cell.  Its records come from the CTA's top table (the first levels of the tree: no global fetch), or
            // the warp fetches them with ONE coalesced 128-bit load per lane; either way they are staged in this warp's
            // shared memory -- swapped into (entry, exit) order when the packet's rays agree on the signs -- and every lane
            // then tests every child record (broadcast LDS) for its own ray.
            const uint32_t count = meta & RT_META_COUNT_MASK;
            const bool in_top = top != nullptr && (meta & RT_META_TOP) != 0u;
            if (lane < 4u * count) {
                float4 v = in_top ? top[4u * ((meta >> RT_META_TOP_SHIFT) & 0xffu) + lane] : RT_LDG4(sc.recs + 4 * (size_t)link + lane);
                if (swap_lo) { const float t = v.x; v.x = v.y; v.y = t; }
                if (swap_hi) { const float t = v.z; v.z = v.w; v.w = t; }
                K.stage[lane] = v;
            }
            if (COUNT && lane == 0 && !in_top) tc.rec_fetch += count;
            __syncwarp();
            uint32_t keep = (1u << count) - 1u;
            if (ANY) keep &= __ldg(sc.blk_occ + (link >> 1));              // children whose subtree may occlude the light
            if (CULL) {
                // lane 4 * child + plane: the corner of the child's box that lies farthest along the plane's inward normal
                const uint32_t child = lane >> 2;
                const float4 pl = K.plane[lane & 3u];
                const float4 b0 = K.stage[4u * child];
                const float2 b1 = *reinterpret_cast<const float2*>(&K.stage[4u * child + 1u]);
                // (the staged pairs may have been swapped into entry / exit order; slots >= count hold stale records: masked below)
                const float ax = pl.x * (pl.x > 0.0f ? fmaxf(b0.x, b0.y) : fminf(b0.x, b0.y));
                const float ay = pl.y * (pl.y > 0.0f ? fmaxf(b0.z, b0.w) : fminf(b0.z, b0.w));
                const float az = pl.z * (pl.z > 0.0f ? fmaxf(b1.x, b1.y) : fminf(b1.x, b1.y));
                const bool outside = (ax + ay + az) - pl.w < -4.0e-6f * (fabsf(ax) + fabsf(ay) + fabsf(az) + fabsf(pl.w));
                unsigned m = __ballot_sync(0xffffffffu, outside);
                m |= m >> 1;
                m |= m >> 2;                                 // bit 4k: some plane has child k outside
                // gather bit 4k of ~m into bit k
                unsigned in = ~m & 0x11111111u;
                in = (in | (in >> 3)) & 0x03030303u;
                in = (in | (in >> 6)) & 0x000f000fu;
                in = (in | (in >> 12)) & 0xffu;
                keep &= in;
            }
            const bool fits = ordered ? packet_cell<true, COUNT>(K.stage, count, sr, t_max, active, K, sp, tc, keep)
                                      : packet_cell<false, COUNT>(K.stage, count, sr, t_max, active, K, sp, tc, keep);
            if (!fits) { overflow = 1u; return true; }
            __syncwarp();
        } else {
            // ---- one leaf: triangles staged the same way, 10 per round (8 with the bounding pyramid); every lane tests every
            // triangle for its own ray.  With the pyramid, lane 4 * triangle + plane first looks whether the triangle's three
            // vertices all lie outside its plane: no ray of the packet can hit such a triangle, and the per-ray loop runs over
            // the others only.
            const uint32_t cnt = meta & ~RT_LEAF_BIT;
            const uint32_t per_round = CULL ? 8u : 10u;
            for (uint32_t first = 0; first < cnt; first += per_round) {
                const uint32_t m = min(per_round, cnt - first);
                uint32_t keep = (1u << m) - 1u;
                if (ANY) {                                   // the triangles that may occlude the light; none: not even staged
                    const uint32_t at = link + first;
                    keep &= __funnelshift_r(__ldg(sc.tri_occ + (at >> 5)), __ldg(sc.tri_occ + (at >> 5) + 1), at & 31u);
                    if (keep == 0u) continue;
                }
                if (lane < 3u * m) K.stage[lane] = RT_LDG4(sc.tris + 3 * (size_t)(link + first) + lane);
                if (COUNT && lane == 0) tc.tri_fetch += m;
                __syncwarp();
                if (CULL) {
                    const uint32_t tri = lane >> 2;
                    const float4 pl = K.plane[lane & 3u];
                    const float4 va = K.stage[3u * tri], vb = K.stage[3u * tri + 1u], vc = K.stage[3u * tri + 2u];   // slots >= m: stale, masked below
                    const float da = (pl.x * va.x + pl.y * va.y + pl.z * va.z) - pl.w;
                    const float db = (pl.x * vb.x + pl.y * vb.y + pl.z * vb.z) - pl.w;
                    const float dc = (pl.x * vc.x + pl.y * vc.y + pl.z * vc.z) - pl.w;
                    const float mag = fabsf(pl.w) + fmaxf(fabsf(va.x), fmaxf(fabsf(vb.x), fabsf(vc.x))) + fmaxf(fabsf(va.y), fmaxf(fabsf(vb.y), fabsf(vc.y))) +
                                      fmaxf(fabsf(va.z), fmaxf(fabsf(vb.z), fabsf(vc.z)));
                    const bool outside = fmaxf(da, fmaxf(db, dc)) < -4.0e-6f * mag;
                    unsigned om = __ballot_sync(0xffffffffu, outside);
                    om |= om >> 1;
                    om |= om >> 2;
                    unsigned in = ~om & 0x11111111u;
                    in = (in | (in >> 3)) & 0x03030303u;
                    in = (in | (in >> 6)) & 0x000f000fu;
                    in = (in | (in >> 12)) & 0xffu;
                    keep &= in;
                }
                for (uint32_t km = keep; km != 0u; km &= km - 1u) {
                    const uint32_t i = (uint32_t)__ffs((int)km) - 1u;
                    const float4 p0 = K.stage[3 * i], p1 = K.stage[3 * i + 1], p2 = K.stage[3 * i + 2];
                    if (COUNT && active) tc.tri_tests++;
                    float t, u, v;
                    if (active && tri_test(p0, p1, p2, o, md, t, u, v)) {
                        const uint32_t tri = link + first + i;
                        if (ANY) {
                            if (t > 0.0f) {
                                V3 q = o + t * d;                // renderer.cpp:351
                                if (length2(p - q) < dist2) { occluded = true; active = false; }   // renderer.cpp:354
                            }
                        } else if (t < t_max || (t == t_max && sc.orig[tri] < best_orig)) {
                            // closest so far; a tie on t goes to the lower original index.  best_orig starts at
                            // INT_MAX (root) or at the index of the hit other parts of a split packet have found
                            t_max = t;
                            best_orig = sc.orig[tri];
                            best.tri = (int32_t)tri; best.t = t; best.u = u; best.v = v;
                        }
                    }
                }
                __syncwarp();
            }
            if (ANY && __ballot_sync(0xffffffffu, active) == 0u) return true;   // every ray of the packet is occluded
        }
        // ---- next cell: nearest first; skip entries no lane can still use
        bool got = false;
        while (sp > 0) {
            --sp;
            const float et = K.t[sp];
            if (__ballot_sync(0xffffffffu, active && et <= t_max) == 0u) continue;
            link = K.link[sp]; meta = K.meta[sp];
            got = true;
            break;
        }
        if (!got) return true;
    }
}

// A packet (or item) that ran out of rounds: every unvisited cell K.link/meta[0, K.saved) becomes one work item of item
// pass `pass` for split record `sidx`.  Returns false when the item region is full (the caller then finishes in place);
// the slots it was handed are still filled (with null items) so that the region never holds garbage.
RT_DEV bool emit_items(const QueueView& q, unsigned int* items_n, const PacketStack& K, int pass, uint32_t sidx)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = (uint32_t)K.saved;
    uint32_t at = 0;
    if (lane == 0) at = atomicAdd(&items_n[pass], n);
    at = __shfl_sync(0xffffffffu, at, 0);
    const bool ok = at + n <= q.item_capacity;
    uint4* region = q.items + (size_t)pass * q.item_capacity;
    for (uint32_t i = lane; i < n && at + i < q.item_capacity; i += 32u)
        region[at + i] = ok ? make_uint4(sidx, K.link[i], K.meta[i], 0u) : make_uint4(0xffffffffu, 0u, 0u, 0u);
    __syncwarp();
    return ok;
}

// Closest hit of a split primary packet, merged over its work items with atomicMin: t >= 0, so the bits of t order like
// t; a tie on t goes to the lower original index -- the rule of packet_trace.
RT_DEV unsigned long long closest_key(float t, int32_t orig) { return ((unsigned long long)__float_as_uint(t) << 32) | (uint32_t)orig; }
constexpr unsigned long long kNoHitKey = ~0ull;

// Packet version of k_primary: a warp takes 32 consecutive ray slots (an 8x4 pixel block) per fetch.
#ifndef RTB_PRIMARY_MINB
#define RTB_PRIMARY_MINB 8   /* measured on cfg4: 8 CTAs/SM (64 registers, some spills) 7.5 ms, 7: 7.6, 6 (80, none): 8.0, 5: 8.6 -- latency-bound */
#endif
#define RTB_PRIMARY_BOUNDS __launch_bounds__(kPrimaryThreads, RTB_PRIMARY_MINB)
template <bool COUNT, bool TOP>
__global__ void RTB_PRIMARY_BOUNDS
k_primary_packet(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    __shared__ PacketStack stacks[kPrimaryThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    __shared__ typename TopStorage<TOP>::type top_table;        // TOP: the first levels of the tree, one bulk asynchronous copy per CTA
    load_top_table(sc, top_table);
    const float4* top = top_pointer(top_table);
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t pps = (uint32_t)wk.patches_per_side;
    const uint32_t total = (wk.tile_end - wk.tile_begin) * pps * pps * (uint32_t)(kPatch * kPatch);
    TraceCounters tc = zero_counters();
    unsigned overflow = 0;
    uint32_t traced = 0;                                                        // lane 0: rays of the packets this warp traced
    // Work fetch: kPrimaryFetch packets per atomic, and the atomic for the NEXT batch is issued before the current
    // batch is traced, so its round trip (11 % of the stall samples when it was waited for) is hidden.
    uint32_t nxt = 0;
    if (lane == 0) nxt = atomicAdd(&cnt->next_patch, 32u * kPrimaryFetch);
    for (;;) {
        const uint32_t first = __shfl_sync(0xffffffffu, nxt, 0);
        if (first >= total) break;
        if (lane == 0) nxt = atomicAdd(&cnt->next_patch, 32u * kPrimaryFetch);
#pragma unroll 1
        for (uint32_t b = 0; b < (uint32_t)kPrimaryFetch; b++) {
            const uint32_t base = first + 32u * b;
            if (base >= total) break;
            const uint32_t slot = base + lane;
            int px = 0, py = 0;
            const bool active = slot < total && slot_pixel(wk, fr, slot, px, py);
            V3 o = v3(0, 0, 0), d = v3(0, 0, 1);
            // a block that the scene does not cover misses without a ray being set up
            const bool inside = active && covered(wk, px, py);
            if (__ballot_sync(0xffffffffu, inside) == 0u) {
                if (slot < total) {
                    q.slot_tri[slot] = -1;
                    if (active) {
                        if (miss_needs_ray(fr)) primary_ray(fr, px, py, o, d);
                        super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
                    }
                }
                continue;
            }
            if (active) primary_ray(fr, px, py, o, d);
            traced += (uint32_t)__popc(__ballot_sync(0xffffffffu, active));
            HitRec best;
            bool occ, live = active;
            unsigned rounds = 0;
            const unsigned long long t0 = COUNT ? global_ns() : 0ull;
            if (!((tune.cull & 1) != 0 && packet_set_cull(K, active, o, o + d, 0.0f))) packet_no_cull(K);
            const bool finished = packet_trace<false, COUNT, true>(sc, K, top, live, o, d, INFINITY, o, 0.0f, best, occ, tc, overflow, tune.primary_rounds, rounds,
                                                                   0u, 0u, 0x7fffffff, nullptr, nullptr, make_drain(&cnt->next_patch, total, tune.primary_min));
            __syncwarp();
            if (COUNT && lane == 0) note_packet(cnt, 0, rounds, global_ns() - t0);
            if (!finished) {
                // out of rounds: the closest hits so far go to a split record, every unvisited cell becomes a work item
                const unsigned am = __ballot_sync(0xffffffffu, active);
                uint32_t sidx = 0;
                if (lane == 0) sidx = atomicAdd(&cnt->p_split, 1u);
                sidx = __shfl_sync(0xffffffffu, sidx, 0);
                if (sidx < q.split_capacity && emit_items(q, cnt->p_items_n, K, 0, sidx)) {
                    if (lane == 0) { q.split_base[sidx] = base; q.split_active[sidx] = am; }
                    q.split_best[(size_t)sidx * 32u + lane] = (active && best.tri >= 0) ? closest_key(best.t, sc.orig[best.tri]) : kNoHitKey;
                    continue;                                                  // k_primary_finish writes these slots
                }
                if (sidx < q.split_capacity && lane == 0) { q.split_base[sidx] = base; q.split_active[sidx] = 0u; }
                live = active;                                                 // no room: trace it here, from the root
                packet_trace<false, COUNT>(sc, K, top, live, o, d, INFINITY, o, 0.0f, best, occ, tc, overflow, 0, rounds);
                __syncwarp();
            }
            if (slot < total) {
                const bool hit = active && best.tri >= 0 && best.t > 0.1f;        // t > 0 (bvh.h:247) and min_t (renderer.cpp:1039)
                q.slot_tri[slot] = hit ? best.tri : -1;
                if (hit) { q.slot_t[slot] = best.t; q.slot_u[slot] = best.u; q.slot_v[slot] = best.v; }
                else if (active) {
                    if (sc.n_shapes > 0) q.slot_t[slot] = (best.tri >= 0 && best.t > 0.0f) ? best.t : -1.0f;   // see k_primary_shapes
                    super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
                }
            }
        }
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (lane == 0 && traced) atomicAdd(&cnt->traced_primary, (unsigned long long)traced);
    if (COUNT) flush_work(tc, &cnt->primary_vol, &cnt->primary_tri, &cnt->primary_fetch);
}

// Item pass of the split primary packets: a warp takes one unvisited cell of a split packet, rebuilds the packet's 32
// primary rays, starts every lane at the closest hit the record holds so far (cells beyond it are pruned), traces from
// that cell and merges what it finds with atomicMin.  An item that runs out of rounds is split again.
template <bool COUNT>
__global__ void RTB_PRIMARY_BOUNDS
k_primary_items(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, Tuning tune, int pass)
{
    __shared__ PacketStack stacks[kPrimaryThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    const float4* top = nullptr;                       // items start deep in the tree: no use for the top table
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = min(cnt->p_items_n[pass], q.item_capacity);
    const uint4* region = q.items + (size_t)pass * q.item_capacity;
    const int budget = pass + 1 < tune.item_passes ? tune.item_rounds : 0;
    TraceCounters tc = zero_counters();
    unsigned overflow = 0;
    for (;;) {
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(&cnt->p_items_next[pass], 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= n) break;
        const uint4 item = region[i];
        const uint32_t sidx = item.x;
        if (sidx == 0xffffffffu) continue;
        const uint32_t base = q.split_base[sidx];
        const uint32_t slot = base + lane;
        const bool active = ((q.split_active[sidx] >> lane) & 1u) != 0u;
        int px = 0, py = 0;
        V3 o = v3(0, 0, 0), d = v3(0, 0, 1);
        if (active) { slot_pixel(wk, fr, slot, px, py); primary_ray(fr, px, py, o, d); }
        unsigned long long* mine = q.split_best + (size_t)sidx * 32u + lane;
        const unsigned long long seen = *((volatile unsigned long long*)mine);
        const float t_start = seen == kNoHitKey ? INFINITY : __uint_as_float((uint32_t)(seen >> 32));
        const int32_t orig_start = seen == kNoHitKey ? 0x7fffffff : (int32_t)(uint32_t)seen;
        HitRec best;
        bool occ, live = active;
        unsigned rounds = 0;
        if (!((tune.cull & 1) != 0 && packet_set_cull(K, active, o, o + d, 0.0f))) packet_no_cull(K);
        bool finished = packet_trace<false, COUNT, true>(sc, K, top, live, o, d, t_start, o, 0.0f, best, occ, tc, overflow, budget, rounds, item.y, item.z, orig_start,
                                                         nullptr, nullptr, make_drain(&cnt->p_items_next[pass], n, tune.item_min));
        __syncwarp();
        if (active && best.tri >= 0) atomicMin(mine, closest_key(best.t, sc.orig[best.tri]));
        if (!finished && !emit_items(q, cnt->p_items_n, K, pass + 1, sidx)) {
            // no room: finish the item here (from its cell again, now pruned by what it has just found)
            const unsigned long long now = *((volatile unsigned long long*)mine);
            const float t2 = now == kNoHitKey ? INFINITY : __uint_as_float((uint32_t)(now >> 32));
            const int32_t o2 = now == kNoHitKey ? 0x7fffffff : (int32_t)(uint32_t)now;
            live = active;
            packet_trace<false, COUNT>(sc, K, top, live, o, d, t2, o, 0.0f, best, occ, tc, overflow, 0, rounds, item.y, item.z, o2);
            __syncwarp();
            if (active && best.tri >= 0) atomicMin(mine, closest_key(best.t, sc.orig[best.tri]));
        }
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (COUNT) flush_work(tc, &cnt->primary_vol, &cnt->primary_tri, &cnt->primary_fetch);
}

// After the item passes: the slot records (or miss colours) of the split primary packets.  The merged key names the
// triangle by its original index; one more ray/triangle test of that triangle reproduces t, u, v bit for bit.
__global__ void __launch_bounds__(kPrimaryThreads)
k_primary_finish(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = min(cnt->p_split, q.split_capacity);
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t sidx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; sidx < n; sidx += warps) {
        const uint32_t am = q.split_active[sidx];
        if (am == 0u) continue;                                                // traced in place after all
        const uint32_t slot = q.split_base[sidx] + lane;
        const unsigned long long key = q.split_best[(size_t)sidx * 32u + lane];
        if ((am >> lane) & 1u) {
            int px = 0, py = 0;
            V3 o, d;
            slot_pixel(wk, fr, slot, px, py);
            primary_ray(fr, px, py, o, d);
            bool hit = false;
            float gated_t = -1.0f;                                             // a BVH hit with 0 < t <= min_t, see k_primary_shapes
            if (key != kNoHitKey) {
                const uint32_t tri = (uint32_t)sc.leaf_of[(uint32_t)key];
                const rt_f4* tp = sc.tris + 3 * (size_t)tri;
                float t, u, v;
                if (tri_test(RT_LDG4(tp), RT_LDG4(tp + 1), RT_LDG4(tp + 2), o, -d, t, u, v)) {
                    if (t > 0.1f) {                                            // min_t, renderer.cpp:1039
                        hit = true;
                        q.slot_tri[slot] = (int32_t)tri; q.slot_t[slot] = t; q.slot_u[slot] = u; q.slot_v[slot] = v;
                    } else if (t > 0.0f)
                        gated_t = t;
                }
            }
            if (!hit) {
                q.slot_tri[slot] = -1;
                if (sc.n_shapes > 0) q.slot_t[slot] = gated_t;
                super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
            }
        } else {
            const uint32_t pps = (uint32_t)wk.patches_per_side;
            if (slot < (wk.tile_end - wk.tile_begin) * pps * pps * (uint32_t)(kPatch * kPatch)) q.slot_tri[slot] = -1;   // slot without a ray
        }
    }
}

// trace_ray's loop over the analytic shapes (renderer.cpp:1029-1037), after the BVH part of the primary rays: a shape
// replaces the closest hit so far when it is strictly closer (or when there is none), in the order the shapes were added;
// then the min_t gate (:1039) decides between hit and miss.  The "closest hit so far" of a slot is slot_t: the BVH hit's
// t, also when that hit is below min_t and the slot therefore counts as a miss (the primary kernels keep it then), else -1.
// One thread per ray slot.  A shape hit is recorded as slot_tri = -2 - shape.
__global__ void k_primary_shapes(SceneView sc, FrameView fr, WorkView wk, QueueView q, uint32_t total, uint32_t* super)
{
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < total; slot += gridDim.x * blockDim.x) {
        int px, py;
        if (!slot_pixel(wk, fr, slot, px, py)) continue;
        V3 o, d;
        primary_ray(fr, px, py, o, d);
        float final_t = q.slot_t[slot];
        int best = -1;
        for (int i = 0; i < sc.n_shapes; i++) {
            float t;
            V3 n;
            int32_t m;
            if (shape_intersect(sc, i, o, d, t, n, m) && (t < final_t || final_t == -1.0f)) { final_t = t; best = i; }
        }
        if (best < 0) continue;
        if (final_t > 0.1f) { q.slot_tri[slot] = -2 - best; q.slot_t[slot] = final_t; }
        else {
            q.slot_tri[slot] = -1;
            super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
        }
    }
}

// Ordered stream compaction of the slot records into the hit queue.  A block owns kCompactSlots consecutive slots:
// every thread counts the hits among its kCompactPerThread consecutive slots, a block-wide exclusive scan places them,
// ONE atomic per block reserves the block's span of the queue.  Inside a span the entries keep slot order, so a warp
// of k_shade / k_reflect that takes 32 consecutive entries gets neighbouring pixels.
constexpr int kCompactThreads = 256;
constexpr int kCompactPerThread = 8;
constexpr int kCompactSlots = kCompactThreads * kCompactPerThread;

__global__ void __launch_bounds__(kCompactThreads)
k_compact(SceneView sc, QueueView q, ChunkCounters* cnt, uint32_t total, int any_reflective)
{
    __shared__ uint32_t warp_hits[kCompactThreads / 32], warp_refl[kCompactThreads / 32];
    __shared__ uint32_t span_hits, span_refl;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t n_blocks = (total + kCompactSlots - 1) / kCompactSlots;
    for (uint32_t blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
        const uint32_t first = blk * kCompactSlots + threadIdx.x * kCompactPerThread;
        uint32_t hits = 0, refl = 0;                         // bit j: slot first + j is a hit / a reflective hit
#pragma unroll
        for (int j = 0; j < kCompactPerThread; j++) {
            const uint32_t slot = first + (uint32_t)j;
            if (slot < total) {
                const int32_t tri = q.slot_tri[slot];
                if (tri != -1) {                             // a triangle (>= 0) or analytic shape -2 - tri
                    hits |= 1u << j;
                    const int32_t mat = tri >= 0 ? load_tri_shade(sc, tri).mat : shape_material(sc, -2 - tri);
                    if (any_reflective && load_material(sc, mat).reflection > 0.0f) refl |= 1u << j;
                }
            }
        }
        // exclusive scan of the per-thread counts over the block
        uint32_t ch = (uint32_t)__popc(hits), cr = (uint32_t)__popc(refl);
        uint32_t ih = ch, ir = cr;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, ih, o), b = __shfl_up_sync(0xffffffffu, ir, o);
            if ((int)lane >= o) { ih += a; ir += b; }
        }
        if (lane == 31) { warp_hits[warp] = ih; warp_refl[warp] = ir; }
        __syncthreads();
        uint32_t oh = ih - ch, orf = ir - cr;
        for (unsigned w = 0; w < warp; w++) { oh += warp_hits[w]; orf += warp_refl[w]; }
        if (threadIdx.x == kCompactThreads - 1) {
            const uint32_t th = oh + ch, tr = orf + cr;
            span_hits = th ? atomicAdd(&cnt->n_hits, th) : 0u;
            span_refl = tr ? atomicAdd(&cnt->n_refl, tr) : 0u;
        }
        __syncthreads();
        uint32_t ph = span_hits + oh, pr = span_refl + orf;
#pragma unroll
        for (int j = 0; j < kCompactPerThread; j++) {
            if (hits & (1u << j)) {
                q.hit_slot[ph] = first + (uint32_t)j;
                if (refl & (1u << j)) q.refl_idx[pr++] = ph;
                ph++;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Light-space ordering of the hit queue (RT_OPT_SHADOW_SORT).  The shadow rays of one point light are the rays FROM the
// light: two hits seen from the light in nearly the same direction have shadow rays through the same cells, whatever
// their depth, whereas 32 neighbouring PIXELS of a thin-strand scene hit strands at unrelated depths (cfg5: a packet of
// queue-order neighbours does 8x the slab tests of its rays traced one by one).  So the queue is reordered before
// k_shade_packet forms its packets: key = Morton code of the hit point's direction from the light on a kSortGrid^2 grid
// (gnomonic map of the cone that holds the scene when the light is outside the scene's bounding sphere, octahedral map of
// the whole sphere otherwise), one counting sort: histogram -> scan of the bins -> scatter.  Which 32 rays share a packet
// never changes a ray's answer (any-hit is decided per ray), so frames stay bit-identical.
constexpr int kSortGrid = 512;
constexpr int kSortBins = kSortGrid * kSortGrid;
constexpr int kSortScanThreads = 1024;                       // bins per block of the two scan kernels
constexpr int kSortScanBlocks = kSortBins / kSortScanThreads;

RT_DEV bool queue_sorted(const QueueView& q, const ChunkCounters* cnt)
{
    return q.sort_mode == 1u || (q.sort_mode == 2u && (unsigned long long)cnt->n_hits * 4ull < (unsigned long long)q.sort_slots);
}
// for the kernels of the shade stage: read the hit queue in the order the sort kernels left it (if they ran)
RT_DEV void pick_hit_queue(QueueView& q, const ChunkCounters* cnt)
{
    if (queue_sorted(q, cnt)) q.hit_slot = q.hit_sorted;
}

struct LightMap {
    V3 ex, ey, ez;          // orthonormal; ez points from the light to the centre of the scene's bounding sphere
    float scale;            // gnomonic: 1 / tan(half angle of the cone); 0: octahedral map
};

RT_DEV uint32_t morton_spread(uint32_t x)                    // 16 bits -> every other bit
{
    x = (x | (x << 8)) & 0x00ff00ffu;
    x = (x | (x << 4)) & 0x0f0f0f0fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

RT_DEV uint32_t light_key(const LightMap& lm, V3 light, V3 p)
{
    const V3 w = p - light;
    const float x = dot(w, lm.ex), y = dot(w, lm.ey), z = dot(w, lm.ez);
    float a, b;
    if (lm.scale > 0.0f) {
        const float iz = lm.scale / fmaxf(z, 1.0e-30f);
        a = x * iz; b = y * iz;
    } else {
        const float s = 1.0f / fmaxf(fabsf(x) + fabsf(y) + fabsf(z), 1.0e-30f);
        a = x * s; b = y * s;
        if (z < 0.0f) {
            const float fa = (1.0f - fabsf(b)) * (a < 0.0f ? -1.0f : 1.0f), fb = (1.0f - fabsf(a)) * (b < 0.0f ? -1.0f : 1.0f);
            a = fa; b = fb;
        }
    }
    // fminf / fmaxf drop a NaN operand: every input lands on the grid
    const uint32_t ia = (uint32_t)fminf(fmaxf((a * 0.5f + 0.5f) * (float)kSortGrid, 0.0f), (float)(kSortGrid - 1));
    const uint32_t ib = (uint32_t)fminf(fmaxf((b * 0.5f + 0.5f) * (float)kSortGrid, 0.0f), (float)(kSortGrid - 1));
    return morton_spread(ia) | (morton_spread(ib) << 1);
}

__global__ void __launch_bounds__(256)
k_sort_keys(FrameView fr, WorkView wk, QueueView q, const ChunkCounters* cnt, LightMap lm, uint32_t* keys, uint32_t* bins)
{
    if (!queue_sorted(q, cnt)) return;
    const uint32_t n = cnt->n_hits;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t slot = q.hit_slot[i];
        int px, py;
        slot_pixel(wk, fr, slot, px, py);
        V3 o, d;
        primary_ray(fr, px, py, o, d);
        const uint32_t key = light_key(lm, fr.light, o + q.slot_t[slot] * d);
        keys[i] = key;
        atomicAdd(&bins[key], 1u);
    }
}

RT_DEV uint32_t block_sum_1024(uint32_t v, uint32_t* warp_part)       // sum over a 1024-thread block, returned to every thread
{
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t w = __reduce_add_sync(0xffffffffu, v);
    __syncthreads();
    if (lane == 0) warp_part[warp] = w;
    __syncthreads();
    const uint32_t t = __reduce_add_sync(0xffffffffu, warp_part[lane]);
    return t;
}

__global__ void __launch_bounds__(kSortScanThreads)
k_sort_partial(QueueView q, const ChunkCounters* cnt, const uint32_t* bins, uint32_t* partial)
{
    __shared__ uint32_t warp_part[32];
    if (!queue_sorted(q, cnt)) return;
    const uint32_t total = block_sum_1024(bins[blockIdx.x * kSortScanThreads + threadIdx.x], warp_part);
    if (threadIdx.x == 0) partial[blockIdx.x] = total;
}

// bins[] (counts) -> exclusive prefix sums over all kSortBins, in place: a block adds up the partial sums of the blocks
// before it and scans its own 1024 bins.
__global__ void __launch_bounds__(kSortScanThreads)
k_sort_scan(QueueView q, const ChunkCounters* cnt, uint32_t* bins, const uint32_t* partial)
{
    __shared__ uint32_t warp_part[32];
    if (!queue_sorted(q, cnt)) return;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t before = block_sum_1024(threadIdx.x < blockIdx.x ? partial[threadIdx.x] : 0u, warp_part);
    static_assert(kSortScanBlocks <= kSortScanThreads, "one thread per preceding block");
    const uint32_t c = bins[blockIdx.x * kSortScanThreads + threadIdx.x];
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, inc, o);
        if ((int)lane >= o) inc += a;
    }
    __syncthreads();
    if (lane == 31) warp_part[warp] = inc;
    __syncthreads();
    uint32_t wsum = warp_part[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t a = __shfl_up_sync(0xffffffffu, wsum, o);
        if ((int)lane >= o) wsum += a;
    }
    const uint32_t warps_before = __shfl_sync(0xffffffffu, wsum - warp_part[lane], warp);
    bins[blockIdx.x * kSortScanThreads + threadIdx.x] = before + warps_before + inc - c;
}

__global__ void __launch_bounds__(256)
k_sort_scatter(QueueView q, const ChunkCounters* cnt, const uint32_t* keys, uint32_t* bins)
{
    if (!queue_sorted(q, cnt)) return;
    uint32_t* sorted = q.hit_sorted;
    const uint32_t n = cnt->n_hits;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        sorted[atomicAdd(&bins[keys[i]], 1u)] = q.hit_slot[i];
}

// The primary ray and hit record of hit-queue entry i.
RT_DEV void queue_ray(const FrameView& fr, const WorkView& wk, const QueueView& q, uint32_t i, V3& o, V3& d, HitRec& hr, uint32_t& pix)
{
    const uint32_t slot = q.hit_slot[i];
    int px, py;
    slot_pixel(wk, fr, slot, px, py);
    pix = (uint32_t)py * (uint32_t)fr.rw + (uint32_t)px;
    hr.tri = q.slot_tri[slot]; hr.t = q.slot_t[slot]; hr.u = q.slot_u[slot]; hr.v = q.slot_v[slot];
    primary_ray(fr, px, py, o, d);
}

template <bool COUNT>
__global__ void __launch_bounds__(kQueueThreads)
k_reflect(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt)
{
    // Tallies of a fan go to a per-entry record that k_shade sums up: the threads of a warp sit at different
    // recursion depths here, so no warp-level reduction is attempted in this kernel.
    const uint32_t n = cnt->n_refl;
    unsigned overflow = 0;
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        const uint32_t i = q.refl_idx[r];
        TraceCounters tc = zero_counters();
        V3 o, d;
        HitRec hr;
        uint32_t pix;
        queue_ray(fr, wk, q, i, o, d, hr, pix);
        Hit hit = make_hit(sc, hr, o, d);
        V3 p;
        MatView m;
        shade_direct(sc, fr, o, d, hit, p, m);                             // updates hit.normal (normal mapping)
        XorShift32 rng;
        rng.state = pixel_seed(pix, fr.s.rng_seed);
        Col c = compute_reflection<COUNT>(sc, fr, d, p, hit, m, 0, rng, &tc);
        q.refl_rgb[3 * (size_t)i + 0] = c.r;
        q.refl_rgb[3 * (size_t)i + 1] = c.g;
        q.refl_rgb[3 * (size_t)i + 2] = c.b;
        q.refl_cnt[3 * (size_t)i + 0] = (unsigned long long)tc.refl_rays | ((unsigned long long)tc.refl_shadow_rays << 32);
        q.refl_cnt[3 * (size_t)i + 1] = tc.vol_tests;
        q.refl_cnt[3 * (size_t)i + 2] = tc.tri_tests;
        overflow |= tc.stack_overflow;
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_reflect_fan: the rough-reflection fan of a hit with one LANE per fan ray (recursion limit 1, the stated setting of
// BASELINE.json's configs[2]).  compute_reflection (rt_device.h) walks a fan sequentially because the reference does and
// two things chain its samples together:
//   (1) the random stream: sample i draws 3 numbers, and when the hit it is SHADED with has a rough reflective material, the
//       nested fan of that hit draws 3 * sample_count more before it finds out that the recursion limit cuts it off
//       (renderer.cpp:283-338 under :1008-1015) -- so where sample i starts in the stream depends on samples 0 .. i-1;
//   (2) the stale hit record: reflection_hit_info lives across the samples (:286), so sample i is shaded with the closest
//       hit seen by samples 0 .. i (a prefix minimum over t, first wins).
// Both are functions of the samples' own closest hits, so the fan is a fixed point: every lane assumes a start offset
// (3 i at first), draws its direction, traces its ray; a segmented scan gives every lane its prefix-minimum hit, from its
// material the draws its nested fan consumes, a prefix sum the true offsets.  Lanes whose offset moved trace again; sample 0
// is right after the first round, sample i after at most i + 1, in practice after one or two (most fan rays hit the sky or
// a material that does not reflect).  Then every lane shades its sample, and lane 0 adds the colours in sample order.
// Same arithmetic as the sequential walk, so the same bits.  Left to k_reflect: recursion limits other than 1 (nested fans
// really trace), normal mapping (shading rewrites the shared record's normal, a third chain), more than 32 samples, the
// instrumented instantiation.
RT_DEV Hit shfl_hit(const Hit& h, int src, int width)
{
    Hit r;
    r.tri = __shfl_sync(0xffffffffu, h.tri, src, width); r.t = __shfl_sync(0xffffffffu, h.t, src, width);
    r.u = __shfl_sync(0xffffffffu, h.u, src, width); r.v = __shfl_sync(0xffffffffu, h.v, src, width);
    r.mat = __shfl_sync(0xffffffffu, h.mat, src, width);
    r.normal = v3(__shfl_sync(0xffffffffu, h.normal.x, src, width), __shfl_sync(0xffffffffu, h.normal.y, src, width), __shfl_sync(0xffffffffu, h.normal.z, src, width));
    r.tangent = v3(__shfl_sync(0xffffffffu, h.tangent.x, src, width), __shfl_sync(0xffffffffu, h.tangent.y, src, width), __shfl_sync(0xffffffffu, h.tangent.z, src, width));
    return r;
}

#ifndef RTB_FAN_MINB
#define RTB_FAN_MINB 6     /* resident CTAs per SM the compiler must allow for k_reflect_fan; measured on cfg3 at 1080p: 3 (168 registers) 4.99 ms, 4: 4.21, 5: 4.04, 6 (80): 3.99 */
#endif
__global__ void __launch_bounds__(kQueueThreads, RTB_FAN_MINB)
k_reflect_fan(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt)
{
    const uint32_t n = cnt->n_refl;
    const int S = fr.s.rough_reflections_sample_count;
    const int G = S <= 16 ? 16 : 32;                          // lanes per fan: two fans per warp up to 16 samples
    const unsigned lane = threadIdx.x & 31u;
    const int sub = (int)(lane & (unsigned)(G - 1));          // this lane's sample
    const uint32_t group = lane / (unsigned)G, per_warp = 32u / (unsigned)G;
    const uint32_t warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    unsigned overflow = 0;
    for (uint32_t first = warp_id * per_warp; first < n; first += n_warps * per_warp) {       // warp-uniform trip count
        const uint32_t r = first + group;
        const bool fan = r < n;
        const uint32_t entry = fan ? q.refl_idx[r] : 0u;
        TraceCounters tc = zero_counters();
        V3 o = v3(0, 0, 0), d = v3(0, 0, 1), p = v3(0, 0, 0);
        HitRec hr;
        hr.tri = -1; hr.t = -1.0f; hr.u = 1.0f; hr.v = 0.0f;
        uint32_t pix = 0;
        Hit hit = fresh_hit();
        MatView m = {};
        float roughness = 0.0f;
        if (fan) {
            queue_ray(fr, wk, q, entry, o, d, hr, pix);
            hit = make_hit(sc, hr, o, d);
            shade_direct(sc, fr, o, d, hit, p, m);            // (no normal mapping on this path: hit.normal is the geometric one)
            if (fr.s.enable_roughness_mapping) {
                float tu, tv;
                hit_texcoords(sc, hit, hit.u, hit.v, tu, tv);
                roughness = tex_floor(sc.tex[RT_TEX_ROUGHNESS], tu, tv).r;
            } else
                roughness = m.roughness;
        }
        const bool rough = fan && roughness > 0.0f;
        // a mirror hit is one sample without a random number: the sequential code, on the fan's first lane
        if (fan && !rough && sub == 0) {
            XorShift32 rng;
            rng.state = pixel_seed(pix, fr.s.rng_seed);
            const Col c = compute_reflection<false>(sc, fr, d, p, hit, m, 0, rng, &tc);
            q.refl_rgb[3 * (size_t)entry + 0] = c.r; q.refl_rgb[3 * (size_t)entry + 1] = c.g; q.refl_rgb[3 * (size_t)entry + 2] = c.b;
            q.refl_cnt[3 * (size_t)entry + 0] = (unsigned long long)tc.refl_rays | ((unsigned long long)tc.refl_shadow_rays << 32);
            q.refl_cnt[3 * (size_t)entry + 1] = 0ull; q.refl_cnt[3 * (size_t)entry + 2] = 0ull;
            overflow |= tc.stack_overflow;
        }
        const bool mine = rough && sub < S;                   // this lane owns a sample of a rough fan
        const V3 nrm = hit.normal;
        const V3 origin = p + 0.01f * nrm;                    // renderer.cpp:291
        const V3 mirror = d - (2 * dot(d, nrm)) * nrm;
        const uint32_t seed = pixel_seed(pix, fr.s.rng_seed);
        int my_off = 3 * sub, traced_off = -1;
        V3 dir = v3(0, 0, 1);
        Hit own = fresh_hit();                                // this sample's own closest hit (triangles, then the shapes)
        bool found = false;
        Hit fh = fresh_hit();                                 // the record this sample is shaded with
        for (int round = 0; round <= S; round++) {
            if (mine && my_off != traced_off) {
                XorShift32 rng;
                rng.state = seed;
                for (int k = 0; k < my_off; k++) rng.next();
                const float rz = rng.bilateral();             // Vector(rand, rand, rand), renderer.cpp:313: evaluated right to left
                const float ry = rng.bilateral();
                const float rx = rng.bilateral();
                V3 rv = normalize(v3(rx, ry, rz));
                if (dot(rv, nrm) < 0) rv = -rv;
                dir = roughness * rv + (1 - roughness) * mirror;
                own = fresh_hit();
                HitRec h2;
                found = trace_closest<false>(sc, origin, dir, h2, &tc);
                if (found) own = complete_hit(sc, h2);
                for (int i = 0; i < sc.n_shapes; i++) {       // renderer.cpp:1029-1037
                    float t;
                    V3 sn;
                    int32_t sm;
                    if (shape_intersect(sc, i, origin, dir, t, sn, sm) && (t < own.t || own.t == -1.0f)) {
                        own.tri = -2 - i; own.t = t; own.normal = sn; own.mat = sm;
                        found = true;
                    }
                }
                traced_off = my_off;
            }
            // prefix minimum over the samples so far, first wins: which sample's record is each sample shaded with
            float bt = (mine && found) ? own.t : INFINITY;
            int bi = sub;
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const float ot = __shfl_up_sync(0xffffffffu, bt, k, G);
                const int oi = __shfl_up_sync(0xffffffffu, bi, k, G);
                if (k < G && sub >= k && !(bt < ot)) { bt = ot; bi = oi; }      // the earlier one stays unless the later is strictly closer
            }
            const bool have = bt != INFINITY;
            const Hit src = shfl_hit(own, bi, G);
            fh = have ? src : fresh_hit();
            // draws the nested fan of that record consumes (the recursion limit stops its rays, not its random numbers)
            int consume = 0;
            if (mine && fr.s.shading_method == RT_SHADING && fh.t > 0.1f) {
                const MatView m2 = load_material(sc, fh.mat);
                if (m2.reflection > 0.0f) {
                    float r2 = m2.roughness;
                    if (fr.s.enable_roughness_mapping) {
                        float tu, tv;
                        hit_texcoords(sc, fh, fh.u, fh.v, tu, tv);
                        r2 = tex_floor(sc.tex[RT_TEX_ROUGHNESS], tu, tv).r;
                    }
                    if (r2 > 0.0f) consume = 3 * S;
                }
            }
            int before = consume;                             // exclusive prefix sum over the fan's lanes
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, before, k, G);
                if (k < G && sub >= k) before += a;
            }
            before -= consume;
            const int new_off = 3 * sub + before;
            const bool moved = mine && new_off != my_off;
            my_off = new_off;
            if (__ballot_sync(0xffffffffu, moved) == 0u) break;
        }
        // every sample's colour: trace_ray_secondary from the gate on (renderer.cpp:1039-1065), with the record above
        Col c = col(0.0f);
        if (mine) {
            tc.refl_rays++;
            if (fh.t > 0.1f) {
                if (fr.s.shading_method != RT_SHADING) c = shade_debug(sc, fr, fh);
                else {
                    V3 p2;
                    MatView m2;
                    const Col direct = shade_direct(sc, fr, origin, dir, fh, p2, m2);
                    bool shadowed = false;
                    if (fr.s.compute_shadows) {
                        tc.refl_shadow_rays++;
                        shadowed = trace_occluded<false>(sc, p2, fh.normal, fr.light, &tc) || (sc.n_shapes > 0 && shapes_occlude(sc, p2, fh.normal, fr.light));
                    }
                    // the nested fan returns (0 / samples) * reflection: its rays are beyond the recursion limit
                    c = shade_compose(fr, m2, direct, shadowed, col(0.0f));
                }
            } else
                c = shade_miss(sc, fr, dir);
        }
        overflow |= tc.stack_overflow;
        // the sum in sample order, on the fan's first lane (renderer.cpp:315-337)
        Col total = col(0.0f);
        for (int i = 0; i < S; i++) {
            const Col ci = col(__shfl_sync(0xffffffffu, c.r, i, G), __shfl_sync(0xffffffffu, c.g, i, G), __shfl_sync(0xffffffffu, c.b, i, G));
            total = total + ci;
        }
        unsigned rays = tc.refl_rays, shadow_rays = tc.refl_shadow_rays;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const unsigned a = __shfl_down_sync(0xffffffffu, rays, k, G), b = __shfl_down_sync(0xffffffffu, shadow_rays, k, G);
            if (k < G && sub + k < G) { rays += a; shadow_rays += b; }
        }
        if (rough && sub == 0) {
            const Col res = total / col((float)S) * col(m.reflection);
            q.refl_rgb[3 * (size_t)entry + 0] = res.r; q.refl_rgb[3 * (size_t)entry + 1] = res.g; q.refl_rgb[3 * (size_t)entry + 2] = res.b;
            q.refl_cnt[3 * (size_t)entry + 0] = (unsigned long long)rays | ((unsigned long long)shadow_rays << 32);
            q.refl_cnt[3 * (size_t)entry + 1] = 0ull; q.refl_cnt[3 * (size_t)entry + 2] = 0ull;
        }
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
}

// Shade + hard shadow + compose + quantise for the queued hits.  Same persistent / refill scheme as k_primary over
// the hit queue: a refilled lane shades its hit (textures, Blinn-Phong) and starts the any-hit state machine of its
// shadow ray; when that ends the lane composes the pixel (with the fan colour k_reflect left, if the material
// reflects) and stores it.
template <bool COUNT>
__global__ void __launch_bounds__(kQueueThreads)
k_shade(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    pick_hit_queue(q, cnt);
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t n = cnt->n_hits;
    TraceCounters tc = zero_counters();
    TraceCounters fan = zero_counters();                      // sums of the per-entry records of k_reflect
    RayState S;
    RayStack K;
    S.mode = RT_MODE_DONE;
    S.occluded = false;
    bool alive = false, exhausted = false;
    uint32_t entry = 0, pix = 0;
    int32_t mat = 0;
    Col direct = col(0.0f);
    for (;;) {
        const unsigned idle = __ballot_sync(0xffffffffu, !alive);
        const int n_idle = __popc(idle);
        if (!exhausted && (n_idle >= tune.shade_refill || n_idle == 32)) {
            uint32_t base = 0;
            const int leader = __ffs(idle) - 1;
            if ((int)lane == leader) base = atomicAdd(&cnt->next_shade, (unsigned)n_idle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + (uint32_t)n_idle >= n) exhausted = true;
            const uint32_t r = base + (uint32_t)__popc(idle & lt_mask);
            if (!alive && r < n) {
                entry = r;
                V3 o, d;
                HitRec hr;
                queue_ray(fr, wk, q, entry, o, d, hr, pix);
                Hit hit = make_hit(sc, hr, o, d);
                if (fr.s.shading_method != RT_SHADING) {
                    super[pix] = quantise_argb(shade_debug(sc, fr, hit));
                    if (q.g_z != nullptr) { q.g_z[pix] = -(o.z + d.z * hr.t); q.g_n[pix] = hit.normal; }
                } else {
                    V3 p;
                    MatView m;
                    direct = shade_direct(sc, fr, o, d, hit, p, m);
                    if (q.g_z != nullptr) { q.g_z[pix] = -(o.z + d.z * hr.t); q.g_n[pix] = hit.normal; }
                    mat = hit.mat;
                    S.occluded = false;
                    S.mode = RT_MODE_DONE;
                    if (fr.s.compute_shadows) any_begin<COUNT>(sc, p, hit.normal, fr.light, S, &tc);
                    alive = true;                             // ends at once when there is no shadow ray to trace
                }
            }
        }
        if (__ballot_sync(0xffffffffu, alive) == 0u) {
            if (exhausted) break;
            continue;
        }
#pragma unroll 1
        for (int it = 0; it < kStepsPerCheck; it++) warp_step<true, COUNT>(sc, S, K, &tc, alive, tune);
        if (alive && S.mode == RT_MODE_DONE) {
            alive = false;
            const MatView m = load_material(sc, mat);
            Col refl = col(0.0f);
            if (m.reflection > 0.0f) {
                refl = col(q.refl_rgb[3 * (size_t)entry], q.refl_rgb[3 * (size_t)entry + 1], q.refl_rgb[3 * (size_t)entry + 2]);
                const unsigned long long packed = q.refl_cnt[3 * (size_t)entry];
                fan.refl_rays += (uint32_t)packed;
                fan.refl_shadow_rays += (uint32_t)(packed >> 32);
                if (COUNT) {                                   // fan rays are single rays: one fetch per test
                    fan.vol_tests += q.refl_cnt[3 * (size_t)entry + 1]; fan.tri_tests += q.refl_cnt[3 * (size_t)entry + 2];
                    fan.rec_fetch += q.refl_cnt[3 * (size_t)entry + 1]; fan.tri_fetch += q.refl_cnt[3 * (size_t)entry + 2];
                }
            }
            bool occluded = S.occluded;
            if (sc.n_shapes > 0 && fr.s.compute_shadows && !occluded) occluded = shapes_occlude_ray(sc, S.o, -S.md, S.p, S.dist2);
            super[pix] = quantise_argb(shade_compose(fr, m, direct, occluded, refl));
        }
    }
    if (tc.stack_overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (COUNT) flush_work(tc, &cnt->shadow_vol, &cnt->shadow_tri, &cnt->shadow_fetch);
    const unsigned rr = __reduce_add_sync(0xffffffffu, fan.refl_rays), rs = __reduce_add_sync(0xffffffffu, fan.refl_shadow_rays);
    if ((threadIdx.x & 31u) == 0) {
        if (rr) atomicAdd(&cnt->refl_rays, (unsigned long long)rr);
        if (rs) atomicAdd(&cnt->refl_shadow_rays, (unsigned long long)rs);
    }
    if (COUNT) flush_work(fan, &cnt->refl_vol, &cnt->refl_tri, &cnt->refl_fetch);
}

// What a lane of the shading kernels knows about its hit-queue entry before the shadow ray is traced.
struct ShadeLane {
    uint32_t pix;
    int32_t mat;
    Col direct;             // diffuse * ao + specular (shade_direct), or the debug colour when !rt
    V3 p, nrm;              // shaded point and (normal-mapped) shading normal: the shadow ray starts at p + nrm * EPSILON
    bool rt;                // RT_SHADING (false: one of the debug shading modes, no further rays)
};

// gbuffer: also store what Renderer::ray_trace keeps for the SSAO pass (renderer.cpp:1104-1111): the z of the hit point and
// the hit's normal as shading left it (normal-mapped when normal mapping is on).  Only the kernel that sees every queue
// entry exactly once asks for it.
RT_DEV ShadeLane shade_prepare(const SceneView& sc, const FrameView& fr, const WorkView& wk, const QueueView& q, uint32_t entry, bool gbuffer = false)
{
    ShadeLane L;
    V3 o, d;
    HitRec hr;
    queue_ray(fr, wk, q, entry, o, d, hr, L.pix);
    Hit hit = make_hit(sc, hr, o, d);
    L.mat = hit.mat;
    L.rt = fr.s.shading_method == RT_SHADING;
    if (!L.rt) { L.direct = shade_debug(sc, fr, hit); L.p = v3(0, 0, 0); L.nrm = v3(0, 0, 1); }
    else {
        MatView m;
        L.direct = shade_direct(sc, fr, o, d, hit, L.p, m);
        L.nrm = hit.normal;
    }
    if (gbuffer && q.g_z != nullptr) {
        q.g_z[L.pix] = -(o.z + d.z * hr.t);
        q.g_n[L.pix] = hit.normal;
    }
    return L;
}

template <bool COUNT>
RT_DEV void shade_store(const SceneView& sc, const FrameView& fr, const QueueView& q, uint32_t entry, const ShadeLane& L, bool occluded,
                        TraceCounters& fan, uint32_t* super)
{
    if (!L.rt) { super[L.pix] = quantise_argb(L.direct); return; }
    if (sc.n_shapes > 0 && fr.s.compute_shadows && !occluded) occluded = shapes_occlude(sc, L.p, L.nrm, fr.light);   // renderer.cpp:376-397
    const MatView m = load_material(sc, L.mat);
    Col refl = col(0.0f);
    if (m.reflection > 0.0f) {
        refl = col(q.refl_rgb[3 * (size_t)entry], q.refl_rgb[3 * (size_t)entry + 1], q.refl_rgb[3 * (size_t)entry + 2]);
        const unsigned long long packed = q.refl_cnt[3 * (size_t)entry];
        fan.refl_rays += (uint32_t)packed;
        fan.refl_shadow_rays += (uint32_t)(packed >> 32);
        if (COUNT) {                                   // fan rays are single rays: one fetch per test
                    fan.vol_tests += q.refl_cnt[3 * (size_t)entry + 1]; fan.tri_tests += q.refl_cnt[3 * (size_t)entry + 2];
                    fan.rec_fetch += q.refl_cnt[3 * (size_t)entry + 1]; fan.tri_fetch += q.refl_cnt[3 * (size_t)entry + 2];
                }
    }
    super[L.pix] = quantise_argb(shade_compose(fr, m, L.direct, occluded, refl));
}

template <bool COUNT>
RT_DEV void shade_epilogue(ChunkCounters* cnt, TraceCounters& tc, TraceCounters& fan, unsigned overflow)
{
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (COUNT) flush_work(tc, &cnt->shadow_vol, &cnt->shadow_tri, &cnt->shadow_fetch);
    const unsigned rr = __reduce_add_sync(0xffffffffu, fan.refl_rays), rs = __reduce_add_sync(0xffffffffu, fan.refl_shadow_rays);
    if ((threadIdx.x & 31u) == 0) {
        if (rr) atomicAdd(&cnt->refl_rays, (unsigned long long)rr);
        if (rs) atomicAdd(&cnt->refl_shadow_rays, (unsigned long long)rs);
    }
    if (COUNT) flush_work(fan, &cnt->refl_vol, &cnt->refl_tri, &cnt->refl_fetch);
}

// Packet version of k_shade: a warp takes 32 consecutive hit-queue entries (neighbouring pixels, k_compact), shades
// them, traces their 32 shadow rays as one packet, composes and stores.  A packet that runs out of rounds
// (RT_OPT_PACKET_ROUNDS) stores the pixels it has an answer for and is split into work items for the rest.
template <bool COUNT, bool TOP>
__global__ void __launch_bounds__(kQueueThreads, RTB_SHADE_MINB)
k_shade_packet(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    pick_hit_queue(q, cnt);
    __shared__ PacketStack stacks[kQueueThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    __shared__ typename TopStorage<TOP>::type top_table;        // TOP: the first levels of the tree, one bulk asynchronous copy per CTA
    load_top_table(sc, top_table);
    const float4* top = top_pointer(top_table);
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = cnt->n_hits;
    TraceCounters tc = zero_counters();
    TraceCounters fan = zero_counters();
    unsigned overflow = 0;
    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&cnt->next_shade, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n) break;
        const uint32_t entry = base + lane;
        const bool valid = entry < n;
        ShadeLane L;
        L.rt = false; L.p = v3(0, 0, 0); L.nrm = v3(0, 0, 1);
        if (valid) L = shade_prepare(sc, fr, wk, q, entry, true);
        bool occluded = false, deferred = false;
        if (fr.s.compute_shadows && fr.s.shading_method == RT_SHADING) {
            bool active = valid && L.rt;
            const V3 so = L.p + 1.0e-4f * L.nrm;                               // Renderer::EPSILON, renderer.h:23
            const V3 sd = active ? normalize(fr.light - L.p) : v3(0, 0, 1);
            const float dist2 = length2(L.p - fr.light);
            const float t_lim = (sqrtf(dist2) + 4.0e-4f) * 1.0001f;
            HitRec unused;
            unsigned rounds = 0;
            const unsigned long long t0 = COUNT ? global_ns() : 0ull;
            if (!((tune.cull & 2) != 0 && packet_set_cull(K, active, fr.light, so, 2.0e-4f))) packet_no_cull(K);
            const bool finished = packet_trace<true, COUNT, true>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow,
                                                                  tune.packet_rounds, rounds, 0u, 0u, 0x7fffffff, nullptr, nullptr,
                                                                  make_drain(&cnt->next_shade, n, tune.packet_min));
            __syncwarp();
            if (COUNT && lane == 0) note_packet(cnt, 1, rounds, global_ns() - t0);
            if (!finished) {
                const unsigned dm = __ballot_sync(0xffffffffu, active);
                uint32_t sidx = 0;
                if (lane == 0) sidx = atomicAdd(&cnt->n_split, 1u);
                sidx = __shfl_sync(0xffffffffu, sidx, 0);
                if (sidx < q.split_capacity && emit_items(q, cnt->items_n, K, 0, sidx)) {
                    if (lane == 0) { q.split_base[sidx] = base; q.split_active[sidx] = dm; q.split_occ[sidx] = 0u; }
                    deferred = active;                                         // k_shade_finish stores these pixels
                } else {
                    if (sidx < q.split_capacity && lane == 0) { q.split_base[sidx] = base; q.split_active[sidx] = 0u; q.split_occ[sidx] = 0u; }
                    const bool before = occluded;                              // no room: finish here, from the root
                    packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, 0, rounds);
                    occluded = occluded || before;
                    __syncwarp();
                }
            }
        }
        if (valid && !deferred) shade_store<COUNT>(sc, fr, q, entry, L, occluded, fan, super);
    }
    shade_epilogue<COUNT>(cnt, tc, fan, overflow);
}

// Item pass `pass` (0 .. kItemPasses-1): a warp takes one work item = one unvisited cell of a split packet, rebuilds the
// packet's 32 shadow rays, traces them from that cell and ORs the newly occluded lanes into the split record.  An item
// that runs out of rounds itself is split again into the next pass's region; the last pass has no budget.
template <bool COUNT>
__global__ void __launch_bounds__(kQueueThreads, RTB_SHADE_MINB)
k_shade_items(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, Tuning tune, int pass)
{
    pick_hit_queue(q, cnt);
    __shared__ PacketStack stacks[kQueueThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    const float4* top = nullptr;                       // items start deep in the tree: no use for the top table
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n_hits = cnt->n_hits;
    const uint32_t n = min(cnt->items_n[pass], q.item_capacity);
    const uint4* region = q.items + (size_t)pass * q.item_capacity;
    const int budget = pass + 1 < tune.item_passes ? tune.item_rounds : 0;
    TraceCounters tc = zero_counters();
    unsigned overflow = 0;
    for (;;) {
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(&cnt->items_next[pass], 1u);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= n) break;
        const uint4 item = region[i];
        const uint32_t sidx = item.x;
        if (sidx == 0xffffffffu) continue;
        const uint32_t base = q.split_base[sidx];
        const uint32_t live = q.split_active[sidx] & ~*((volatile uint32_t*)&q.split_occ[sidx]);
        const uint32_t entry = base + lane;
        bool active = entry < n_hits && ((live >> lane) & 1u) != 0u;
        if (__ballot_sync(0xffffffffu, active) == 0u) continue;                // every ray has been answered meanwhile
        ShadeLane L;
        L.rt = false; L.p = v3(0, 0, 0); L.nrm = v3(0, 0, 1);
        if (active) L = shade_prepare(sc, fr, wk, q, entry);
        const V3 so = L.p + 1.0e-4f * L.nrm;
        const V3 sd = active ? normalize(fr.light - L.p) : v3(0, 0, 1);
        const float dist2 = length2(L.p - fr.light);
        const float t_lim = (sqrtf(dist2) + 4.0e-4f) * 1.0001f;
        HitRec unused;
        bool occluded = false;
        unsigned rounds = 0;
        if (!((tune.cull & 2) != 0 && packet_set_cull(K, active, fr.light, so, 2.0e-4f))) packet_no_cull(K);
        bool finished = packet_trace<true, COUNT, true>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, budget, rounds,
                                                        item.y, item.z, 0x7fffffff, nullptr, nullptr, make_drain(&cnt->items_next[pass], n, tune.item_min));
        __syncwarp();
        if (!finished && !emit_items(q, cnt->items_n, K, pass + 1, sidx)) {
            const bool before = occluded;                                      // no room: finish the item here
            packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, 0, rounds, item.y, item.z);
            occluded = occluded || before;
            __syncwarp();
        }
        const unsigned om = __ballot_sync(0xffffffffu, occluded);
        if (om != 0u && lane == 0) atomicOr(&q.split_occ[sidx], om);
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (COUNT) flush_work(tc, &cnt->shadow_vol, &cnt->shadow_tri, &cnt->shadow_fetch);
}

// After the item passes: composes and stores the pixels of the split packets' unanswered lanes with the merged answers.
template <bool COUNT>
__global__ void __launch_bounds__(kQueueThreads)
k_shade_finish(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super)
{
    pick_hit_queue(q, cnt);
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n_hits = cnt->n_hits;
    const uint32_t n = min(cnt->n_split, q.split_capacity);
    TraceCounters tc = zero_counters();
    TraceCounters fan = zero_counters();
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t sidx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; sidx < n; sidx += warps) {
        const uint32_t entry = q.split_base[sidx] + lane;
        if (entry < n_hits && ((q.split_active[sidx] >> lane) & 1u) != 0u) {
            const ShadeLane L = shade_prepare(sc, fr, wk, q, entry);
            shade_store<COUNT>(sc, fr, q, entry, L, ((q.split_occ[sidx] >> lane) & 1u) != 0u, fan, super);
        }
    }
    shade_epilogue<COUNT>(cnt, tc, fan, 0u);
}


// ---------------------------------------------------------------------------------------------------------------------
// Fused item scheduling (Tuning::fused, the default).  The item passes above are separate launches: six per stage, each
// with its own ramp-up and tail, which is a third of the frame time of a short launch (one of 8 tile shards of a 4K frame:
// 0.6 of 2.4 ms, measured).  Here the packet kernel's own persistent warps consume the work items while the launch is
// still running: one queue per stage (kSubQueues ticket queues), a warp looks for an item before it takes the next
// packet (items belong to the longest packets: starting them early shortens the critical path), and the warp that
// completes the last item of a split record stores that record's pixels.  One launch per stage, no item generations to
// wait for; the price is that items of one record run concurrently and prune each other less (an item reads the answers
// found so far when it starts).  Results cannot differ from the pass-by-pass schedule: any-hit answers are OR-ed, closest
// hits merged with the same 64-bit atomicMin.
//
// Protocol.  Producer (a packet or item that ran out of rounds): reserve n tickets in its home sub-queue (atomicAdd n),
// raise the record's pending count and the stage's reserved total by n, write the n slots nearest cell first, fence, set
// each slot's ready flag to this launch's tag.  Consumer: if next < n take ticket t = next by compare-and-swap, wait for
// slot t's flag, run the item, OR / min its
// answers into the record, fence, lower the record's pending count -- whoever reaches zero finishes the record -- and count
// the item as done.  A warp that finds neither a packet nor an item leaves -- except the PARKED warps (the CTAs with the
// lowest indices, about one per SM), which stay and poll with back-off until every packet has completed and
// done == reserved (read in that order: nothing that could still emit is running then); late items are served by them
// and by the warps that are still at work.  Nobody ever waits for a warp that is not running.
RT_DEV uint2 sq_snapshot(const SubQueue* sq)                                   // (n, next) in one 8-byte load
{
    uint2 v;
    asm volatile("ld.volatile.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(sq));
    return v;
}

RT_DEV bool fq_all_done(const FusedTotals* ft, uint32_t total_packets)
{
    // ordered reads: packets, then items done, then items reserved (an item's children are reserved before it is counted
    // as done: with every packet complete and done == reserved read in that order, nothing that could still emit is running)
    const uint32_t pd = ld_vol(&ft->packets_done);
    if (pd != total_packets) return false;
    __threadfence();
    const uint32_t done = ld_vol(&ft->done);
    __threadfence();
    const uint32_t n = ld_vol(&ft->reserved);
    return done == n;
}

// Round budget of a packet claimed when `rem` more packets per resident warp are still unclaimed, and of the items
// emitted around that time (guided self-scheduling): early in the launch a packet may run long -- there is plenty of other
// work to keep the SMs busy meanwhile --, near the end it is cut after a few rounds so that its cells spread over the
// warps that are running out of packets.  The launch's tail is about one budget long instead of one whole packet.
// (A budget that shrinks steadily over the launch -- 8 + 8 * rem -- split half of all packets and made the launch 5x slower:
// an item re-does the shading set-up of its 32 rays for a few rounds of traversal.  Only the last round of claims is cut short.)
RT_DEV int fq_budget(int max_rounds, uint32_t rem) { return max_rounds > 0 ? (rem == 0u ? max(8, max_rounds / 4) : max_rounds) : 0; }

RT_DEV uint32_t fq_home() { return (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) % (uint32_t)kSubQueues; }
RT_DEV uint32_t fq_sub_capacity(const QueueView& q) { return q.item_capacity * (uint32_t)kItemPasses / (uint32_t)kSubQueues; }

// The unvisited cells K.link/meta[0, K.saved) of split record `sidx` become items of generation `gen` in the emitting
// warp's home sub-queue.  `first`: the emitter is the packet itself (sets the record's pending count) rather than one of
// its items (raises it).  The caller has written the split record and fenced.  Returns false when the sub-queue is full:
// nothing was published and the caller finishes its rays in place (slots it was handed below the capacity get null items).
RT_DEV bool fq_emit(const QueueView& q, ChunkCounters* cnt, int stage, const PacketStack& K, uint32_t sidx, uint32_t gen, bool first)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = (uint32_t)K.saved, cap = fq_sub_capacity(q), home = fq_home();
    uint32_t at = 0;
    if (lane == 0) at = atomicAdd(&cnt->sq[stage][home].n, n);
    at = __shfl_sync(0xffffffffu, at, 0);
    const bool ok = at + n <= cap;
    if (ok && lane == 0) {
        if (first) atomicExch(&q.split_pending[sidx], n);
        else atomicAdd(&q.split_pending[sidx], n);
        atomicAdd(&cnt->ft[stage].reserved, n);
        __threadfence();
    }
    __syncwarp();
    const size_t region = (size_t)home * cap;
    for (uint32_t i = lane; i < n && at + i < cap; i += 32u) {
        const uint32_t j = n - 1u - i;                                          // the stack's top is the nearest cell: it goes first
        q.items[region + at + i] = ok ? make_uint4(sidx, K.link[j], K.meta[j], gen) : make_uint4(0xffffffffu, 0u, 0u, 0u);
        __threadfence();
        *((volatile uint32_t*)&q.item_ready[region + at + i]) = q.tag;
    }
    __syncwarp();
    return ok;
}

// Takes one item if there is one: from the warp's home sub-queue (`scan` false: one 8-byte load) or from any sub-queue,
// nearest to home first (`scan` true: every lane looks at one).  0: nothing queued (where it looked); 1: `item` holds one;
// 2: something was queued but another warp took it first.  A ticket is claimed with compare-and-swap on the value just
// read, so a warp never holds a ticket for an item that does not exist yet.
RT_DEV int fq_take(const QueueView& q, ChunkCounters* cnt, int stage, bool scan, uint4& item)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t cap = fq_sub_capacity(q), home = fq_home();
    const uint32_t mine_q = (home + lane) % (uint32_t)kSubQueues;
    uint2 v = make_uint2(0u, 0u);
    if (scan || lane == 0) v = sq_snapshot(&cnt->sq[stage][mine_q]);
    const bool avail = v.y < v.x && v.y < cap;                                  // tickets beyond the capacity are void: nothing behind them
    const unsigned am = __ballot_sync(0xffffffffu, avail);
    if (am == 0u) return 0;
    const int src = __ffs(am) - 1;
    const uint32_t sub = (home + (uint32_t)src) % (uint32_t)kSubQueues;
    const uint32_t t = __shfl_sync(0xffffffffu, v.y, src);
    int won = 0;
    if (lane == 0) won = atomicCAS(&cnt->sq[stage][sub].next, t, t + 1u) == t;
    if (!__shfl_sync(0xffffffffu, won, 0)) return 2;
    const size_t slot = (size_t)sub * cap + t;
    if (lane == 0) {
        while (ld_vol(&q.item_ready[slot]) != q.tag) __nanosleep(40);           // its producer is between reserving and publishing
        __threadfence();
    }
    __syncwarp();
    item = __ldcg(&q.items[slot]);
    return 1;
}

// One shadow item: the packet's 32 shadow rays from one unvisited cell (as k_shade_items), then completion.
template <bool COUNT>
RT_DEV void shade_item_fused(const SceneView& sc, const FrameView& fr, const WorkView& wk, const QueueView& q, ChunkCounters* cnt, uint32_t* super,
                             int item_budget, PacketStack& K, const float4* top, const uint4 item, uint32_t n_hits, TraceCounters& tc, TraceCounters& fan,
                             unsigned& overflow)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t sidx = item.x;
    if (sidx == 0xffffffffu) return;                                           // a null item (its emission found the sub-queue full): nothing to do
    const uint32_t base = __ldcg(&q.split_base[sidx]), am = __ldcg(&q.split_active[sidx]);   // written by another SM during this launch: not through L1
    const uint32_t live = am & ~ld_vol(&q.split_occ[sidx]);
    const uint32_t entry = base + lane;
    bool active = entry < n_hits && ((live >> lane) & 1u) != 0u;
    if (__ballot_sync(0xffffffffu, active) != 0u) {                            // else: every ray has been answered meanwhile
        ShadeLane L;
        L.rt = false; L.p = v3(0, 0, 0); L.nrm = v3(0, 0, 1);
        if (active) L = shade_prepare(sc, fr, wk, q, entry);
        const V3 so = L.p + 1.0e-4f * L.nrm;
        const V3 sd = active ? normalize(fr.light - L.p) : v3(0, 0, 1);
        const float dist2 = length2(L.p - fr.light);
        const float t_lim = (sqrtf(dist2) + 4.0e-4f) * 1.0001f;
        HitRec unused;
        bool occluded = false;
        unsigned rounds = 0;
        const int budget = item.w + 1u < kFusedGenerations ? item_budget : 0;
        const bool finished = packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, budget, rounds, item.y, item.z,
                                                        0x7fffffff, &q.split_occ[sidx]);
        __syncwarp();
        if (!finished && !fq_emit(q, cnt, 1, K, sidx, item.w + 1u, false)) {
            const bool before = occluded;                                      // no room: finish the item here
            packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, 0, rounds, item.y, item.z, 0x7fffffff,
                                      &q.split_occ[sidx]);
            occluded = occluded || before;
            __syncwarp();
        }
        const unsigned om = __ballot_sync(0xffffffffu, occluded);
        if (om != 0u && lane == 0) atomicOr(&q.split_occ[sidx], om);
    }
    // completion: the record's last item stores its pixels
    uint32_t left = 0;
    if (lane == 0) {
        __threadfence();
        left = atomicSub(&q.split_pending[sidx], 1u);
    }
    left = __shfl_sync(0xffffffffu, left, 0);
    if (left == 1u) {
        uint32_t occ = 0;
        if (lane == 0) { __threadfence(); occ = atomicOr(&q.split_occ[sidx], 0u); }
        occ = __shfl_sync(0xffffffffu, occ, 0);
        if (entry < n_hits && ((am >> lane) & 1u) != 0u) {
            const ShadeLane L = shade_prepare(sc, fr, wk, q, entry);
            shade_store<COUNT>(sc, fr, q, entry, L, ((occ >> lane) & 1u) != 0u, fan, super);
        }
    }
    if (lane == 0) { __threadfence(); atomicAdd(&cnt->ft[1].done, 1u); }
}

// k_shade_packet with fused item scheduling: one launch shades, traces and stores every queued hit.
template <bool COUNT>
__global__ void __launch_bounds__(kQueueThreads, RTB_SHADE_MINB)
k_shade_fused(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    __shared__ PacketStack stacks[kQueueThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    const float4* top = nullptr;                       // (the fused experiment runs without the top table)
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t n = cnt->n_hits;
    const uint32_t total_packets = (n + 31u) >> 5;
    const bool shadows = fr.s.compute_shadows && fr.s.shading_method == RT_SHADING;
    TraceCounters tc = zero_counters();
    TraceCounters fan = zero_counters();
    unsigned overflow = 0;
    bool more = true;
    uint32_t my_packets = 0;                                                    // packets this warp completed, reported once (one hot atomic less per packet)
    unsigned backoff = 250u;
    const uint32_t per_round = 32u * gridDim.x * (kQueueThreads / 32);          // queue entries the grid's warps claim in one round of claims
    uint32_t rem = n / per_round;                                               // packets per warp still unclaimed, as of this warp's last claim
    for (;;) {
        uint4 item;
        const int got = (shadows && tune.packet_rounds > 0) ? fq_take(q, cnt, 1, !more, item) : 0;
        if (got == 1) {
            shade_item_fused<COUNT>(sc, fr, wk, q, cnt, super, fq_budget(tune.item_rounds, more ? rem : 0u), K, top, item, n, tc, fan, overflow);
            backoff = 250u;
            continue;
        }
        if (!more) {
            if (got == 2) continue;                                             // items are queued, other warps were faster: try again
            // no packet left to claim and no item queued right now.  Most warps leave: late items (emitted by the packets
            // and items still running) are served by those running warps themselves and by the PARKED warps -- the CTAs
            // with the lowest indices, about one per SM -- which poll the queue, backing off, until everything is complete.
            if (!(shadows && tune.packet_rounds > 0) || blockIdx.x >= kParkCtas) break;
            bool done = false;
            if (lane == 0) done = fq_all_done(&cnt->ft[1], total_packets);
            if (__shfl_sync(0xffffffffu, done ? 1 : 0, 0)) break;
            __nanosleep(backoff);
            backoff = min(backoff * 2u, 4000u);
            continue;
        }
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&cnt->next_shade, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n) {
            more = false;
            if (lane == 0 && my_packets) { __threadfence(); atomicAdd(&cnt->ft[1].packets_done, my_packets); }
            continue;
        }
        const uint32_t entry = base + lane;
        const bool valid = entry < n;
        rem = (n - base) / per_round;
        ShadeLane L;
        L.rt = false; L.p = v3(0, 0, 0); L.nrm = v3(0, 0, 1);
        if (valid) L = shade_prepare(sc, fr, wk, q, entry, true);
        bool occluded = false, deferred = false;
        if (shadows) {
            bool active = valid && L.rt;
            const V3 so = L.p + 1.0e-4f * L.nrm;                               // Renderer::EPSILON, renderer.h:23
            const V3 sd = active ? normalize(fr.light - L.p) : v3(0, 0, 1);
            const float dist2 = length2(L.p - fr.light);
            const float t_lim = (sqrtf(dist2) + 4.0e-4f) * 1.0001f;
            HitRec unused;
            unsigned rounds = 0;
            const unsigned long long t0 = COUNT ? global_ns() : 0ull;
            const bool finished = packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow,
                                                            fq_budget(tune.packet_rounds, rem), rounds);
            __syncwarp();
            if (COUNT && lane == 0) note_packet(cnt, 1, rounds, global_ns() - t0);
            if (!finished) {
                const unsigned dm = __ballot_sync(0xffffffffu, active);
                uint32_t sidx = 0xffffffffu;
                if (lane == 0) {
                    sidx = atomicAdd(&cnt->n_split, 1u);
                    if (sidx < q.split_capacity) { q.split_base[sidx] = base; q.split_active[sidx] = dm; q.split_occ[sidx] = 0u; __threadfence(); }
                }
                sidx = __shfl_sync(0xffffffffu, sidx, 0);
                if (sidx < q.split_capacity && fq_emit(q, cnt, 1, K, sidx, 0u, true)) deferred = active;   // the record's last item stores these pixels
                else {
                    const bool before = occluded;                              // no room: finish here, from the root
                    packet_trace<true, COUNT>(sc, K, top, active, so, sd, t_lim, L.p, dist2, unused, occluded, tc, overflow, 0, rounds);
                    occluded = occluded || before;
                    __syncwarp();
                }
            }
        }
        if (valid && !deferred) shade_store<COUNT>(sc, fr, q, entry, L, occluded, fan, super);
        ++my_packets;
    }
    shade_epilogue<COUNT>(cnt, tc, fan, overflow);
}

// The slot records (or miss colour) of one split primary record once all its items have completed (as k_primary_finish).
RT_DEV void primary_finish_record(const SceneView& sc, const FrameView& fr, const WorkView& wk, const QueueView& q, uint32_t* super, uint32_t sidx,
                                  uint32_t total)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t am = __ldcg(&q.split_active[sidx]);                        // written by another SM during this launch: not through L1
    const uint32_t slot = __ldcg(&q.split_base[sidx]) + lane;
    if ((am >> lane) & 1u) {
        const unsigned long long key = atomicMin(q.split_best + (size_t)sidx * 32u + lane, kNoHitKey);   // a coherent read
        int px = 0, py = 0;
        V3 o, d;
        slot_pixel(wk, fr, slot, px, py);
        primary_ray(fr, px, py, o, d);
        bool hit = false;
        float gated_t = -1.0f;                                                 // a BVH hit with 0 < t <= min_t, see k_primary_shapes
        if (key != kNoHitKey) {
            const uint32_t tri = (uint32_t)sc.leaf_of[(uint32_t)key];
            const rt_f4* tp = sc.tris + 3 * (size_t)tri;
            float t, u, v;
            if (tri_test(RT_LDG4(tp), RT_LDG4(tp + 1), RT_LDG4(tp + 2), o, -d, t, u, v)) {
                if (t > 0.1f) {                                                // min_t, renderer.cpp:1039
                    hit = true;
                    q.slot_tri[slot] = (int32_t)tri; q.slot_t[slot] = t; q.slot_u[slot] = u; q.slot_v[slot] = v;
                } else if (t > 0.0f)
                    gated_t = t;
            }
        }
        if (!hit) {
            q.slot_tri[slot] = -1;
            if (sc.n_shapes > 0) q.slot_t[slot] = gated_t;
            super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
        }
    } else if (slot < total)
        q.slot_tri[slot] = -1;                                                 // slot without a ray
}

template <bool COUNT>
RT_DEV void primary_item_fused(const SceneView& sc, const FrameView& fr, const WorkView& wk, const QueueView& q, ChunkCounters* cnt, uint32_t* super,
                               int item_budget, PacketStack& K, const float4* top, const uint4 item, uint32_t total, TraceCounters& tc, unsigned& overflow)
{
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t sidx = item.x;
    if (sidx == 0xffffffffu) return;                                           // a null item (its emission found the sub-queue full): nothing to do
    const uint32_t base = __ldcg(&q.split_base[sidx]);
    const uint32_t slot = base + lane;
    const bool active = ((__ldcg(&q.split_active[sidx]) >> lane) & 1u) != 0u;
    int px = 0, py = 0;
    V3 o = v3(0, 0, 0), d = v3(0, 0, 1);
    if (active) { slot_pixel(wk, fr, slot, px, py); primary_ray(fr, px, py, o, d); }
    unsigned long long* mine = q.split_best + (size_t)sidx * 32u + lane;
    const unsigned long long seen = *((volatile unsigned long long*)mine);
    const float t_start = seen == kNoHitKey ? INFINITY : __uint_as_float((uint32_t)(seen >> 32));
    const int32_t orig_start = seen == kNoHitKey ? 0x7fffffff : (int32_t)(uint32_t)seen;
    HitRec best;
    bool occ, live = active;
    unsigned rounds = 0;
    const int budget = item.w + 1u < kFusedGenerations ? item_budget : 0;
    const bool finished = packet_trace<false, COUNT>(sc, K, top, live, o, d, t_start, o, 0.0f, best, occ, tc, overflow, budget, rounds, item.y, item.z, orig_start,
                                                     nullptr, q.split_best + (size_t)sidx * 32u);
    __syncwarp();
    if (active && best.tri >= 0) atomicMin(mine, closest_key(best.t, sc.orig[best.tri]));
    if (!finished && !fq_emit(q, cnt, 0, K, sidx, item.w + 1u, false)) {
        // no room: finish the item here (from its cell again, now pruned by what it has just found)
        const unsigned long long now = *((volatile unsigned long long*)mine);
        const float t2 = now == kNoHitKey ? INFINITY : __uint_as_float((uint32_t)(now >> 32));
        const int32_t o2 = now == kNoHitKey ? 0x7fffffff : (int32_t)(uint32_t)now;
        live = active;
        packet_trace<false, COUNT>(sc, K, top, live, o, d, t2, o, 0.0f, best, occ, tc, overflow, 0, rounds, item.y, item.z, o2, nullptr,
                                   q.split_best + (size_t)sidx * 32u);
        __syncwarp();
        if (active && best.tri >= 0) atomicMin(mine, closest_key(best.t, sc.orig[best.tri]));
    }
    __threadfence();                                                           // this lane's atomicMin before the pending count drops
    __syncwarp();
    uint32_t left = 0;
    if (lane == 0) left = atomicSub(&q.split_pending[sidx], 1u);
    left = __shfl_sync(0xffffffffu, left, 0);
    if (left == 1u) {
        __threadfence();
        primary_finish_record(sc, fr, wk, q, super, sidx, total);
    }
    if (lane == 0) { __threadfence(); atomicAdd(&cnt->ft[0].done, 1u); }
}

// k_primary_packet with fused item scheduling.
template <bool COUNT>
__global__ void RTB_PRIMARY_BOUNDS
k_primary_fused(SceneView sc, FrameView fr, WorkView wk, QueueView q, ChunkCounters* cnt, uint32_t* super, Tuning tune)
{
    __shared__ PacketStack stacks[kPrimaryThreads / 32];
    PacketStack& K = stacks[threadIdx.x >> 5];
    const float4* top = nullptr;                       // (the fused experiment runs without the top table)
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t pps = (uint32_t)wk.patches_per_side;
    const uint32_t total = (wk.tile_end - wk.tile_begin) * pps * pps * (uint32_t)(kPatch * kPatch);
    const uint32_t total_packets = total >> 5;                                  // a tile's slots are a multiple of 64
    TraceCounters tc = zero_counters();
    unsigned overflow = 0;
    uint32_t traced = 0;                                                        // lane 0: rays of the packets this warp traced
    uint32_t nxt = 0;                                                           // the packet claimed for the NEXT iteration (its atomic's round trip is hidden)
    if (lane == 0) nxt = atomicAdd(&cnt->next_patch, 32u);
    bool more = true;
    uint32_t my_packets = 0;                                                    // packets this warp completed, reported once
    unsigned backoff = 250u;
    const uint32_t per_round = 32u * gridDim.x * (kPrimaryThreads / 32);        // ray slots the grid's warps claim in one round of claims
    uint32_t rem = total / per_round;                                           // packets per warp still unclaimed, as of this warp's last claim
    for (;;) {
        uint4 item;
        const int got = tune.primary_rounds > 0 ? fq_take(q, cnt, 0, !more, item) : 0;
        if (got == 1) {
            primary_item_fused<COUNT>(sc, fr, wk, q, cnt, super, fq_budget(tune.item_rounds, more ? rem : 0u), K, top, item, total, tc, overflow);
            backoff = 250u;
            continue;
        }
        if (!more) {
            if (got == 2) continue;                                             // items are queued, other warps were faster: try again
            if (tune.primary_rounds <= 0 || blockIdx.x >= kParkCtas) break;     // see k_shade_fused: only the parked warps wait for late items
            bool done = false;
            if (lane == 0) done = fq_all_done(&cnt->ft[0], total_packets);
            if (__shfl_sync(0xffffffffu, done ? 1 : 0, 0)) break;
            __nanosleep(backoff);
            backoff = min(backoff * 2u, 4000u);
            continue;
        }
        const uint32_t base = __shfl_sync(0xffffffffu, nxt, 0);
        if (base >= total) {
            more = false;
            if (lane == 0 && my_packets && tune.primary_rounds > 0) { __threadfence(); atomicAdd(&cnt->ft[0].packets_done, my_packets); }
            continue;
        }
        if (lane == 0) nxt = atomicAdd(&cnt->next_patch, 32u);
        rem = (total - base) / per_round;
        const uint32_t slot = base + lane;
        int px = 0, py = 0;
        const bool active = slot_pixel(wk, fr, slot, px, py);
        V3 o = v3(0, 0, 0), d = v3(0, 0, 1);
        // a block that the scene does not cover misses without a ray being set up
        const bool inside = active && covered(wk, px, py);
        bool deferred = false;
        if (__ballot_sync(0xffffffffu, inside) == 0u) {
            q.slot_tri[slot] = -1;
            if (active) {
                if (miss_needs_ray(fr)) primary_ray(fr, px, py, o, d);
                super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
            }
        } else {
            if (active) primary_ray(fr, px, py, o, d);
            traced += (uint32_t)__popc(__ballot_sync(0xffffffffu, active));
            HitRec best;
            bool occ, live = active;
            unsigned rounds = 0;
            const unsigned long long t0 = COUNT ? global_ns() : 0ull;
            const bool finished = packet_trace<false, COUNT>(sc, K, top, live, o, d, INFINITY, o, 0.0f, best, occ, tc, overflow,
                                                             fq_budget(tune.primary_rounds, rem), rounds);
            __syncwarp();
            if (COUNT && lane == 0) note_packet(cnt, 0, rounds, global_ns() - t0);
            if (!finished) {
                // out of rounds: the closest hits so far go to a split record, every unvisited cell becomes a work item
                const unsigned am = __ballot_sync(0xffffffffu, active);
                uint32_t sidx = 0xffffffffu;
                if (lane == 0) sidx = atomicAdd(&cnt->p_split, 1u);
                sidx = __shfl_sync(0xffffffffu, sidx, 0);
                if (sidx < q.split_capacity) {
                    if (lane == 0) { q.split_base[sidx] = base; q.split_active[sidx] = am; }
                    q.split_best[(size_t)sidx * 32u + lane] = (active && best.tri >= 0) ? closest_key(best.t, sc.orig[best.tri]) : kNoHitKey;
                    __threadfence();
                    __syncwarp();
                    deferred = fq_emit(q, cnt, 0, K, sidx, 0u, true);           // the record's last item writes these slots
                }
                if (!deferred) {
                    live = active;                                             // no room: trace it here, from the root
                    packet_trace<false, COUNT>(sc, K, top, live, o, d, INFINITY, o, 0.0f, best, occ, tc, overflow, 0, rounds);
                    __syncwarp();
                }
            }
            if (!deferred) {
                const bool hit = active && best.tri >= 0 && best.t > 0.1f;        // t > 0 (bvh.h:247) and min_t (renderer.cpp:1039)
                q.slot_tri[slot] = hit ? best.tri : -1;
                if (hit) { q.slot_t[slot] = best.t; q.slot_u[slot] = best.u; q.slot_v[slot] = best.v; }
                else if (active) {
                    if (sc.n_shapes > 0) q.slot_t[slot] = (best.tri >= 0 && best.t > 0.0f) ? best.t : -1.0f;   // see k_primary_shapes
                    super[(size_t)py * fr.rw + px] = quantise_argb(shade_miss(sc, fr, d));
                }
            }
        }
        ++my_packets;
    }
    if (overflow) atomicOr(&cnt->stack_overflow, 1u);
    if (lane == 0 && traced) atomicAdd(&cnt->traced_primary, (unsigned long long)traced);
    if (COUNT) flush_work(tc, &cnt->primary_vol, &cnt->primary_tri, &cnt->primary_fetch);
}

// The tiles that lie outside the screen-space bound of the scene (WorkView::cull_*): every sample is a miss
// (renderer.cpp:1052-1065).  One thread per supersampled pixel, rows of a tile are contiguous in the sample buffer.
__global__ void k_fill_miss(SceneView sc, FrameView fr, WorkView wk, uint32_t* super)
{
    const uint32_t n_tiles = wk.tile_end - wk.tile_begin;
    const uint32_t background = quantise_argb(shade_miss(sc, fr, v3(0, 0, 1)));
    if (!miss_needs_ray(fr) && (wk.tile_px & 3) == 0 && (fr.rw & 3) == 0 && (reinterpret_cast<uintptr_t>(super) & 15u) == 0) {
        // constant colour, rows of a tile are whole 16-byte groups: one 128-bit store per thread and step
        const uint32_t groups_per_row = (uint32_t)wk.tile_px >> 2;
        const uint32_t per_tile = groups_per_row * (uint32_t)wk.tile_px;
        const uint4 c4 = make_uint4(background, background, background, background);
        for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const uint32_t tile = wk.tiles[wk.tile_begin + t];
            const int x0 = (int)(tile % (uint32_t)wk.tiles_x) * wk.tile_px, y0 = (int)(tile / (uint32_t)wk.tiles_x) * wk.tile_px;
            for (uint32_t g = threadIdx.x; g < per_tile; g += blockDim.x) {
                const int px = x0 + (int)((g % groups_per_row) << 2), py = y0 + (int)(g / groups_per_row);
                if (px < fr.rw && py < fr.rh) *reinterpret_cast<uint4*>(super + (size_t)py * fr.rw + px) = c4;
            }
        }
        return;
    }
    const uint32_t per_tile = (uint32_t)wk.tile_px * (uint32_t)wk.tile_px;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t tile = wk.tiles[wk.tile_begin + t];
        const int x0 = (int)(tile % (uint32_t)wk.tiles_x) * wk.tile_px, y0 = (int)(tile / (uint32_t)wk.tiles_x) * wk.tile_px;
        for (uint32_t g = threadIdx.x; g < per_tile; g += blockDim.x) {
            const int px = x0 + (int)(g % (uint32_t)wk.tile_px), py = y0 + (int)(g / (uint32_t)wk.tile_px);
            if (px >= fr.rw || py >= fr.rh) continue;
            uint32_t c = background;
            if (miss_needs_ray(fr)) {
                V3 o, d;
                primary_ray(fr, px, py, o, d);
                c = quantise_argb(shade_miss(sc, fr, d));
            }
            super[(size_t)py * fr.rw + px] = c;
        }
    }
}

// ImageUtils::downscale_image_qt_ARGB32 -- imageUtils.h:98-147: per channel, sum of the factor^2 quantised samples
// divided (integer, truncating) by factor^2.  One thread per final pixel of the owned tiles.
// Tiles at list positions >= n_box were not traced (they lie outside the screen-space bound of the scene) and their miss
// colour does not depend on the ray: every one of their samples would be `fill`, whose box filter is `fill` again, so
// the final pixel is written directly and the samples never exist (no 0.5 GB constant round trip through HBM).
__global__ void k_resolve(const uint32_t* super, uint32_t* out, WorkView wk, int tile_size, int factor, int width, int height, uint32_t n_box,
                          uint32_t fill)
{
    const uint32_t per_tile = (uint32_t)tile_size * (uint32_t)tile_size;
    const uint64_t total = (uint64_t)(wk.tile_end - wk.tile_begin) * per_tile;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t tpos = wk.tile_begin + (uint32_t)(g / per_tile);
        const uint32_t tile = wk.tiles[tpos];
        const uint32_t in = (uint32_t)(g % per_tile);
        const int x = (int)(tile % (uint32_t)wk.tiles_x) * tile_size + (int)(in % (uint32_t)tile_size);
        const int y = (int)(tile / (uint32_t)wk.tiles_x) * tile_size + (int)(in / (uint32_t)tile_size);
        if (x >= width || y >= height) continue;
        if (tpos >= n_box) { out[(size_t)y * width + x] = fill; continue; }
        const int rw = width * factor;
        int ar = 0, ag = 0, ab = 0;
        for (int i = 0; i < factor; i++) {
            const uint32_t* row = super + (size_t)(y * factor + i) * rw + (size_t)x * factor;
            for (int j = 0; j < factor; j++) {
                uint32_t c = __ldg(row + j);
                ar += (int)((c >> 16) & 0xffu);
                ag += (int)((c >> 8) & 0xffu);
                ab += (int)(c & 0xffu);
            }
        }
        const int ff = factor * factor;
        ar /= ff; ag /= ff; ab /= ff;
        out[(size_t)y * width + x] = 0xff000000u | ((uint32_t)(ar & 0xff) << 16) | ((uint32_t)(ag & 0xff) << 8) | (uint32_t)(ab & 0xff);
    }
}

// Tile pack / unpack between the row-major frame and the tile-major staging buffer of the all-gather.
__global__ void k_pack_tiles(const uint32_t* frame, uint32_t* staging, WorkView wk, int tile_size, int width, int height, int unpack,
                             uint32_t* frame_out)
{
    const uint32_t per_tile = (uint32_t)tile_size * (uint32_t)tile_size;
    const uint64_t total = (uint64_t)(wk.tile_end - wk.tile_begin) * per_tile;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t tile = wk.tiles[wk.tile_begin + (uint32_t)(g / per_tile)];
        const uint32_t in = (uint32_t)(g % per_tile);
        const int x = (int)(tile % (uint32_t)wk.tiles_x) * tile_size + (int)(in % (uint32_t)tile_size);
        const int y = (int)(tile / (uint32_t)wk.tiles_x) * tile_size + (int)(in / (uint32_t)tile_size);
        if (x >= width || y >= height) {
            if (!unpack) staging[g] = 0u;
            continue;
        }
        if (unpack) frame_out[(size_t)y * width + x] = staging[g];
        else staging[g] = frame[(size_t)y * width + x];
    }
}

// The other half of the gather in ONE launch: `gathered` holds the staging buffers of all `mod` shards back to back
// (per_shard tiles each, padded), `lists` their tile indices (0xffffffff = padding).  Tiles of shard `self` are skipped
// (they are already in the frame).
__global__ void k_unpack_gathered(const uint32_t* gathered, uint32_t* frame, const uint32_t* lists, uint32_t per_shard, int mod, int self,
                                  int tiles_x, int tile_size, int width, int height)
{
    const uint32_t per_tile = (uint32_t)tile_size * (uint32_t)tile_size;
    const uint64_t total = (uint64_t)per_shard * (uint64_t)mod * per_tile;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t slot = (uint32_t)(g / per_tile);                  // = shard * per_shard + tile position
        if ((int)(slot / per_shard) == self) continue;
        const uint32_t tile = lists[slot];
        if (tile == 0xffffffffu) continue;
        const uint32_t in = (uint32_t)(g % per_tile);
        const int x = (int)(tile % (uint32_t)tiles_x) * tile_size + (int)(in % (uint32_t)tile_size);
        const int y = (int)(tile / (uint32_t)tiles_x) * tile_size + (int)(in / (uint32_t)tile_size);
        if (x < width && y < height) frame[(size_t)y * width + x] = gathered[g];
    }
}

// Batched BVH::intersect (bvh.h:307).
__global__ void __launch_bounds__(kQueueThreads)
k_intersect(SceneView sc, const float* o3, const float* d3, size_t n, const int32_t* orig, int32_t* tri_id, float* t, float* u,
            float* v, unsigned int* overflow)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        V3 o = v3(o3[3 * i], o3[3 * i + 1], o3[3 * i + 2]);
        V3 d = v3(d3[3 * i], d3[3 * i + 1], d3[3 * i + 2]);
        HitRec hr;
        TraceCounters tc = zero_counters();
        bool found = trace_closest<false>(sc, o, d, hr, &tc);
        if (tc.stack_overflow) atomicOr(overflow, 1u);
        if (tri_id) tri_id[i] = found ? orig[hr.tri] : -1;
        if (t) t[i] = found ? hr.t : -1.0f;
        if (u) u[i] = found ? hr.u : 0.0f;
        if (v) v[i] = found ? hr.v : 0.0f;
    }
}

// Batched Renderer::is_shadowed (renderer.cpp:340-402).
__global__ void __launch_bounds__(kQueueThreads)
k_occluded(SceneView sc, V3 light, const float* p3, const float* n3, size_t n, uint8_t* occluded, unsigned int* overflow)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        V3 p = v3(p3[3 * i], p3[3 * i + 1], p3[3 * i + 2]);
        V3 nn = v3(n3[3 * i], n3[3 * i + 1], n3[3 * i + 2]);
        TraceCounters tc = zero_counters();
        occluded[i] = (trace_occluded<false>(sc, p, nn, light, &tc) || (sc.n_shapes > 0 && shapes_occlude(sc, p, nn, light))) ? 1 : 0;
        if (tc.stack_overflow) atomicOr(overflow, 1u);
    }
}

// Primary rays only (renderer.cpp:1083-1098), pixel-major.
__global__ void k_raygen(FrameView fr, float* o3, float* d3)
{
    const size_t n = (size_t)fr.rw * fr.rh;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        V3 o, d;
        primary_ray(fr, (int)(i % (size_t)fr.rw), (int)(i / (size_t)fr.rw), o, d);
        o3[3 * i] = o.x; o3[3 * i + 1] = o.y; o3[3 * i + 2] = o.z;
        d3[3 * i] = d.x; d3[3 * i + 1] = d.y; d3[3 * i + 2] = d.z;
    }
}

} // namespace rtb
