// rtb200.cu -- implementation of the C ABI in include/rtb200.h: context, HBM-resident scene, wavefront driver.
// There is no CPU path: every entry point that computes launches the kernels of kernels.cuh on the context's device.
#include "../../include/rtb200.h"

#include <cuda_runtime.h>
#include <omp.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "kernels.cuh"
#include "scene_layout.h"
#include "octree_device.cuh"
#include "light_cull.cuh"
#include "ssao.cuh"
#include "raster.cuh"
#include "host_common.h"

using namespace rtb;

namespace {

constexpr uint64_t kChunkPixels = 1ull << 28;     // supersampled pixels per wavefront chunk (bounds queue memory: 20 B per pixel)
constexpr int kMaxChunks = 256;
constexpr uint32_t kCoverBoxes = 4096;           // the screen coverage's box set: the deepest level of the wide tree with at most this many nodes

thread_local std::string g_create_error;
std::atomic<unsigned long long> g_alloc_generation{0};   // bumped whenever a device buffer moves: invalidates the captured frame graphs

double now_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t count)
    {
        if (count <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) n = count;
        g_alloc_generation++;
        return e;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        g_alloc_generation++;
    }
};

struct Texture {
    void* d = nullptr;
    int w = 0, h = 0, format = 0;
};

enum Stage { ST_PRIMARY = 0, ST_COMPACT, ST_REFLECT, ST_SHADE, ST_RESOLVE, ST_COUNT };

struct TimedLaunch {
    int stage;
    cudaEvent_t a, b;
    const char* label;      // non-null: a single launch timed for RTB200_TRACE only (not added to the stage sums)
};

// Device copy of a shard's tile list (owned_tiles), uploaded once per (frame size, tile size, shard) and kept.
struct TileList {
    uint32_t* d = nullptr;
    uint32_t count = 0;
    int tiles_x = 0;
    std::vector<uint32_t> host;
    // the list split by the screen-space bound of the scene (rt_render_device): tiles that can contain a hit are traced,
    // the others only get the miss colour.  Re-uploaded when the bound changes.
    uint32_t* d_split = nullptr;         // traced tiles first, then the others; `count` entries
    std::vector<uint32_t> split_host;
    uint32_t n_traced = 0;
    uint64_t split_cover = 0;            // cover_generation the split was made with
    int32_t split_tile_px = 0;
    bool split_valid = false;
    float last_hit_fraction = -1.0f;     // hits per traced ray slot of the last frame rendered with this list (-1: none yet)
};
typedef std::tuple<int, int, int, int, int> TileKey;      // width, height, tile_size, tile_mod, tile_rem (-1: all shards, padded)

} // namespace

constexpr int kLanes = 2;        // chunks in flight by default
constexpr int kMaxLanes = 6;     // ... at most (RT_OPT_LANES)

// The per-frame work buffers of ONE wavefront chunk in flight.
struct QueueSet {
    DevBuf<uint32_t> hit_slot, refl_idx, split_base, split_active, split_occ, item_ready, split_pending;
    DevBuf<uint32_t> hit_sorted, sort_keys, sort_bins;       // light-space ordering of the hit queue (RT_OPT_SHADOW_SORT)
    DevBuf<unsigned long long> split_best, refl_cnt;
    DevBuf<uint4> items;
    DevBuf<int32_t> tri;
    DevBuf<float> t, u, v, refl_rgb;
    void release()
    {
        hit_slot.release(); refl_idx.release(); split_base.release(); split_active.release(); split_occ.release(); split_best.release();
        item_ready.release(); split_pending.release(); hit_sorted.release(); sort_keys.release(); sort_bins.release();
        refl_cnt.release(); items.release(); tri.release(); t.release(); u.release(); v.release(); refl_rgb.release();
    }
};

struct Pending {                          // a frame that has been enqueued (rt_render_device_begin) and not yet ended
    bool active = false;
    ChunkCounters* host_cnt = nullptr;    // pinned, so that the read-back really is asynchronous
    size_t host_cap = 0;
    uint32_t n_chunks = 0, launches = 0;
    bool count = false, shadow = false;
    bool raster = false;                  // a raster_trace frame: `primary_rays` = the fragments whose ray was tested against their piece
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    uint64_t primary_rays = 0;
    bool has_key = false;                 // the tile list of the frame and its traced ray slots (for TileList::last_hit_fraction)
    int key[5] = {0, 0, 0, 0, 0};
    uint64_t traced_slots = 0;
};

// Device copies of the caller's triangle arrays and the temporaries of the device octree build (octree_device.cuh); kept
// between builds: set_object_transform rebuilds the tree again and again (renderer.cpp:214-224).
struct DeviceBuild {
    DevBuf<float> xyz9, uv6, centroid, c_nr, c_fr;
    DevBuf<int32_t> mat;
    DevBuf<unsigned long long> keys[2];
    DevBuf<uint32_t> idx[2], hist, sums, counts, c_begin, c_end, c_first, c_info, c_size, c_rec, c_block;
    DevBuf<uint32_t> w_src, w_members, w_need; // build_wide_tree: the record of recs[] behind each wide node, a frontier's blocks,
                                              // each node's packet stack need (k_wb_size)
    DevBuf<float> w_boxes;                    // build_wide_tree: the box set of the screen coverage (k_wb_boxes)
    DevBuf<devbuild::Stats> stats;
    bool tris_on_device = false;             // xyz9 / uv6 / mat above hold the caller's current triangles
    std::vector<M4> host_pending;            // transforms applied to the device copy but not yet to RtContext::xyz9
    void release()
    {
        xyz9.release(); uv6.release(); centroid.release(); c_nr.release(); c_fr.release(); mat.release(); keys[0].release(); keys[1].release();
        idx[0].release(); idx[1].release(); hist.release(); sums.release(); counts.release(); c_begin.release(); c_end.release(); c_first.release();
        c_info.release(); c_size.release(); c_rec.release(); c_block.release(); w_src.release(); w_members.release(); w_boxes.release(); stats.release();
    }
};

struct RtContext {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // the stream in use
    cudaStream_t own_stream = nullptr;   // created by rt_create
    std::string error;

    // host copy of the caller's triangles (set_object_transform re-transforms and rebuilds, renderer.cpp:214-224)
    std::vector<float> xyz9, uv6;
    std::vector<int32_t> mat;
    bool has_uv = false, has_mat = false;
    int32_t max_mat_index = -1, min_mat_index = 0;

    bool bvh_valid = false;
    RtBvhInfo info{};
    DevBuf<float4> d_recs, d_tris, d_shade, d_mats, d_top;
    DevBuf<float4> d_wrecs;              // the wide copy of the tree for the packet kernels (build_wide_tree)
    bool wide_tree = false;              // d_wrecs holds it (RT_OPT_LEAF_SPLIT > 0); else the packets traverse d_recs
    uint64_t n_wrecs = 0;                // records in d_wrecs
    uint32_t wide_stack = 0;             // the most packet stack entries a traversal of d_wrecs can hold (build_wide_tree)
    uint64_t tree_serial = 0;            // bumped by every build of the tree (rt_build_bvh, rt_transform_triangles)
    int top_n = 0;                       // records of the top table, built over the array the packets traverse
    DevBuf<int32_t> d_orig, d_leaf_of;
    std::vector<HostShape> shapes;       // analytic shapes, in the order they were added
    DevBuf<float4> d_shapes;
    uint32_t n_tris = 0;
    int n_mats = 0;
    bool any_reflective = false;
    Texture tex[RT_TEX_COUNT];

    M4 proj_inv{}, cam_to_world{};
    V3 cam_pos{0, 0, 0};
    V3 light{3, 3, 2};                            // PointLight default, scene/light.h:8
    bool camera_set = false;

    // per-frame work buffers
    DevBuf<uint32_t> d_super, d_frame;
    std::map<TileKey, TileList> tile_lists;
    QueueSet qs[kMaxLanes];              // ray queues of the wavefront chunks in flight (one per lane, see rt_render_device_begin)
    cudaStream_t lane_stream[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // streams of lanes 1.. (created on first use; lane 0 = the context's stream)
    cudaEvent_t lane_fork = nullptr, lane_join[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    DevBuf<ChunkCounters> d_counters;
    DevBuf<unsigned int> d_flag;
    std::vector<cudaEvent_t> event_pool;
    size_t events_used = 0;
    std::vector<TimedLaunch> timed;
    size_t stack_limit_set = 0;
    bool opt_count_work = false;
    int opt_leaf_split = 8;
    Tuning tune{16, 16, 8, 1, -256, -16, -256, 0, 0, 0, 0, kItemPasses, 3};
    uint32_t frame_serial = 0;           // tags the ready flags of the fused item queues: (serial << 2) | stage
    uint64_t opt_chunk_pixels = kChunkPixels;
    Pending pending;
    uint32_t* h_frame = nullptr;         // pinned staging buffer of rt_frame_to_host / rt_render
    size_t h_frame_cap = 0;
    cudaEvent_t copy_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // one per slice of that copy
    int grids[2][11] = {{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}};   // persistent-grid sizes of the kernels, by COUNT flag
    int grid_intersect = 0, grid_occluded = 0, grid_fan = 0;           // the same for the batch kernels (per context: its device's occupancy)
    bool opt_screen_cull = true;
    int opt_lanes = kLanes;
    bool opt_top_table = false;
    int opt_shadow_sort = 2;
    bool opt_device_build = true;
    DeviceBuild db;
    // SSAO post-process (ssao.cuh): G-buffers, counts, and the camera's forward projection (rt_set_projection)
    DevBuf<float> d_gz;
    DevBuf<V3> d_gn;
    DevBuf<int> d_ao;
    // hybrid raster path (raster.cuh): z-keys and pixel points per supersampled pixel, work units of the large pieces,
    // per-thread shading records of the pieces being shaded
    DevBuf<unsigned long long> d_rkeys;
    DevBuf<float2> d_rxy;
    DevBuf<RasterUnit> d_runits;
    DevBuf<unsigned int> d_rcount;
    DevBuf<float4> d_rfrag;
    size_t raster_smem_set = 0;
    // The frame as a CUDA graph (RT_OPT_GRAPH): when a frame's launch sequence is byte for byte the one of the frame before
    // (same settings, camera, light, buffers, options), it is captured once and replayed with one cudaGraphLaunch.
    bool opt_graph = true;
    bool opt_fan_lanes = true;           // RT_OPT_FAN_LANES
    bool capturing = false;              // stage timers are off while the launches are being captured
    struct FrameGraph { std::string key; cudaGraphExec_t exec; uint32_t launches; };
    std::vector<FrameGraph> graphs;      // the last few captured frames (a sharded frame alternates between two output buffers)
    std::vector<std::string> seen_keys;  // serialised launch parameters of the last few frames that were enqueued the ordinary way
    size_t raster_units0 = (size_t)1 << 18;   // first size of the unit list (RT_OPT_RASTER_UNITS); grown when a frame needs more
    M4 proj{};
    float proj_fov = 45.0f, proj_aspect = 1.0f;
    bool proj_set = false;
    float root_lo[3] = {0, 0, 0}, root_hi[3] = {0, 0, 0};   // the root cell's axis-aligned box (first three slabs)
    // The screen coverage of the primary packets (screen_coverage): a box set whose union holds every triangle, taken from the
    // upper levels of the tree at every build, and one bit per 8x4 block of the supersampled frame, set when the block's rays
    // can reach a box.  Rebuilt at the first frame after its inputs change, like the light masks.
    std::vector<float> cover_boxes;      // 6 per box: lo xyz, hi xyz (the records' padded axis slabs)
    struct CoverInputs { M4 proj_inv, cam_to_world; V3 cam_pos; int32_t rw, rh; uint64_t tree; } cover_in{};
    bool cover_valid = false;
    bool cover_bound = false;            // false: no bound exists, every block is traced (wk.cover = null)
    int32_t cover_words = 0;             // 32-bit words per row of blocks
    std::vector<uint32_t> h_cover;
    DevBuf<uint32_t> d_cover;
    uint64_t cover_generation = 0;       // part of the frame-graph key and of the tile split

    // per-light masks of the shadow packets (light_cull.cuh), over the array the packets traverse; rebuilt at the first frame
    // after their inputs change
    bool opt_light_cull = true;          // RT_OPT_LIGHT_CULL
    DevBuf<uint32_t> d_tri_occ, d_blk_occ, d_rec_parent;
    struct LightMaskInputs { V3 light; float span; uint32_t all_set; uint64_t tree; } mask_in{}, mask_next{};
    uint32_t mask_words = 0, mask_recs = 0;   // words of tri_occ, records of the traversed array
    bool mask_valid = false;
    uint64_t mask_generation = 0;        // part of the frame-graph key

    // rt_render_work_map: one RtPixelWork per final pixel, allocated at the first call and grown as needed.  Plain cudaMalloc,
    // not a DevBuf: the map is no input of any captured frame, so (re)allocating it must not invalidate the frame graphs.
    unsigned long long* d_work_map = nullptr;
    size_t work_map_pixels = 0;
    unsigned long long* frame_work_map = nullptr;   // set for the duration of one rt_render_work_map frame: forces COUNT, no graph
    std::vector<unsigned long long*> work_map_ptrs; // the pointer once per chunk, the source of its copy into the chunks' counters

    // batch query staging
    DevBuf<float> b_a, b_b, b_t, b_u, b_v;
    DevBuf<int32_t> b_id;
    DevBuf<uint8_t> b_occ;
};

namespace {

int fail(RtContext* ctx, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->error = buf;
    else g_create_error = buf;
    return code;
}

#define RT_CUDA(ctx, expr)                                                                                  \
    do {                                                                                                    \
        cudaError_t e__ = (expr);                                                                           \
        if (e__ != cudaSuccess) return fail(ctx, RT_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__));   \
    } while (0)

int bind(RtContext* ctx)
{
    RT_CUDA(ctx, cudaSetDevice(ctx->device));
    return RT_OK;
}

cudaEvent_t next_event(RtContext* ctx)
{
    if (ctx->events_used == ctx->event_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ctx->event_pool.push_back(e);
    }
    return ctx->event_pool[ctx->events_used++];
}

struct ScopedTimer {
    RtContext* ctx;
    TimedLaunch tl;
    cudaStream_t stream;
    bool on;
    ScopedTimer(RtContext* c, int stage, cudaStream_t st = nullptr, const char* label = nullptr) : ctx(c), stream(st ? st : c->stream)
    {
        static const bool trace = getenv("RTB200_TRACE") != nullptr;
        on = (label == nullptr || trace) && !c->capturing;
        if (!on) return;
        tl.stage = stage;
        tl.label = label;
        tl.a = next_event(c);
        tl.b = next_event(c);
        cudaEventRecord(tl.a, stream);
    }
    ~ScopedTimer()
    {
        if (!on) return;
        cudaEventRecord(tl.b, stream);
        ctx->timed.push_back(tl);
    }
};

SceneView scene_view(const RtContext* ctx)
{
    SceneView sc;
    memset(&sc, 0, sizeof(sc));
    sc.recs = ctx->d_recs.p;
    sc.top = ctx->d_top.p;
    sc.top_n = ctx->top_n;
    sc.tris = ctx->d_tris.p;
    sc.shade = ctx->d_shade.p;
    sc.mats = ctx->d_mats.p;
    sc.orig = ctx->d_orig.p;
    sc.leaf_of = ctx->d_leaf_of.p;
    sc.shapes = ctx->d_shapes.p;
    sc.n_shapes = (int32_t)ctx->shapes.size();
    sc.n_mats = ctx->n_mats;
    sc.n_tris = ctx->n_tris;
    for (int i = 0; i < RT_TEX_COUNT; i++) {
        sc.tex[i].data = ctx->tex[i].d;
        sc.tex[i].w = ctx->tex[i].w;
        sc.tex[i].h = ctx->tex[i].h;
        sc.tex[i].format = ctx->tex[i].format;
    }
    return sc;
}

// The view of the packet kernels (packet_trace and the kernels of its work items): the wide tree.  The single-ray kernels
// keep the reference-shaped recs[], whose traversal tallies are those of the host emulation.
SceneView packet_view(const RtContext* ctx)
{
    SceneView sc = scene_view(ctx);
    if (ctx->wide_tree) sc.recs = ctx->d_wrecs.p;
    sc.tri_occ = ctx->d_tri_occ.p;
    sc.blk_occ = (const uint16_t*)ctx->d_blk_occ.p;
    return sc;
}

// Decides whether the light-cull masks must be rebuilt for the next frame (the light's bits, the tree, the analytic shapes
// or RT_OPT_LIGHT_CULL changed) and sizes their buffers.  The rebuild itself is enqueued by build_light_masks on the
// frame's stream before the frame's launches or graph, never inside a captured graph; mask_generation goes into the graph
// key, so a graph is only replayed over the masks it was captured with.
int plan_light_masks(RtContext* ctx, bool& rebuild)
{
    RtContext::LightMaskInputs in;
    memset(&in, 0, sizeof(in));                                               // compared bytewise
    in.light = ctx->light;
    in.tree = ctx->tree_serial;
    in.all_set = ctx->opt_light_cull ? 0u : 1u;
    // span: the longest shadow ray, from a hit point in the root box or on an analytic sphere (light_cull.cuh)
    double far2 = 0.0;
    auto corners = [&](const double lo[3], const double hi[3]) {
        for (int c = 0; c < 8; c++) {
            const double x = (c & 1 ? hi[0] : lo[0]) - in.light.x, y = (c & 2 ? hi[1] : lo[1]) - in.light.y, z = (c & 4 ? hi[2] : lo[2]) - in.light.z;
            far2 = std::max(far2, x * x + y * y + z * z);
        }
    };
    const double rlo[3] = {ctx->root_lo[0], ctx->root_lo[1], ctx->root_lo[2]}, rhi[3] = {ctx->root_hi[0], ctx->root_hi[1], ctx->root_hi[2]};
    corners(rlo, rhi);
    for (const HostShape& sh : ctx->shapes) {
        if (sh.bits >> 31) { in.all_set = 1u; continue; }                      // a plane: hit points anywhere
        const double r = std::sqrt((double)sh.radius2);
        const double lo[3] = {sh.a[0] - r, sh.a[1] - r, sh.a[2] - r}, hi[3] = {sh.a[0] + r, sh.a[1] + r, sh.a[2] + r};
        corners(lo, hi);
    }
    in.span = (float)(1.01 * std::sqrt(far2) + 1e-3);
    if (!std::isfinite(in.span)) in.all_set = 1u;
    rebuild = !ctx->mask_valid || memcmp(&in, &ctx->mask_in, sizeof(in)) != 0;
    if (!rebuild) return RT_OK;
    const uint64_t n_recs = ctx->wide_tree ? ctx->n_wrecs : ctx->info.child_records;
    ctx->mask_words = ctx->n_tris / 32u + 2u;                                   // + 1: a leaf round reads the word after its bits
    ctx->mask_recs = (uint32_t)n_recs;
    RT_CUDA(ctx, ctx->d_tri_occ.ensure(ctx->mask_words));
    RT_CUDA(ctx, ctx->d_blk_occ.ensure(ctx->mask_recs / 4u + 1u));             // 16 bits per even record
    RT_CUDA(ctx, ctx->d_rec_parent.ensure(ctx->mask_recs));
    ctx->mask_next = in;
    ctx->mask_generation++;
    return RT_OK;
}

int build_light_masks(RtContext* ctx, cudaStream_t st)
{
    using namespace lightcull;
    ScopedTimer tm(ctx, ST_SHADE, st, "light_mask");
    const RtContext::LightMaskInputs& in = ctx->mask_next;
    const uint32_t n_words = ctx->mask_words, n_recs = ctx->mask_recs, blk_bytes = (n_recs / 4u + 1u) * 4u;
    if (in.all_set) {
        RT_CUDA(ctx, cudaMemsetAsync(ctx->d_tri_occ.p, 0xff, n_words * sizeof(uint32_t), st));
        RT_CUDA(ctx, cudaMemsetAsync(ctx->d_blk_occ.p, 0xff, blk_bytes, st));
    } else {
        const float4* recs = ctx->wide_tree ? ctx->d_wrecs.p : ctx->d_recs.p;
        RT_CUDA(ctx, cudaMemsetAsync(ctx->d_blk_occ.p, 0, blk_bytes, st));
        k_lc_tris<<<ctx->sm_count * 8, 256, 0, st>>>(ctx->d_tris.p, ctx->n_tris, n_words, in.light, in.span, ctx->d_tri_occ.p);
        k_lc_parents<<<ctx->sm_count * 8, 256, 0, st>>>(recs, n_recs, ctx->d_rec_parent.p);
        k_lc_leaves<<<ctx->sm_count * 8, 256, 0, st>>>(recs, n_recs, ctx->d_rec_parent.p, ctx->d_tri_occ.p, ctx->d_blk_occ.p);
    }
    RT_CUDA(ctx, cudaGetLastError());
    ctx->mask_in = in;
    ctx->mask_valid = true;
    return RT_OK;
}

int validate_settings(RtContext* ctx, const RtSettings* s)
{
    std::string why;
    int r = check_settings(s, why);
    return r ? fail(ctx, r, "%s", why.c_str()) : RT_OK;
}

int validate_scene_for_render(RtContext* ctx, const RtSettings* s)
{
    SceneFacts f;
    f.bvh_valid = ctx->bvh_valid; f.camera_set = ctx->camera_set; f.n_tris = ctx->n_tris; f.n_mats = ctx->n_mats;
    f.min_mat_index = ctx->min_mat_index; f.max_mat_index = ctx->max_mat_index;
    for (int i = 0; i < RT_TEX_COUNT; i++) f.tex_format[i] = ctx->tex[i].format;
    f.n_shapes = (int)ctx->shapes.size();
    for (const HostShape& sh : ctx->shapes) {
        const int m = (int)(sh.bits & 0x7fffffffu);
        f.shape_min_mat = std::min(f.shape_min_mat, m);
        f.shape_max_mat = std::max(f.shape_max_mat, m);
    }
    std::string why;
    int r = check_scene_for_render(f, s, why);
    return r ? fail(ctx, r, "%s", why.c_str()) : RT_OK;
}

FrameView frame_view(const RtContext* ctx, const RtSettings* s)
{
    FrameView fr;
    memset(&fr, 0, sizeof(fr));
    fr.proj_inv = ctx->proj_inv;
    fr.cam_to_world = ctx->cam_to_world;
    fr.cam_pos = ctx->cam_pos;
    fr.light = ctx->light;
    fr.factor = s->enable_ssaa ? s->ssaa_factor : 1;                                // renderer.cpp:116-120
    fr.rw = s->image_width * fr.factor;
    fr.rh = s->image_height * fr.factor;
    fr.s = *s;
    return fr;
}

int check_tile_args(RtContext* ctx, int tile_size, int tile_mod, int tile_rem)
{
    if (tile_size <= 0 || tile_mod <= 0 || tile_rem < 0 || tile_rem >= tile_mod)
        return fail(ctx, RT_ERR_INVALID, "tile_size %d tile_mod %d tile_rem %d", tile_size, tile_mod, tile_rem);
    return RT_OK;
}

int grid_for(const RtContext* ctx, const void* kernel, int threads)
{
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0);
    if (per_sm < 1) per_sm = 1;
    return ctx->sm_count * per_sm;                 // persistent grid: a whole number of CTAs per SM
}

// Inverse of a 4x4 row-major matrix (Gauss-Jordan with partial pivoting); false when it is singular.
bool invert4(const double a[16], double out[16])
{
    double m[4][8];
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) { m[i][j] = a[4 * i + j]; m[i][4 + j] = i == j ? 1.0 : 0.0; }
    for (int c = 0; c < 4; c++) {
        int piv = c;
        for (int r = c + 1; r < 4; r++) if (std::fabs(m[r][c]) > std::fabs(m[piv][c])) piv = r;
        if (std::fabs(m[piv][c]) < 1e-300) return false;
        if (piv != c) for (int j = 0; j < 8; j++) std::swap(m[piv][j], m[c][j]);
        const double d = 1.0 / m[c][c];
        for (int j = 0; j < 8; j++) m[c][j] *= d;
        for (int r = 0; r < 4; r++) {
            if (r == c) continue;
            const double f = m[r][c];
            if (f != 0.0) for (int j = 0; j < 8; j++) m[r][j] -= f * m[c][j];
        }
    }
    for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out[4 * i + j] = m[i][4 + j];
    return true;
}

// Screen coverage of a box set for the supersampled frame rw x rh.  Bit bx % 32 of word by * words_per_row + bx / 32 of `bits`
// belongs to the 8x4 block (bx, by) -- the footprint of one primary packet -- and is set when a ray that primary_ray generates
// for a sample of the block can make tri_test accept a triangle inside one of the boxes (6 floats each: lo xyz, hi xyz).
// Returns false when no bound can be given and every block must be traced: a matrix is singular, the ray origin is not the
// projection centre, a line of sight does not project back to its own pixel (rt_set_camera accepts any matrices), or the
// rounding bounds do not hold.  A box that is not safely in front of the camera covers the whole frame.  DESIGN.md §4
// derives the margin; `margin_scale` multiplies it (1 = the derived margin).  Everything here is double precision.
bool screen_coverage(const M4& cam_to_world, const M4& proj_inv, V3 cam_pos, int rw, int rh, const float* boxes, size_t n_boxes,
                     double margin_scale, std::vector<uint32_t>& bits, int32_t& words_per_row)
{
    const int bw = (rw + 7) / 8, bh = (rh + 3) / 4;
    words_per_row = (bw + 31) / 32;
    bits.assign((size_t)words_per_row * (size_t)bh, 0u);
    auto set_blocks = [&](int bx0, int by0, int bx1, int by1) {
        for (int by = by0; by <= by1; by++) {
            uint32_t* row = bits.data() + (size_t)by * words_per_row;
            for (int w = bx0 >> 5; w <= bx1 >> 5; w++) {
                const int lo = std::max(bx0 - 32 * w, 0), hi = std::min(bx1 - 32 * w, 31);
                row[w] |= (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
            }
        }
    };
    if (n_boxes == 0) return true;                                              // nothing to hit
    double c2w[16], pinv[16], w2c[16], proj[16];
    for (int i = 0; i < 16; i++) { c2w[i] = (&cam_to_world.m[0][0])[i]; pinv[i] = (&proj_inv.m[0][0])[i]; }
    if (!invert4(c2w, w2c) || !invert4(pinv, proj)) return false;
    // the ray origin must be the projection centre: camera_to_world * (0,0,0)
    const double w0 = c2w[15];
    if (!(std::fabs(w0) > 1e-12)) return false;
    const double centre[3] = {c2w[3] / w0, c2w[7] / w0, c2w[11] / w0};
    const double pos[3] = {cam_pos.x, cam_pos.y, cam_pos.z};
    double scale = 1.0, dc = 0.0;
    for (int k = 0; k < 3; k++) scale = std::max(scale, std::fabs(centre[k]));
    for (int k = 0; k < 3; k++) {
        if (!(std::fabs(centre[k] - pos[k]) <= 1e-5 * scale)) return false;
        dc += (centre[k] - pos[k]) * (centre[k] - pos[k]);
    }
    dc = std::sqrt(dc);
    // The bound only means something if the rays primary_ray shoots are the projection's own lines of sight: the ray of
    // NDC (x, y) runs from the view-space origin through proj_inv * (x, y, -1), so every point of it must project back to
    // (x, y) with positive clip w.  That holds for the reference's Perspective; rt_set_camera accepts any matrix
    // (orthographic, off-centre, ...), so it is checked on the frame's corners and centre, at two depths each.
    for (int k = 0; k < 5; k++) {
        const double nx = k == 4 ? 0.0 : (k & 1 ? 1.0 : -1.0), ny = k == 4 ? 0.0 : (k & 2 ? 1.0 : -1.0);
        double v[4];
        for (int i = 0; i < 4; i++) v[i] = pinv[4 * i] * nx + pinv[4 * i + 1] * ny - pinv[4 * i + 2] + pinv[4 * i + 3];
        if (!(std::fabs(v[3]) > 1e-12)) return false;
        for (int i = 0; i < 3; i++) v[i] /= v[3];
        for (const double along : {1.0, 7.5}) {
            const double q[4] = {v[0] * along, v[1] * along, v[2] * along, 1.0};
            double c[4];
            for (int i = 0; i < 4; i++) c[i] = proj[4 * i] * q[0] + proj[4 * i + 1] * q[1] + proj[4 * i + 2] * q[2] + proj[4 * i + 3] * q[3];
            if (!(c[3] > 0.0) || !(std::fabs(c[0] / c[3] - nx) < 1e-4) || !(std::fabs(c[1] / c[3] - ny) < 1e-4)) return false;
        }
    }
    // Rounding of primary_ray's direction (DESIGN.md §4): bounds on the float error of vs = proj_inv (x, y, -1), of
    // ws = cam_to_world vs and of ws - cam_pos over the whole frame, from the magnitudes of the matrices' terms.  vs and
    // ws are linear-fractional in (x, y), so their extremes over the frame are at its corners; both denominators must
    // keep one sign there.
    const double eps = 0x1p-24;
    double VS[3] = {0, 0, 0}, WS[3] = {0, 0, 0}, ws_c[4][3], wmin = 1e300, w2min = 1e300, wsign = 0.0, w2sign = 0.0;
    for (int k = 0; k < 4; k++) {
        const double h[4] = {k & 1 ? 1.0 : -1.0, k & 2 ? 1.0 : -1.0, -1.0, 1.0};
        double vh[4], wh[4];
        for (int i = 0; i < 4; i++) vh[i] = pinv[4 * i] * h[0] + pinv[4 * i + 1] * h[1] + pinv[4 * i + 2] * h[2] + pinv[4 * i + 3] * h[3];
        if (k == 0) wsign = vh[3] < 0.0 ? -1.0 : 1.0;
        if (!(vh[3] * wsign > 0.0)) return false;
        wmin = std::min(wmin, std::fabs(vh[3]));
        const double vs[4] = {vh[0] / vh[3], vh[1] / vh[3], vh[2] / vh[3], 1.0};
        for (int i = 0; i < 4; i++) wh[i] = c2w[4 * i] * vs[0] + c2w[4 * i + 1] * vs[1] + c2w[4 * i + 2] * vs[2] + c2w[4 * i + 3];
        if (k == 0) w2sign = wh[3] < 0.0 ? -1.0 : 1.0;
        if (!(wh[3] * w2sign > 0.0)) return false;
        w2min = std::min(w2min, std::fabs(wh[3]));
        for (int i = 0; i < 3; i++) {
            ws_c[k][i] = wh[i] / wh[3];
            VS[i] = std::max(VS[i], std::fabs(vs[i]));
            WS[i] = std::max(WS[i], std::fabs(ws_c[k][i]));
        }
    }
    double e1[4], ev[3], e2[4], e3n = 0.0;
    for (int i = 0; i < 4; i++)                          // 4 products and sums, and the rounding of x and y (2 eps each)
        e1[i] = 6.0 * eps * (std::fabs(pinv[4 * i]) + std::fabs(pinv[4 * i + 1]) + std::fabs(pinv[4 * i + 2]) + std::fabs(pinv[4 * i + 3]));
    if (!(wmin > 2.0 * e1[3])) return false;
    for (int i = 0; i < 3; i++) ev[i] = (e1[i] + VS[i] * e1[3]) / (wmin - e1[3]) + 2.0 * eps * VS[i];   // 1 / w, then * (1 / w)
    for (int i = 0; i < 4; i++) {
        double s2 = std::fabs(c2w[4 * i + 3]), p2 = 0.0;
        for (int j = 0; j < 3; j++) { s2 += std::fabs(c2w[4 * i + j]) * VS[j]; p2 += std::fabs(c2w[4 * i + j]) * ev[j]; }
        e2[i] = 4.0 * eps * s2 + p2;
    }
    if (!(w2min > 2.0 * e2[3])) return false;
    for (int i = 0; i < 3; i++) {
        const double ew = (e2[i] + WS[i] * e2[3]) / (w2min - e2[3]) + 2.0 * eps * WS[i];
        const double e3 = ew + eps * (WS[i] + std::fabs(pos[i]));                  // ws - cam_pos
        e3n += e3 * e3;
    }
    e3n = std::sqrt(e3n);
    // every ws lies in the plane of the frame's corners: its distance from the camera bounds |ws - cam_pos| from below
    double u[3], v[3], n[3];
    for (int i = 0; i < 3; i++) { u[i] = ws_c[1][i] - ws_c[0][i]; v[i] = ws_c[2][i] - ws_c[0][i]; }
    n[0] = u[1] * v[2] - u[2] * v[1]; n[1] = u[2] * v[0] - u[0] * v[2]; n[2] = u[0] * v[1] - u[1] * v[0];
    const double nn = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    const double lmin = std::fabs(n[0] * (ws_c[0][0] - pos[0]) + n[1] * (ws_c[0][1] - pos[1]) + n[2] * (ws_c[0][2] - pos[2])) / nn;
    if (!(lmin > 4.0 * e3n)) return false;
    const double e_dir = 2.0 * e3n / lmin + 5.0 * eps;     // |d - D| for the unit exact direction D; normalize adds 5 eps
    const double kTriRel = 0x1p-14;                          // tri_test's acceptance outside its triangle, relative
    const double pos_max = std::max(std::fabs(pos[0]), std::max(std::fabs(pos[1]), std::fabs(pos[2])));
    const double ndc_slack = 1e-9;                           // the double-precision projection below
    for (size_t b = 0; b < n_boxes; b++) {
        const float* bx = boxes + 6 * b;
        bool finite = true, empty = false;
        double lo[3], hi[3], bmax = 0.0;
        for (int k = 0; k < 3; k++) {
            lo[k] = bx[k]; hi[k] = bx[3 + k];
            finite &= std::isfinite(lo[k]) && std::isfinite(hi[k]);
            empty |= lo[k] > hi[k];
            bmax = std::max(bmax, std::max(std::fabs(lo[k]), std::fabs(hi[k])));
        }
        if (empty) continue;                                  // holds nothing: k_wb_boxes' (+inf, -inf) for the nodes it leaves out
        if (!finite) { set_blocks(0, 0, bw - 1, bh - 1); return true; }
        double sfar = 0.0;
        for (int c = 0; c < 8; c++) {
            double d2 = 0.0;
            for (int k = 0; k < 3; k++) { const double x = ((c >> k) & 1 ? hi[k] : lo[k]) - pos[k]; d2 += x * x; }
            sfar = std::max(sfar, std::sqrt(d2));
        }
        const double e_tri = kTriRel * (pos_max + bmax + sfar);
        const double reach = (sfar + e_tri) * (1.0 + 5.0 * eps);                // the farthest accepted point, along the ray
        const double r = margin_scale * (e_tri + reach * e_dir + dc * (2.0 + reach / lmin));
        double xmin = 1e300, xmax = -1e300, ymin = 1e300, ymax = -1e300;
        bool whole = false;
        for (int c = 0; c < 8 && !whole; c++) {
            const double p[4] = {(c & 1 ? hi[0] + r : lo[0] - r), (c & 2 ? hi[1] + r : lo[1] - r), (c & 4 ? hi[2] + r : lo[2] - r), 1.0};
            double vv[4], cc[4];
            for (int i = 0; i < 4; i++) vv[i] = w2c[4 * i] * p[0] + w2c[4 * i + 1] * p[1] + w2c[4 * i + 2] * p[2] + w2c[4 * i + 3] * p[3];
            if (!(std::fabs(vv[3]) > 1e-12)) { whole = true; break; }
            for (int i = 0; i < 3; i++) vv[i] /= vv[3];
            vv[3] = 1.0;
            for (int i = 0; i < 4; i++) cc[i] = proj[4 * i] * vv[0] + proj[4 * i + 1] * vv[1] + proj[4 * i + 2] * vv[2] + proj[4 * i + 3] * vv[3];
            // in front of the camera with margin: clip w is the view depth of a perspective projection
            if (!(cc[3] > 1e-3 * (1.0 + std::fabs(vv[2])))) { whole = true; break; }
            const double nx = cc[0] / cc[3], ny = cc[1] / cc[3];
            if (!std::isfinite(nx) || !std::isfinite(ny)) { whole = true; break; }
            xmin = std::min(xmin, nx); xmax = std::max(xmax, nx); ymin = std::min(ymin, ny); ymax = std::max(ymax, ny);
        }
        if (whole) { set_blocks(0, 0, bw - 1, bh - 1); return true; }
        // samples whose pixel centre (p + 0.5) / n * 2 - 1 lies in [min, max]
        const double lim = 1e9;
        const double px0 = std::ceil(std::max(-lim, (xmin - ndc_slack + 1.0) * 0.5 * rw - 0.5)), px1 = std::floor(std::min(lim, (xmax + ndc_slack + 1.0) * 0.5 * rw - 0.5));
        const double py0 = std::ceil(std::max(-lim, (ymin - ndc_slack + 1.0) * 0.5 * rh - 0.5)), py1 = std::floor(std::min(lim, (ymax + ndc_slack + 1.0) * 0.5 * rh - 0.5));
        const int x0 = (int)std::max(0.0, px0), x1 = (int)std::min((double)rw - 1, px1);
        const int y0 = (int)std::max(0.0, py0), y1 = (int)std::min((double)rh - 1, py1);
        if (x0 > x1 || y0 > y1) continue;
        set_blocks(x0 >> 3, y0 >> 2, x1 >> 3, y1 >> 2);
    }
    return true;
}

// Any block of supersampled pixels [x0, x1] x [y0, y1] covered
bool cover_any(const std::vector<uint32_t>& bits, int32_t words_per_row, int x0, int y0, int x1, int y1)
{
    const int bx0 = x0 >> 3, bx1 = x1 >> 3;
    for (int by = y0 >> 2; by <= y1 >> 2; by++) {
        const uint32_t* row = bits.data() + (size_t)by * words_per_row;
        for (int w = bx0 >> 5; w <= bx1 >> 5; w++) {
            const int lo = std::max(bx0 - 32 * w, 0), hi = std::min(bx1 - 32 * w, 31);
            if (row[w] & (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u)) return true;
        }
    }
    return false;
}

// Brings the screen coverage up to date for the frame: rebuilt when the camera, the projection, the frame size or the tree
// changed, and uploaded on the context's stream before the frame's launches or graph (never inside a capture).  The frame
// before may still read the old bitmap, so the upload waits for it; a camera that does not move costs nothing.
int update_cover(RtContext* ctx, const FrameView& fr)
{
    RtContext::CoverInputs in;
    memset(&in, 0, sizeof(in));                                               // compared bytewise
    in.proj_inv = ctx->proj_inv; in.cam_to_world = ctx->cam_to_world; in.cam_pos = ctx->cam_pos;
    in.rw = fr.rw; in.rh = fr.rh; in.tree = ctx->tree_serial;
    if (ctx->cover_valid && memcmp(&in, &ctx->cover_in, sizeof(in)) == 0) return RT_OK;
    ctx->cover_valid = false;
    const double t0 = now_ms();
    ctx->cover_bound = screen_coverage(ctx->cam_to_world, ctx->proj_inv, ctx->cam_pos, fr.rw, fr.rh, ctx->cover_boxes.data(),
                                       ctx->cover_boxes.size() / 6, 1.0, ctx->h_cover, ctx->cover_words);
    const double t1 = now_ms();
    double t2 = t1;
    if (ctx->cover_bound) {
        RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        t2 = now_ms();
        RT_CUDA(ctx, ctx->d_cover.ensure(ctx->h_cover.size()));
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_cover.p, ctx->h_cover.data(), ctx->h_cover.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    static const bool trace = getenv("RTB200_TRACE") != nullptr;
    if (trace) {
        size_t set = 0;
        for (uint32_t w : ctx->h_cover) set += (size_t)__builtin_popcount(w);
        const size_t blocks = (size_t)((fr.rw + 7) / 8) * (size_t)((fr.rh + 3) / 4);
        fprintf(stderr, "[rtb200] screen coverage: %zu boxes, bound %d, %.4f of the blocks covered, build %.3f ms, upload %.3f ms\n",
                ctx->cover_boxes.size() / 6, (int)ctx->cover_bound, ctx->cover_bound ? (double)set / (double)blocks : 1.0, t1 - t0, now_ms() - t2);
    }
    ctx->cover_in = in;
    ctx->cover_valid = true;
    ctx->cover_generation++;
    return RT_OK;
}

// The shard's tile list on the device (cached).  tile_rem = -1: the lists of ALL tile_mod shards, each padded with
// 0xffffffff to the longest one (the layout of the gathered staging buffer).
int get_tile_list(RtContext* ctx, const RtSettings* s, int tile_size, int tile_mod, int tile_rem, TileList** out)
{
    const TileKey key(s->image_width, s->image_height, tile_size, tile_mod, tile_rem);
    auto it = ctx->tile_lists.find(key);
    if (it == ctx->tile_lists.end()) {
        if (ctx->tile_lists.size() > 64) {                         // a caller cycling through frame sizes: start over
            RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            for (auto& kv : ctx->tile_lists) { cudaFree(kv.second.d); cudaFree(kv.second.d_split); }
            ctx->tile_lists.clear();
        }
        TileList tl;
        if (tile_rem >= 0) tl.host = owned_tiles(s, tile_size, tile_mod, tile_rem, &tl.tiles_x);
        else {
            std::vector<std::vector<uint32_t>> per(tile_mod);
            size_t longest = 0;
            for (int r = 0; r < tile_mod; r++) { per[r] = owned_tiles(s, tile_size, tile_mod, r, &tl.tiles_x); longest = std::max(longest, per[r].size()); }
            tl.host.assign(longest * tile_mod, 0xffffffffu);
            for (int r = 0; r < tile_mod; r++) std::copy(per[r].begin(), per[r].end(), tl.host.begin() + (size_t)r * longest);
        }
        tl.count = (uint32_t)tl.host.size();
        if (tl.count) {
            RT_CUDA(ctx, cudaMalloc((void**)&tl.d, tl.host.size() * sizeof(uint32_t)));
            RT_CUDA(ctx, cudaMemcpy(tl.d, tl.host.data(), tl.host.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        it = ctx->tile_lists.emplace(key, std::move(tl)).first;
    }
    *out = &it->second;
    return RT_OK;
}

// The frame of reference of the light-space queue order (kernels.cuh, LightMap): ez from the light to the centre of the
// root cell's box; a gnomonic map of the cone around the box's bounding sphere when the light is outside it.
LightMap make_light_map(const RtContext* ctx)
{
    LightMap lm;
    const V3 c = v3(0.5f * (ctx->root_lo[0] + ctx->root_hi[0]), 0.5f * (ctx->root_lo[1] + ctx->root_hi[1]), 0.5f * (ctx->root_lo[2] + ctx->root_hi[2]));
    const V3 h = v3(0.5f * (ctx->root_hi[0] - ctx->root_lo[0]), 0.5f * (ctx->root_hi[1] - ctx->root_lo[1]), 0.5f * (ctx->root_hi[2] - ctx->root_lo[2]));
    const float radius = std::sqrt(h.x * h.x + h.y * h.y + h.z * h.z);
    V3 z = c - ctx->light;
    const float dist = std::sqrt(z.x * z.x + z.y * z.y + z.z * z.z);
    if (!(dist > 1.0e-20f) || !std::isfinite(dist)) { z = v3(0, 0, 1); }
    else z = v3(z.x / dist, z.y / dist, z.z / dist);
    const V3 up = std::fabs(z.y) < 0.9f ? v3(0, 1, 0) : v3(1, 0, 0);
    V3 x = v3(up.y * z.z - up.z * z.y, up.z * z.x - up.x * z.z, up.x * z.y - up.y * z.x);
    const float xl = std::sqrt(x.x * x.x + x.y * x.y + x.z * x.z);
    x = v3(x.x / xl, x.y / xl, x.z / xl);
    lm.ex = x;
    lm.ey = v3(z.y * x.z - z.z * x.y, z.z * x.x - z.x * x.z, z.x * x.y - z.y * x.x);
    lm.ez = z;
    lm.scale = 0.0f;
    if (std::isfinite(dist) && std::isfinite(radius) && dist > radius * 1.05f && radius > 0.0f) {
        const float tan_half = radius / std::sqrt(dist * dist - radius * radius);
        lm.scale = 1.0f / tan_half;
    }
    return lm;
}


void transform_host_vertices(RtContext* ctx, const M4& t)
{
    const long long n = (long long)(ctx->xyz9.size() / 3);
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < n; i++) {                                            // Transform::operator()(Triangle), mat.cpp:133-140
        V3 p = xform_point(t, v3(ctx->xyz9[3 * i], ctx->xyz9[3 * i + 1], ctx->xyz9[3 * i + 2]));
        ctx->xyz9[3 * i] = p.x; ctx->xyz9[3 * i + 1] = p.y; ctx->xyz9[3 * i + 2] = p.z;
    }
}

void apply_pending_host_transforms(RtContext* ctx)
{
    for (const M4& t : ctx->db.host_pending) transform_host_vertices(ctx, t);
    ctx->db.host_pending.clear();
}

// keeps the first `keep` elements
template <typename T>
cudaError_t grow_keep(DevBuf<T>& b, size_t count, size_t keep, cudaStream_t st)
{
    if (count <= b.n) return cudaSuccess;
    T* fresh = nullptr;
    cudaError_t e = cudaMalloc((void**)&fresh, count * sizeof(T));
    if (e != cudaSuccess) return e;
    if (b.p && keep) e = cudaMemcpyAsync(fresh, b.p, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (b.p) cudaFree(b.p);
    b.p = fresh;
    b.n = count;
    return e;
}

// exclusive scan of `count` counters in place (octree_device.cuh); their sum goes to *total unless it is null
int scan_counts(RtContext* ctx, uint32_t* data, size_t count, uint32_t* total)
{
    using namespace devbuild;
    DeviceBuild& D = ctx->db;
    const cudaStream_t st = ctx->stream;
    const uint32_t blocks = (uint32_t)((count + kScanBlock - 1) / kScanBlock);
    RT_CUDA(ctx, D.sums.ensure(std::max<uint32_t>(blocks, 1)));
    k_scan_sums<<<blocks, 1024, 0, st>>>(data, count, D.sums.p);
    k_scan_top<<<1, 1024, 0, st>>>(D.sums.p, blocks, total);
    k_scan_apply<<<blocks, 1024, 0, st>>>(data, count, D.sums.p);
    return RT_OK;
}

// The box set of the screen coverage when the packets traverse recs[] itself: the root cell's box
void root_cover_box(RtContext* ctx)
{
    ctx->cover_boxes.assign({ctx->root_lo[0], ctx->root_lo[1], ctx->root_lo[2], ctx->root_hi[0], ctx->root_hi[1], ctx->root_hi[2]});
}

// wrecs[], the wide copy of recs[] that the packet kernels traverse (octree_device.cuh: k_wb_*), and the top table over
// it.  Runs after either builder has put its n_records records in d_recs; the node arrays of the device build are reused
// (a wide node is one record of recs[], so n_records bounds their number).
int build_wide_tree(RtContext* ctx, uint64_t n_records)
{
    using namespace devbuild;
    DeviceBuild& D = ctx->db;
    const cudaStream_t st = ctx->stream;
    const size_t cap = (size_t)n_records;
    RT_CUDA(ctx, D.w_src.ensure(cap)); RT_CUDA(ctx, D.w_need.ensure(cap)); RT_CUDA(ctx, D.c_first.ensure(cap)); RT_CUDA(ctx, D.c_info.ensure(cap));
    RT_CUDA(ctx, D.c_size.ensure(cap)); RT_CUDA(ctx, D.c_rec.ensure(cap)); RT_CUDA(ctx, D.c_block.ensure(cap)); RT_CUDA(ctx, D.stats.ensure(1));
    Cells C;
    memset(&C, 0, sizeof(C));
    C.first_child = D.c_first.p; C.info = D.c_info.p; C.size = D.c_size.p; C.rec = D.c_rec.p; C.block = D.c_block.p;
    {
        const uint32_t zero = 0u, root_block = 2u;                              // the root node is record 0, its block starts at 2
        RT_CUDA(ctx, cudaMemcpyAsync(D.w_src.p, &zero, 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(C.rec, &zero, 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(C.block, &root_block, 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));                                // the sources are on this stack frame
    }
    const float4* recs = ctx->d_recs.p;
    uint32_t* d_total = (uint32_t*)&D.stats.p->top_n;                           // borrowed until the top table is built
    std::vector<uint32_t> level_first, level_count;
    uint32_t root_size = 0, limit = kWideBlock;
    // the collapse with limit kWideBlock; narrower (limit halved) only when its packet stack bound would exceed RT_STACK_SIZE
    for (;; limit /= 2u) {
        level_first.assign(1, 0u); level_count.assign(1, 1u);
        for (;;) {
            const uint32_t lf = level_first.back(), lc = level_count.back();
            RT_CUDA(ctx, D.counts.ensure(lc));
            RT_CUDA(ctx, D.w_members.ensure(kWideBlock * (size_t)lc));
            k_wb_collapse<<<(lc + 255) / 256, 256, 0, st>>>(recs, D.w_src.p, lf, lc, limit, C.info, D.counts.p, D.w_members.p);
            if (int r = scan_counts(ctx, D.counts.p, lc, d_total)) return r;
            uint32_t total = 0;
            RT_CUDA(ctx, cudaMemcpyAsync(&total, d_total, 4, cudaMemcpyDeviceToHost, st));
            RT_CUDA(ctx, cudaStreamSynchronize(st));
            if (total == 0) break;
            if ((size_t)lf + lc + total > cap) return fail(ctx, RT_ERR_STATE, "wide tree: more nodes than child records");
            k_wb_children<<<(lc + 255) / 256, 256, 0, st>>>(C, D.w_src.p, lf, lc, D.counts.p, D.w_members.p, lf + lc);
            level_first.push_back(lf + lc); level_count.push_back(total);
        }
        for (int l = (int)level_first.size() - 1; l >= 0; l--)
            k_wb_size<<<(level_count[l] + 255) / 256, 256, 0, st>>>(C, D.w_need.p, level_first[l], level_count[l]);
        uint32_t need = 0;
        RT_CUDA(ctx, cudaMemcpyAsync(&root_size, C.size, 4, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaMemcpyAsync(&need, D.w_need.p, 4, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        ctx->wide_stack = need + 1u;
        if (ctx->wide_stack <= RT_STACK_SIZE) break;
        if (limit <= 1u) return fail(ctx, RT_ERR_INVALID, "tree too deep for the packet stack (%u > %d entries)", ctx->wide_stack, RT_STACK_SIZE);
    }
    const uint32_t n_nodes = level_first.back() + level_count.back();
    {
        // the box set of the screen coverage: the nodes of the deepest level with at most kCoverBoxes of them, and the leaves
        // above it (k_wb_boxes); one copy to the host per build
        size_t lv = 0;
        while (lv + 1 < level_first.size() && level_count[lv + 1] <= kCoverBoxes) lv++;
        const uint32_t n_box = level_first[lv] + level_count[lv];
        RT_CUDA(ctx, D.w_boxes.ensure(6 * (size_t)n_box));
        k_wb_boxes<<<(n_box + 255) / 256, 256, 0, st>>>(recs, D.w_src.p, C.info, n_box, level_first[lv], D.w_boxes.p);
        ctx->cover_boxes.resize(6 * (size_t)n_box);
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->cover_boxes.data(), D.w_boxes.p, 6 * (size_t)n_box * sizeof(float), cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
    }
    const uint64_t n_wide = 2ull + root_size;
    ctx->n_wrecs = n_wide;
    RT_CUDA(ctx, ctx->d_wrecs.ensure(4 * n_wide));
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_wrecs.p, 0, 4 * n_wide * sizeof(float4), st));
    Params P;
    memset(&P, 0, sizeof(P));                                                   // leaf_split 0: k_ob_place skips no level
    for (size_t l = 0; l < level_first.size(); l++)
        k_ob_place<<<(level_count[l] + 255) / 256, 256, 0, st>>>(C, level_first[l], level_count[l], P);
    k_wb_records<<<(n_nodes + 255) / 256, 256, 0, st>>>(recs, D.w_src.p, C, n_nodes, (float4*)ctx->d_wrecs.p);
    k_ob_top_table<<<1, 32, 0, st>>>((float4*)ctx->d_wrecs.p, (float4*)ctx->d_top.p, D.stats.p);
    uint32_t top_n = 0;
    RT_CUDA(ctx, cudaMemcpyAsync(&top_n, &D.stats.p->top_n, 4, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    RT_CUDA(ctx, cudaGetLastError());
    ctx->top_n = (int)top_n;
    ctx->wide_tree = true;
    if (getenv("RTB200_TRACE"))
        fprintf(stderr, "[rtb200] wide tree: %llu records on %zu levels (narrow: %llu), blocks of <= %u, packet stack <= %u of %d\n",
                (unsigned long long)n_wide, level_first.size(), (unsigned long long)n_records, limit, ctx->wide_stack, RT_STACK_SIZE);
    return RT_OK;
}

// rt_build_bvh on the device (octree_device.cuh).  n > 0.
int build_bvh_device(RtContext* ctx, int max_depth, int leaf_max)
{
    using namespace devbuild;
    DeviceBuild& D = ctx->db;
    const size_t n = ctx->xyz9.size() / 9;
    const cudaStream_t st = ctx->stream;
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    const double t0 = now_ms();
    if (!D.tris_on_device) {
        apply_pending_host_transforms(ctx);
        RT_CUDA(ctx, D.xyz9.ensure(9 * n));
        RT_CUDA(ctx, cudaMemcpyAsync(D.xyz9.p, ctx->xyz9.data(), 9 * n * sizeof(float), cudaMemcpyHostToDevice, st));
        if (ctx->has_uv) { RT_CUDA(ctx, D.uv6.ensure(6 * n)); RT_CUDA(ctx, cudaMemcpyAsync(D.uv6.p, ctx->uv6.data(), 6 * n * sizeof(float), cudaMemcpyHostToDevice, st)); }
        if (ctx->has_mat) { RT_CUDA(ctx, D.mat.ensure(n)); RT_CUDA(ctx, cudaMemcpyAsync(D.mat.p, ctx->mat.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st)); }
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        D.tris_on_device = true;
    }
    const double t1 = now_ms();

    Params P;
    P.max_depth = max_depth; P.leaf_max = leaf_max; P.leaf_split = ctx->opt_leaf_split;
    P.total_depth = std::min(kMaxKeyLevels, max_depth + (ctx->opt_leaf_split > 0 ? kExtraLevels : 0));
    P.s3 = std::sqrt(3.0f) / 3;
    const uint32_t n32 = (uint32_t)n;
    const int wide = ctx->sm_count * 8;
    static const bool trace = getenv("RTB200_TRACE") != nullptr;
    double t_phase = t1;
    auto trace_phase = [&](const char* what) {
        if (!trace) return;
        cudaStreamSynchronize(st);
        const double t = now_ms();
        fprintf(stderr, "[rtb200]   device octree: %s %.2f ms\n", what, t - t_phase);
        t_phase = t;
    };
    RT_CUDA(ctx, D.stats.ensure(1)); RT_CUDA(ctx, D.centroid.ensure(3 * n));
    for (int k = 0; k < 2; k++) { RT_CUDA(ctx, D.keys[k].ensure(n)); RT_CUDA(ctx, D.idx[k].ensure(n)); }
    k_ob_init<<<1, 1, 0, st>>>(D.stats.p);
    k_ob_centroids<<<wide, 256, 0, st>>>(D.xyz9.p, n32, D.centroid.p, D.stats.p);
    k_ob_keys<<<wide, 256, 0, st>>>(D.centroid.p, n32, D.stats.p, P, D.keys[0].p, D.idx[0].p);

    // ---- stable radix sort of (key, index), 8 bits per pass over the 3 * total_depth bits in use
    const uint32_t n_units = (n32 + kSortUnit - 1) / kSortUnit;
    const size_t n_hist = (size_t)256 * n_units;
    const uint32_t hist_blocks = (uint32_t)((n_hist + kScanBlock - 1) / kScanBlock);
    RT_CUDA(ctx, D.hist.ensure(n_hist));
    int cur = 0;
    const int passes = (3 * P.total_depth + 7) / 8;
    (void)hist_blocks;
    for (int pass = 0; pass < passes; pass++) {
        k_rs_count<<<(n_units + 3) / 4, 128, 0, st>>>(D.keys[cur].p, n32, 8 * pass, n_units, D.hist.p);
        if (int r = scan_counts(ctx, D.hist.p, n_hist, nullptr)) return r;
        k_rs_scatter<<<(n_units + 3) / 4, 128, 0, st>>>(D.keys[cur].p, D.idx[cur].p, n32, 8 * pass, n_units, D.hist.p, D.keys[cur ^ 1].p, D.idx[cur ^ 1].p);
        cur ^= 1;
    }
    const unsigned long long* keys = D.keys[cur].p;
    const uint32_t* idx = D.idx[cur].p;                                         // (k_ob_refine reorders ranges of it in place)
    trace_phase("keys + sort");

    // ---- cells, level by level
    size_t cap = 0;
    auto cells_view = [&]() {
        Cells C;
        C.begin = D.c_begin.p; C.end = D.c_end.p; C.first_child = D.c_first.p; C.info = D.c_info.p; C.nr = D.c_nr.p; C.fr = D.c_fr.p;
        C.size = D.c_size.p; C.rec = D.c_rec.p; C.block = D.c_block.p;
        return C;
    };
    auto reserve_cells = [&](size_t want, size_t keep) -> int {
        if (want <= cap) return RT_OK;
        const size_t c = std::max(want, cap * 2);
        RT_CUDA(ctx, grow_keep(D.c_begin, c, keep, st)); RT_CUDA(ctx, grow_keep(D.c_end, c, keep, st)); RT_CUDA(ctx, grow_keep(D.c_first, c, keep, st));
        RT_CUDA(ctx, grow_keep(D.c_info, c, keep, st)); RT_CUDA(ctx, grow_keep(D.c_size, c, keep, st)); RT_CUDA(ctx, grow_keep(D.c_rec, c, keep, st));
        RT_CUDA(ctx, grow_keep(D.c_block, c, keep, st)); RT_CUDA(ctx, grow_keep(D.c_nr, 7 * c, 7 * keep, st)); RT_CUDA(ctx, grow_keep(D.c_fr, 7 * c, 7 * keep, st));
        cap = std::min({D.c_begin.n, D.c_end.n, D.c_first.n, D.c_info.n, D.c_size.n, D.c_rec.n, D.c_block.n, D.c_nr.n / 7, D.c_fr.n / 7});
        return RT_OK;
    };
    cap = std::min({D.c_begin.n, D.c_end.n, D.c_first.n, D.c_info.n, D.c_size.n, D.c_rec.n, D.c_block.n, D.c_nr.n / 7, D.c_fr.n / 7});
    if (int r = reserve_cells(n / 2 + 4096, 0)) return r;
    {
        const uint32_t root[4] = {0u, n32, 0u, 1u << 10};                        // begin, end, first child, info: a reference cell
        RT_CUDA(ctx, cudaMemcpyAsync(D.c_begin.p, &root[0], 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(D.c_end.p, &root[1], 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(D.c_info.p, &root[3], 4, cudaMemcpyHostToDevice, st));
        const uint32_t place[2] = {0u, 2u};                                     // the root's record and its children's block
        RT_CUDA(ctx, cudaMemcpyAsync(D.c_rec.p, &place[0], 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaMemcpyAsync(D.c_block.p, &place[1], 4, cudaMemcpyHostToDevice, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));                                // the sources are on this stack frame
    }
    std::vector<uint32_t> level_first, level_count;
    level_first.push_back(0); level_count.push_back(1);
    uint32_t* d_total = (uint32_t*)&D.stats.p->top_n;                           // borrowed until the top table is built
    for (int depth = 0; depth <= P.max_depth + 16; depth++) {
        const uint32_t lf = level_first.back(), lc = level_count.back();
        RT_CUDA(ctx, D.counts.ensure(lc));
        k_ob_split<<<(lc + 255) / 256, 256, 0, st>>>(keys, cells_view(), lf, lc, depth, P, D.counts.p, D.stats.p);
        if (int r = scan_counts(ctx, D.counts.p, lc, d_total)) return r;
        uint32_t total = 0;
        RT_CUDA(ctx, cudaMemcpyAsync(&total, d_total, 4, cudaMemcpyDeviceToHost, st));
        RT_CUDA(ctx, cudaStreamSynchronize(st));
        if (total == 0) break;
        if ((size_t)lf + lc + total >= (size_t)0xffffffffu) return fail(ctx, RT_ERR_INVALID, "too many octree cells");
        if (P.leaf_split > 0)
            k_ob_refine<<<std::min<uint32_t>((lc + 7) / 8, (uint32_t)wide), 256, 0, st>>>(cells_view(), lf, lc, P, D.centroid.p, D.idx[cur].p, D.idx[cur ^ 1].p);
        if (int r = reserve_cells((size_t)lf + lc + total, (size_t)lf + lc)) return r;
        k_ob_children<<<(lc + 255) / 256, 256, 0, st>>>(keys, cells_view(), lf, lc, depth, P, D.counts.p, lf + lc);
        level_first.push_back(lf + lc); level_count.push_back(total);
    }
    const uint32_t n_cells = level_first.back() + level_count.back();
    const Cells C = cells_view();
    trace_phase("cells");
    // ---- leaf-order triangle arrays
    k_ob_leaf_order<<<wide, 256, 0, st>>>(C, n_cells, idx, D.idx[cur ^ 1].p);
    idx = D.idx[cur ^ 1].p;
    RT_CUDA(ctx, ctx->d_tris.ensure(3 * n)); RT_CUDA(ctx, ctx->d_shade.ensure(2 * n)); RT_CUDA(ctx, ctx->d_orig.ensure(n)); RT_CUDA(ctx, ctx->d_leaf_of.ensure(n));
    k_ob_triangles<<<wide, 256, 0, st>>>(D.xyz9.p, ctx->has_uv ? D.uv6.p : nullptr, ctx->has_mat ? D.mat.p : nullptr, idx, n32,
                                         (float4*)ctx->d_tris.p, (float4*)ctx->d_shade.p, ctx->d_orig.p, ctx->d_leaf_of.p);
    for (int l = (int)level_first.size() - 1; l >= 0; l--)
        k_ob_bounds<<<(level_count[l] + 127) / 128, 128, 0, st>>>((const float4*)ctx->d_tris.p, C, level_first[l], level_count[l], P);
    trace_phase("triangles + bounds");
    uint32_t root_size = 0;
    RT_CUDA(ctx, cudaMemcpyAsync(&root_size, D.c_size.p, 4, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t n_records = 2ull + root_size;
    if (n_records >= (1ull << 28)) return fail(ctx, RT_ERR_INVALID, "scene needs %llu child records (limit 2^28)", (unsigned long long)n_records);
    RT_CUDA(ctx, ctx->d_recs.ensure(4 * n_records));
    RT_CUDA(ctx, ctx->d_top.ensure(4 * RT_TOP_RECORDS));
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_recs.p, 0, 4 * n_records * sizeof(float4), st));
    for (size_t l = 0; l < level_first.size(); l++)
        k_ob_place<<<(level_count[l] + 255) / 256, 256, 0, st>>>(C, level_first[l], level_count[l], P);
    k_ob_records<<<(n_cells + 255) / 256, 256, 0, st>>>(C, n_cells, P, (float4*)ctx->d_recs.p);
    const bool packets_wide = P.leaf_split > 0;                                 // the top table goes over the array the packets traverse
    if (!packets_wide) k_ob_top_table<<<1, 32, 0, st>>>((float4*)ctx->d_recs.p, (float4*)ctx->d_top.p, D.stats.p);
    Stats hs;
    F4 root_rec[2];
    RT_CUDA(ctx, cudaMemcpyAsync(&hs, D.stats.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaMemcpyAsync(root_rec, ctx->d_recs.p, sizeof(root_rec), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    RT_CUDA(ctx, cudaGetLastError());
    ctx->top_n = (int)hs.top_n;
    if (packets_wide) if (int r = build_wide_tree(ctx, n_records)) return r;
    const double t2 = now_ms();

    ctx->n_tris = n32;
    ctx->root_lo[0] = root_rec[0].x; ctx->root_lo[1] = root_rec[0].z; ctx->root_lo[2] = root_rec[1].x;
    ctx->root_hi[0] = root_rec[0].y; ctx->root_hi[1] = root_rec[0].w; ctx->root_hi[2] = root_rec[1].y;
    if (!ctx->wide_tree) root_cover_box(ctx);
    RtBvhInfo& bi = ctx->info;
    bi.triangles = n;
    bi.interior = hs.interior;
    bi.nodes = 1 + 8 * hs.interior;                                             // every split allocates all 8 children (bvh.h:159-166)
    bi.leaves = bi.nodes - bi.interior;
    bi.empty_leaves = 8 * hs.interior - hs.nonempty_children;
    bi.max_depth_reached = hs.max_depth; bi.max_leaf_size = hs.max_leaf;
    bi.child_records = n_records;
    bi.device_bytes = (4 * n_records + 3 * n + 2 * n) * sizeof(F4) + n * sizeof(int32_t);
    bi.build_ms = t2 - t1;
    bi.upload_ms = t1 - t0;
    ctx->bvh_valid = true;
    if (getenv("RTB200_TRACE"))
        fprintf(stderr, "[rtb200] device octree: %u cells on %zu levels, %llu records, upload %.1f ms, build %.1f ms\n", n_cells, level_first.size(),
                (unsigned long long)n_records, t1 - t0, t2 - t1);
    return RT_OK;
}

bool tune_packets_hint(const RtContext* ctx) { return ctx->tune.packets != 0; }

int ensure_stack(RtContext* ctx, const RtSettings* s)
{
    // k_reflect recurses (trace_ray_secondary); every level holds two traversal stacks.
    size_t want = 4096 + (size_t)(std::max(0, s->max_recursion_depth) + 2) * 3072;
    if (want > ctx->stack_limit_set) {
        RT_CUDA(ctx, cudaDeviceSetLimit(cudaLimitStackSize, want));
        ctx->stack_limit_set = want;
    }
    return RT_OK;
}

} // namespace

extern "C" {

void rt_default_settings(RtSettings* s)
{
    if (s) default_settings(s);
}

uint32_t rt_pixel_seed(uint32_t pixel_index, uint32_t rng_seed) { return pixel_seed(pixel_index, rng_seed); }

void rt_perspective_inverse(float fov, float aspect, float znear, float zfar, float proj_inv_out[16])
{
    M4 inv = invert_matrix(perspective_matrix(fov, aspect, znear, zfar));
    memcpy(proj_inv_out, inv.m, sizeof(inv.m));
}

void rt_invert_transform(const float m[16], float out[16])
{
    M4 a;
    memcpy(a.m, m, sizeof(a.m));
    M4 inv = invert_matrix(a);
    memcpy(out, inv.m, sizeof(inv.m));
}

void rt_transform_point(const float m[16], const float p[3], float out[3])
{
    M4 a;
    memcpy(a.m, m, sizeof(a.m));
    V3 q = xform_point(a, v3(p[0], p[1], p[2]));
    out[0] = q.x; out[1] = q.y; out[2] = q.z;
}

int rt_create(int device, RtContext** out)
{
    if (!out) return fail(nullptr, RT_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, RT_ERR_CUDA, "no CUDA device: %s (this library has no CPU path)", cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(nullptr, RT_ERR_INVALID, "device %d of %d", device, count);
    RtContext* ctx = new RtContext();
    ctx->device = device;
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ERR_CUDA, "device init: %s", cudaGetErrorString(e));
    }
    ctx->own_stream = ctx->stream;
    ctx->sm_count = prop.multiProcessorCount;
    // identity camera looking down -z, like a default-constructed Camera (scene/camera.h:11,29-30)
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) ctx->cam_to_world.m[i][j] = ctx->proj_inv.m[i][j] = (i == j) ? 1.0f : 0.0f;
    *out = ctx;
    return RT_OK;
}

void rt_destroy(RtContext* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->d_recs.release(); ctx->d_wrecs.release(); ctx->d_top.release(); ctx->d_tris.release(); ctx->d_shade.release(); ctx->d_mats.release(); ctx->d_orig.release(); ctx->d_leaf_of.release(); ctx->d_shapes.release();
    for (auto& t : ctx->tex) if (t.d) cudaFree(t.d);
    ctx->d_super.release(); ctx->d_frame.release(); ctx->db.release(); ctx->d_gz.release(); ctx->d_gn.release(); ctx->d_ao.release();
    for (auto& g : ctx->graphs) cudaGraphExecDestroy(g.exec);
    ctx->d_rkeys.release(); ctx->d_rxy.release(); ctx->d_runits.release(); ctx->d_rcount.release(); ctx->d_rfrag.release();
    for (auto& kv : ctx->tile_lists) { cudaFree(kv.second.d); cudaFree(kv.second.d_split); }
    for (auto& qs : ctx->qs) qs.release();
    for (auto st : ctx->lane_stream) if (st) cudaStreamDestroy(st);
    if (ctx->lane_fork) cudaEventDestroy(ctx->lane_fork);
    for (auto e : ctx->lane_join) if (e) cudaEventDestroy(e);
    ctx->d_counters.release(); ctx->d_flag.release();
    if (ctx->d_work_map) cudaFree(ctx->d_work_map);
    ctx->b_a.release(); ctx->b_b.release(); ctx->b_t.release(); ctx->b_u.release(); ctx->b_v.release(); ctx->b_id.release(); ctx->b_occ.release();
    if (ctx->pending.host_cnt) cudaFreeHost(ctx->pending.host_cnt);
    if (ctx->h_frame) cudaFreeHost(ctx->h_frame);
    for (auto e : ctx->copy_ev) if (e) cudaEventDestroy(e);
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* rt_last_error(const RtContext* ctx) { return ctx ? ctx->error.c_str() : g_create_error.c_str(); }

int rt_set_option(RtContext* ctx, int option, int64_t value)
{
    if (!ctx) return RT_ERR_INVALID;
    switch (option) {
    case RT_OPT_COUNT_WORK: ctx->opt_count_work = value != 0; return RT_OK;
    case RT_OPT_LEAF_SPLIT:
        if (value < 0 || value > 1024) return fail(ctx, RT_ERR_INVALID, "leaf split %lld", (long long)value);
        ctx->opt_leaf_split = (int)value;
        ctx->bvh_valid = false;                          // takes effect at the next rt_build_bvh
        return RT_OK;
    case RT_OPT_REFILL_PRIMARY:
    case RT_OPT_REFILL_SHADE:
        if (value < 1 || value > 32) return fail(ctx, RT_ERR_INVALID, "refill threshold %lld outside [1,32]", (long long)value);
        (option == RT_OPT_REFILL_PRIMARY ? ctx->tune.primary_refill : ctx->tune.shade_refill) = (int32_t)value;
        return RT_OK;
    case RT_OPT_TRI_BATCH:
        if (value < 1 || value > 32) return fail(ctx, RT_ERR_INVALID, "triangle batch %lld outside [1,32]", (long long)value);
        ctx->tune.tri_batch = (int32_t)value;
        return RT_OK;
    case RT_OPT_PACKETS:
        ctx->tune.packets = value != 0;
        return RT_OK;
    case RT_OPT_PACKET_ROUNDS:
        if (value < -(1 << 30) || value > (1 << 30)) return fail(ctx, RT_ERR_INVALID, "packet rounds %lld", (long long)value);
        ctx->tune.packet_rounds = (int32_t)value;
        return RT_OK;
    case RT_OPT_PRIMARY_ROUNDS:
        if (value < -(1 << 30) || value > (1 << 30)) return fail(ctx, RT_ERR_INVALID, "primary rounds %lld", (long long)value);
        ctx->tune.primary_rounds = (int32_t)value;
        return RT_OK;
    case RT_OPT_ITEM_ROUNDS:
        if (value == 0 || value < -(1 << 30) || value > (1 << 30)) return fail(ctx, RT_ERR_INVALID, "item rounds %lld", (long long)value);
        ctx->tune.item_rounds = (int32_t)value;
        return RT_OK;
    case RT_OPT_FUSED_ITEMS: ctx->tune.fused = value != 0; return RT_OK;
    case RT_OPT_TOP_TABLE: ctx->opt_top_table = value != 0; return RT_OK;
    case RT_OPT_ITEM_PASSES:
        if (value < 1 || value > kItemPasses) return fail(ctx, RT_ERR_INVALID, "item passes %lld outside [1,%d]", (long long)value, kItemPasses);
        ctx->tune.item_passes = (int32_t)value;
        return RT_OK;
    case RT_OPT_DEVICE_BUILD: ctx->opt_device_build = value != 0; return RT_OK;
    case RT_OPT_SHADOW_SORT:
        if (value < 0 || value > 2) return fail(ctx, RT_ERR_INVALID, "shadow sort %lld outside [0,2]", (long long)value);
        ctx->opt_shadow_sort = (int)value;
        return RT_OK;
    case RT_OPT_SCREEN_CULL: ctx->opt_screen_cull = value != 0; return RT_OK;
    case RT_OPT_LANES:
        if (value < 0 || value > kMaxLanes) return fail(ctx, RT_ERR_INVALID, "lanes %lld outside [0,%d]", (long long)value, kMaxLanes);
        ctx->opt_lanes = value == 1 ? kLanes : (int)std::max<int64_t>(value, 1);   // 0: one chunk at a time; 1: the default (2); n: n chunks in flight
        return RT_OK;
    case RT_OPT_GRAPH: ctx->opt_graph = value != 0; return RT_OK;
    case RT_OPT_LIGHT_CULL: ctx->opt_light_cull = value != 0; return RT_OK;
    case RT_OPT_FAN_LANES: ctx->opt_fan_lanes = value != 0; return RT_OK;
    case RT_OPT_PACKET_CULL:
        if (value < 0 || value > 3) return fail(ctx, RT_ERR_INVALID, "packet cull %lld outside [0,3]", (long long)value);
        ctx->tune.cull = (int32_t)value;
        return RT_OK;
    case RT_OPT_RASTER_UNITS:
        if (value < 1 || value > (1ll << 28)) return fail(ctx, RT_ERR_INVALID, "raster unit list of %lld entries outside [1, 2^28]", (long long)value);
        ctx->d_runits.release();
        ctx->raster_units0 = (size_t)value;
        return RT_OK;
    case RT_OPT_CHUNK_PIXELS:
        if (value < 256 || value > (1ll << 31)) return fail(ctx, RT_ERR_INVALID, "chunk of %lld pixels outside [256, 2^31] (ray slots are 32-bit)", (long long)value);
        ctx->opt_chunk_pixels = (uint64_t)value;
        return RT_OK;
    default: return fail(ctx, RT_ERR_INVALID, "unknown option %d", option);
    }
}

int rt_set_stream(RtContext* ctx, void* cuda_stream)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return RT_OK;
}

int rt_set_triangles(RtContext* ctx, const float* xyz9, const float* uv6, const int32_t* mat, size_t n)
{
    if (!ctx) return RT_ERR_INVALID;
    if (n && !xyz9) return fail(ctx, RT_ERR_INVALID, "xyz9 is NULL");
    if (n > 0x7fffffffu / 3) return fail(ctx, RT_ERR_INVALID, "too many triangles");
    ctx->xyz9.assign(xyz9, xyz9 + 9 * n);
    ctx->has_uv = uv6 != nullptr;
    ctx->has_mat = mat != nullptr;
    if (uv6) ctx->uv6.assign(uv6, uv6 + 6 * n); else ctx->uv6.clear();
    if (mat) ctx->mat.assign(mat, mat + n); else ctx->mat.clear();
    ctx->min_mat_index = n ? (mat ? *std::min_element(mat, mat + n) : -1) : 0;
    ctx->max_mat_index = n ? (mat ? *std::max_element(mat, mat + n) : -1) : -1;
    ctx->bvh_valid = false;
    ctx->db.tris_on_device = false;
    ctx->db.host_pending.clear();
    return RT_OK;
}

int rt_build_bvh(RtContext* ctx, int max_depth, int leaf_max_obj_count)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (max_depth < 0 || max_depth > RT_MAX_TREE_DEPTH) return fail(ctx, RT_ERR_INVALID, "max_depth %d outside [0,%d]", max_depth, RT_MAX_TREE_DEPTH);
    if (leaf_max_obj_count < 0) return fail(ctx, RT_ERR_INVALID, "leaf_max_obj_count %d", leaf_max_obj_count);
    const size_t n = ctx->xyz9.size() / 9;
    ctx->bvh_valid = false;                              // whatever happens below, the previous tree is gone
    ctx->wide_tree = false;
    ctx->cover_boxes.clear();
    ctx->tree_serial++;
    if (ctx->opt_device_build && n > 0) return build_bvh_device(ctx, max_depth, leaf_max_obj_count);
    apply_pending_host_transforms(ctx);
    double t0 = now_ms();
    FlatScene flat;
    build_flat_scene(ctx->xyz9.data(), ctx->has_uv ? ctx->uv6.data() : nullptr, ctx->has_mat ? ctx->mat.data() : nullptr, n,
                     max_depth, leaf_max_obj_count, ctx->opt_leaf_split, flat);
    double t1 = now_ms();
    if (flat.n_records >= (1ull << 28)) return fail(ctx, RT_ERR_INVALID, "scene needs %llu child records (limit 2^28)", (unsigned long long)flat.n_records);
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    RT_CUDA(ctx, ctx->d_recs.ensure(flat.recs.size()));
    RT_CUDA(ctx, ctx->d_tris.ensure(flat.tris.size()));
    RT_CUDA(ctx, ctx->d_shade.ensure(flat.shade.size()));
    RT_CUDA(ctx, ctx->d_orig.ensure(flat.orig.size()));
    RT_CUDA(ctx, ctx->d_leaf_of.ensure(flat.orig.size()));
    RawVector<int32_t> leaf_of(flat.orig.size());
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < (long long)flat.orig.size(); i++) leaf_of[(size_t)flat.orig[i]] = (int32_t)i;
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_recs.p, flat.recs.data(), flat.recs.size() * sizeof(F4), cudaMemcpyHostToDevice, ctx->stream));
    RT_CUDA(ctx, ctx->d_top.ensure(4 * RT_TOP_RECORDS));
    if (!flat.top.empty()) RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_top.p, flat.top.data(), flat.top.size() * sizeof(F4), cudaMemcpyHostToDevice, ctx->stream));
    ctx->top_n = (int)(flat.top.size() / 4);
    if (n) {
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_tris.p, flat.tris.data(), flat.tris.size() * sizeof(F4), cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_shade.p, flat.shade.data(), flat.shade.size() * sizeof(F4), cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_orig.p, flat.orig.data(), flat.orig.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_leaf_of.p, leaf_of.data(), leaf_of.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double t2 = now_ms();
    if (n && ctx->opt_leaf_split > 0)                   // replaces the top table over recs[] by one over wrecs[]
        if (int r = build_wide_tree(ctx, flat.n_records)) return r;
    const double wide_ms = now_ms() - t2;
    ctx->n_tris = (uint32_t)n;
    {
        const F4 *q0 = &flat.recs[0], *q1 = &flat.recs[1];                       // (near, far) pairs of the three axis slabs
        ctx->root_lo[0] = q0->x; ctx->root_lo[1] = q0->z; ctx->root_lo[2] = q1->x;
        ctx->root_hi[0] = q0->y; ctx->root_hi[1] = q0->w; ctx->root_hi[2] = q1->y;
    }
    if (!ctx->wide_tree && n) root_cover_box(ctx);
    RtBvhInfo& bi = ctx->info;
    bi.triangles = n;
    bi.nodes = flat.nodes; bi.leaves = flat.leaves; bi.empty_leaves = flat.empty_leaves; bi.interior = flat.interior;
    bi.max_depth_reached = flat.max_depth_reached; bi.max_leaf_size = flat.max_leaf_size;
    bi.child_records = flat.n_records;
    bi.device_bytes = (flat.recs.size() + flat.tris.size() + flat.shade.size()) * sizeof(F4) + flat.orig.size() * sizeof(int32_t);
    bi.build_ms = t1 - t0 + wide_ms;
    bi.upload_ms = t2 - t1;
    ctx->bvh_valid = true;
    return RT_OK;
}

int rt_bvh_info(const RtContext* ctx, RtBvhInfo* out)
{
    if (!ctx || !out) return RT_ERR_INVALID;
    if (!ctx->bvh_valid) return RT_ERR_STATE;
    *out = ctx->info;
    return RT_OK;
}

int rt_transform_triangles(RtContext* ctx, const float m[16], int max_depth, int leaf_max_obj_count)
{
    if (!ctx || !m) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    M4 t;
    memcpy(t.m, m, sizeof(t.m));
    ctx->bvh_valid = false;
    if (ctx->opt_device_build && ctx->db.tris_on_device && !ctx->xyz9.empty()) {
        // the vertices are transformed where the builder reads them; the host copy catches up only if it is ever needed
        devbuild::k_ob_transform<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(ctx->db.xyz9.p, ctx->xyz9.size() / 3, t);
        RT_CUDA(ctx, cudaGetLastError());
        ctx->db.host_pending.push_back(t);
    } else {
        apply_pending_host_transforms(ctx);
        transform_host_vertices(ctx, t);
        ctx->db.tris_on_device = false;
    }
    return rt_build_bvh(ctx, max_depth, leaf_max_obj_count);
}

int rt_set_materials(RtContext* ctx, const RtMaterial* mats, size_t n)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (n && !mats) return fail(ctx, RT_ERR_INVALID, "mats is NULL");
    static_assert(sizeof(RtMaterial) == 64, "RtMaterial is read as 4 float4");
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    RT_CUDA(ctx, ctx->d_mats.ensure(4 * n));
    if (n) RT_CUDA(ctx, cudaMemcpy(ctx->d_mats.p, mats, n * sizeof(RtMaterial), cudaMemcpyHostToDevice));
    ctx->n_mats = (int)n;
    ctx->any_reflective = false;
    for (size_t i = 0; i < n; i++)
        if (mats[i].reflection > 0.0f) ctx->any_reflective = true;
    return RT_OK;
}

static int upload_shapes(RtContext* ctx)
{
    if (int r = bind(ctx)) return r;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    RT_CUDA(ctx, ctx->d_shapes.ensure(2 * ctx->shapes.size()));
    if (!ctx->shapes.empty())
        RT_CUDA(ctx, cudaMemcpy(ctx->d_shapes.p, ctx->shapes.data(), ctx->shapes.size() * sizeof(HostShape), cudaMemcpyHostToDevice));
    return RT_OK;
}

int rt_add_sphere(RtContext* ctx, const float center[3], float radius, int32_t mat_index)
{
    if (!ctx || !center) return RT_ERR_INVALID;
    if (mat_index < 0) return fail(ctx, RT_ERR_INVALID, "material index %d", mat_index);
    ctx->shapes.push_back(make_sphere(center, radius, mat_index));
    return upload_shapes(ctx);
}

int rt_add_plane(RtContext* ctx, const float point[3], const float normal[3], int32_t mat_index)
{
    if (!ctx || !point || !normal) return RT_ERR_INVALID;
    if (mat_index < 0) return fail(ctx, RT_ERR_INVALID, "material index %d", mat_index);
    ctx->shapes.push_back(make_plane(point, normal, mat_index));
    return upload_shapes(ctx);
}

int rt_clear_analytic_shapes(RtContext* ctx)
{
    if (!ctx) return RT_ERR_INVALID;
    ctx->shapes.clear();
    return RT_OK;
}

static int set_texture(RtContext* ctx, int slot, const void* data, int width, int height, int format)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (slot < 0 || slot >= RT_TEX_COUNT) return fail(ctx, RT_ERR_INVALID, "texture slot %d", slot);
    if (!data || width <= 0 || height <= 0) return fail(ctx, RT_ERR_INVALID, "texture %dx%d", width, height);
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));                      // a frame in flight may still read the old texels
    Texture& t = ctx->tex[slot];
    const size_t bytes = (size_t)width * height * (format == 1 ? 4 : 16);
    const size_t had = (size_t)t.w * t.h * (t.format == 1 ? 4 : 16);
    if (!t.d || had != bytes) {                                            // a map of the same size is replaced in place
        if (t.d) cudaFree(t.d);
        t = Texture();
        RT_CUDA(ctx, cudaMalloc(&t.d, bytes));
    }
    t.w = 0; t.h = 0; t.format = 0;
    RT_CUDA(ctx, cudaMemcpy(t.d, data, bytes, cudaMemcpyHostToDevice));
    t.w = width; t.h = height; t.format = format;
    return RT_OK;
}

int rt_set_texture_f32(RtContext* ctx, int slot, const float* rgba, int width, int height) { return set_texture(ctx, slot, rgba, width, height, 2); }
int rt_set_texture_u8(RtContext* ctx, int slot, const uint8_t* rgba, int width, int height) { return set_texture(ctx, slot, rgba, width, height, 1); }

int rt_clear_texture(RtContext* ctx, int slot)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (slot < 0 || slot >= RT_TEX_COUNT) return fail(ctx, RT_ERR_INVALID, "texture slot %d", slot);
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->tex[slot].d) cudaFree(ctx->tex[slot].d);
    ctx->tex[slot] = Texture();
    return RT_OK;
}

int rt_set_camera(RtContext* ctx, const float proj_inv[16], const float cam_to_world[16], const float position[3])
{
    if (!ctx || !proj_inv || !cam_to_world || !position) return RT_ERR_INVALID;
    memcpy(ctx->proj_inv.m, proj_inv, 64);
    memcpy(ctx->cam_to_world.m, cam_to_world, 64);
    ctx->cam_pos = v3(position[0], position[1], position[2]);
    ctx->camera_set = true;
    return RT_OK;
}

int rt_set_projection(RtContext* ctx, float fov, float aspect, float znear, float zfar)
{
    if (!ctx) return RT_ERR_INVALID;
    if (!(aspect > 0.0f) || !(zfar > znear)) return fail(ctx, RT_ERR_INVALID, "projection: aspect %g, znear %g, zfar %g", aspect, znear, zfar);
    ctx->proj = perspective_matrix(fov, aspect, znear, zfar);                     // Camera::_perspective_proj_mat, scene/camera.cpp:5-19
    ctx->proj_fov = fov;
    ctx->proj_aspect = aspect;
    ctx->proj_set = true;
    return RT_OK;
}

int rt_set_light(RtContext* ctx, const float position[3])
{
    if (!ctx || !position) return RT_ERR_INVALID;
    ctx->light = v3(position[0], position[1], position[2]);
    return RT_OK;
}

// screen_coverage for the camera of rt_set_camera, without a context: a host-only entry point of the library, not part of
// include/rtb200.h, for tests/test_screen_coverage.py.  Writes the bitmap to bits (room for n_words); returns 1 when it
// bounds the scene, 0 when no bound exists (every block is traced), RT_ERR_INVALID on bad arguments.
int rt_screen_coverage(const float proj_inv[16], const float cam_to_world[16], const float position[3], int rw, int rh,
                       const float* boxes, size_t n_boxes, double margin_scale, uint32_t* bits, size_t n_words)
{
    if (!proj_inv || !cam_to_world || !position || rw <= 0 || rh <= 0 || (n_boxes && !boxes) || !bits) return RT_ERR_INVALID;
    M4 pinv, c2w;
    memcpy(pinv.m, proj_inv, 64);
    memcpy(c2w.m, cam_to_world, 64);
    std::vector<uint32_t> out;
    int32_t words = 0;
    const bool bound = screen_coverage(c2w, pinv, v3(position[0], position[1], position[2]), rw, rh, boxes, n_boxes, margin_scale, out, words);
    if (out.size() > n_words) return RT_ERR_INVALID;
    std::copy(out.begin(), out.end(), bits);
    return bound ? 1 : 0;
}

int rt_tile_count(const RtSettings* s, int tile_size, int tile_mod, int tile_rem)
{
    if (!s || tile_size <= 0 || tile_mod <= 0 || tile_rem < 0 || tile_rem >= tile_mod) return RT_ERR_INVALID;
    return (int)owned_tiles(s, tile_size, tile_mod, tile_rem, nullptr).size();
}

int rt_render_device_begin(RtContext* ctx, const RtSettings* s, uint32_t* d_argb_out, int tile_size, int tile_mod, int tile_rem)
{
    if (!ctx) return RT_ERR_INVALID;
    if (ctx->pending.active) return fail(ctx, RT_ERR_STATE, "rt_render_device_begin: the previous frame has not been ended (rt_render_device_end)");
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (int r = validate_scene_for_render(ctx, s)) return r;
    if (int r = check_tile_args(ctx, tile_size, tile_mod, tile_rem)) return r;
    if (!d_argb_out) return fail(ctx, RT_ERR_INVALID, "d_argb_out is NULL");
    const bool ssao = s->enable_ssao != 0;
    const bool raster = s->hybrid_rasterization_tracing != 0;
    if (raster && tile_mod != 1) return fail(ctx, RT_ERR_UNSUPPORTED, "hybrid_rasterization_tracing renders the whole frame on one GPU (one z-buffer)");
    if (raster && !ctx->proj_set) return fail(ctx, RT_ERR_STATE, "hybrid_rasterization_tracing: the projection has not been set (rt_set_projection)");
    if (ssao && tile_mod != 1) return fail(ctx, RT_ERR_UNSUPPORTED, "enable_ssao needs the whole frame on one GPU: its samples read the z-buffer of neighbouring tiles");
    if (ssao && !ctx->proj_set) return fail(ctx, RT_ERR_STATE, "enable_ssao: the projection has not been set (rt_set_projection)");

    bool rebuild_masks = false;                                                // before the views: it may move the mask buffers
    if (ctx->tune.packets && s->compute_shadows && s->shading_method == RT_SHADING)
        if (int r = plan_light_masks(ctx, rebuild_masks)) return r;
    const FrameView fr = frame_view(ctx, s);
    const SceneView sc = scene_view(ctx);
    const SceneView scp = packet_view(ctx);
    const bool resolve = fr.factor > 1;
    const bool reflect = ctx->any_reflective && s->shading_method == RT_SHADING;
    if (reflect) if (int r = ensure_stack(ctx, s)) return r;

    TileList* tl = nullptr;
    if (int r = get_tile_list(ctx, s, tile_size, tile_mod, tile_rem, &tl)) return r;
    const std::vector<uint32_t>& owned = tl->host;
    const int tiles_x = tl->tiles_x;
    WorkView wk = {};
    wk.tiles_x = tiles_x;
    wk.tile_px = tile_size * fr.factor;
    wk.patches_per_side = (wk.tile_px + kPatch - 1) / kPatch;
    // Tiles without a block that the scene's screen coverage (screen_coverage) marks cannot contain a hit: they get no ray
    // slots, no queue entries and no traversal, only the miss colour (k_fill_miss).  The wavefront below runs over the other
    // tiles, and its packets test their own block's bit.
    const bool has_shapes = !ctx->shapes.empty();                             // planes are unbounded: no screen-space bound
    const bool cull = ctx->opt_screen_cull && ctx->tune.packets && !has_shapes && !raster;
    if (cull) if (int r = update_cover(ctx, fr)) return r;
    wk.cover = (cull && ctx->cover_bound) ? ctx->d_cover.p : nullptr;
    wk.cover_words = wk.cover ? ctx->cover_words : 0;
    const bool classify = wk.cover != nullptr && tl->count > 0;
    if (classify) {
        if (!tl->split_valid || tl->split_cover != ctx->cover_generation || tl->split_tile_px != wk.tile_px) {
            std::vector<uint32_t> in, out;
            for (uint32_t tile : owned) {
                const int x0 = (int)(tile % (uint32_t)tiles_x) * wk.tile_px, y0 = (int)(tile / (uint32_t)tiles_x) * wk.tile_px;
                const int x1 = std::min(x0 + wk.tile_px, fr.rw) - 1, y1 = std::min(y0 + wk.tile_px, fr.rh) - 1;
                const bool hit = cover_any(ctx->h_cover, ctx->cover_words, x0, y0, x1, y1);
                (hit ? in : out).push_back(tile);
            }
            tl->n_traced = (uint32_t)in.size();
            tl->split_host = in;
            tl->split_host.insert(tl->split_host.end(), out.begin(), out.end());
            if (!tl->d_split) RT_CUDA(ctx, cudaMalloc((void**)&tl->d_split, tl->count * sizeof(uint32_t)));
            RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));                  // the previous frame may still read the old split
            RT_CUDA(ctx, cudaMemcpy(tl->d_split, tl->split_host.data(), tl->count * sizeof(uint32_t), cudaMemcpyHostToDevice));
            tl->split_cover = ctx->cover_generation;
            tl->split_tile_px = wk.tile_px;
            tl->split_valid = true;
        }
    }
    const uint32_t n_traced = raster ? 0u : (classify ? tl->n_traced : tl->count);   // raster_trace: no primary rays, the wavefront below has no chunks
    const std::vector<uint32_t> tiles(classify ? tl->split_host.begin() : owned.begin(), (classify ? tl->split_host.begin() : owned.begin()) + n_traced);
    const uint64_t px_per_tile = (uint64_t)wk.patches_per_side * wk.patches_per_side * kPatch * kPatch;
    uint32_t tiles_per_chunk = (uint32_t)std::max<uint64_t>(1, ctx->opt_chunk_pixels / px_per_tile);
    if ((tiles.size() + tiles_per_chunk - 1) / tiles_per_chunk > (size_t)kMaxChunks)
        tiles_per_chunk = (uint32_t)((tiles.size() + kMaxChunks - 1) / kMaxChunks);
    // Two chunks are in flight at a time, each on its own stream ("lane") with its own queues: the persistent kernels of
    // one chunk fill the SMs that the other chunk's kernels leave idle while their last, longest packets finish (within
    // one stream a kernel cannot start before the previous one has ended completely).  A frame that fits one chunk is cut
    // in two for that purpose.
    const int n_lanes = (ctx->opt_lanes > 1 && tune_packets_hint(ctx)) ? (int)std::min<size_t>((size_t)ctx->opt_lanes, std::max<size_t>(tiles.size(), 1)) : 1;
    if (n_lanes > 1 && tiles.size() <= (size_t)tiles_per_chunk * (n_lanes - 1)) tiles_per_chunk = (uint32_t)((tiles.size() + n_lanes - 1) / n_lanes);
    // chunk c covers tiles [bounds[c], bounds[c + 1])
    std::vector<uint32_t> bounds;
    for (size_t b = 0; b < tiles.size(); b += tiles_per_chunk) bounds.push_back((uint32_t)b);
    bounds.push_back((uint32_t)tiles.size());
    const uint32_t n_chunks = (uint32_t)bounds.size() - 1u;
    uint32_t largest_chunk = 0;
    for (uint32_t c = 0; c < n_chunks; c++) largest_chunk = std::max(largest_chunk, bounds[c + 1] - bounds[c]);
    const size_t qcap = (size_t)largest_chunk * px_per_tile;

    RT_CUDA(ctx, ctx->d_counters.ensure(std::max<uint32_t>(n_chunks, 1)));
    // Round budgets.  Positive option values are fixed budgets.  Negative ones (the defaults) are adaptive: a packet is
    // split after 8 |n| rounds at the latest, and after |n| / 4 rounds as soon as its launch has no unfetched packets left
    // (Drain, kernels.cuh) -- a packet is only worth splitting when it would otherwise be the tail of its launch.  The same
    // for the work items of a pass, with |n| rounds as the minimum.  Primary packets are only split in SHORT launches (fewer
    // than 256 packets per resident warp, e.g. one of 8 tile shards of a 4K frame): a long launch hides its stragglers,
    // and the item passes of a stage that splits nothing still cost their launches (measured: +0.3 ms on a whole 4K frame).
    const int pw = grid_for(ctx, (const void*)k_primary_packet<false, false>, kPrimaryThreads) * (kPrimaryThreads / 32);
    const bool short_launch = (uint64_t)owned.size() * px_per_tile / 32 < (uint64_t)256 * (uint64_t)pw;
    auto largest = [](int32_t v) { return v >= 0 ? v : std::min<int32_t>(-v, 1 << 27) * 8; };
    auto least = [](int32_t v, int div) { return v >= 0 ? 0 : std::max<int32_t>(1, -v / div); };
    Tuning tune = ctx->tune;
    tune.packet_rounds = largest(ctx->tune.packet_rounds); tune.packet_min = least(ctx->tune.packet_rounds, 4);
    tune.item_rounds = largest(ctx->tune.item_rounds); tune.item_min = least(ctx->tune.item_rounds, 1);
    tune.primary_rounds = largest(ctx->tune.primary_rounds); tune.primary_min = least(ctx->tune.primary_rounds, 4);
    if (ctx->tune.primary_rounds < 0 && !short_launch) tune.primary_rounds = tune.primary_min = 0;
    if (tune.fused && tune.packets) {
        // fused item scheduling: the values are the LARGEST budgets -- a packet's own budget shrinks as the launch runs out
        // of packets (fq_budget, kernels.cuh) --, so nothing depends on the length of the launch
        auto magnitude = [](int32_t v) { return v >= 0 ? v : -v; };
        tune.packet_rounds = magnitude(ctx->tune.packet_rounds);
        tune.item_rounds = magnitude(ctx->tune.item_rounds);
        tune.primary_rounds = magnitude(ctx->tune.primary_rounds);
        tune.packet_min = tune.item_min = tune.primary_min = 0;
    }
    const bool tail = tune.packets && tune.packet_rounds > 0 && s->compute_shadows && s->shading_method == RT_SHADING;
    const bool psplit = tune.packets && tune.primary_rounds > 0;
    // light-space ordering of the hit queue before the shadow packets are formed (kernels.cuh).  Not with reflection fans:
    // their queue indexes the hit queue in compaction order.
    // In the adaptive mode the kernels decide on the device (sparse hits: fewer than 1 in 4 ray slots); when the last frame of
    // the same tile list was clearly dense, the five launches are not even enqueued (they matter to a short launch).
    const bool sort_hits = ctx->opt_shadow_sort && tune.packets && !tune.fused && !reflect && s->compute_shadows && s->shading_method == RT_SHADING &&
                           !(ctx->opt_shadow_sort == 2 && tl->last_hit_fraction >= 0.3f);
    LightMap light_map;
    memset(&light_map, 0, sizeof(light_map));
    if (sort_hits) light_map = make_light_map(ctx);
    // split records and work items of the packets that run out of rounds; a packet that finds them full is finished in
    // place.  Primary and shadow packets never run at the same time and share the storage.
    const size_t split_cap = (tail || psplit) ? std::min<size_t>(std::max<size_t>(qcap / 32, 1024), (size_t)1 << 20) : 0;
    const size_t item_cap = (tail || psplit) ? std::min<size_t>(std::max<size_t>(qcap / 4, (size_t)1 << 14), (size_t)1 << 21) : 0;
    for (int l = 0; l < n_lanes; l++) {
        QueueSet& Q = ctx->qs[l];
        if (tail || psplit) {
            RT_CUDA(ctx, Q.split_base.ensure(split_cap)); RT_CUDA(ctx, Q.split_active.ensure(split_cap)); RT_CUDA(ctx, Q.split_occ.ensure(split_cap));
            RT_CUDA(ctx, Q.items.ensure(item_cap * kItemPasses));
            if (tune.fused) {
                if (Q.item_ready.n < item_cap * kItemPasses) {                   // fresh flags must not look like a tag
                    RT_CUDA(ctx, Q.item_ready.ensure(item_cap * kItemPasses));
                    RT_CUDA(ctx, cudaMemsetAsync(Q.item_ready.p, 0, Q.item_ready.n * sizeof(uint32_t), ctx->stream));
                }
                RT_CUDA(ctx, Q.split_pending.ensure(split_cap));
            }
        }
        if (psplit) RT_CUDA(ctx, Q.split_best.ensure(split_cap * 32));
        RT_CUDA(ctx, Q.hit_slot.ensure(qcap)); RT_CUDA(ctx, Q.tri.ensure(qcap)); RT_CUDA(ctx, Q.t.ensure(qcap));
        RT_CUDA(ctx, Q.u.ensure(qcap)); RT_CUDA(ctx, Q.v.ensure(qcap));
        if (reflect) { RT_CUDA(ctx, Q.refl_idx.ensure(qcap)); RT_CUDA(ctx, Q.refl_rgb.ensure(3 * qcap)); RT_CUDA(ctx, Q.refl_cnt.ensure(3 * qcap)); }
        if (sort_hits) {
            RT_CUDA(ctx, Q.hit_sorted.ensure(qcap)); RT_CUDA(ctx, Q.sort_keys.ensure(qcap));
            RT_CUDA(ctx, Q.sort_bins.ensure((size_t)kSortBins + kSortScanBlocks));
        }
    }
    uint32_t* super = d_argb_out;
    if (resolve) {
        RT_CUDA(ctx, ctx->d_super.ensure((size_t)fr.rw * fr.rh));
        super = ctx->d_super.p;
    }
    if (ssao) {
        const size_t px = (size_t)fr.rw * fr.rh;
        RT_CUDA(ctx, ctx->d_gz.ensure(px)); RT_CUDA(ctx, ctx->d_gn.ensure(px)); RT_CUDA(ctx, ctx->d_ao.ensure(px));
    }
    wk.tiles = classify ? tl->d_split : tl->d;
    QueueView qv[kMaxLanes];
    memset(qv, 0, sizeof(qv));                                                 // padding too: the views are part of the frame-graph key
    for (int l = 0; l < n_lanes; l++) {
        QueueSet& Q = ctx->qs[l];
        QueueView& q = qv[l];
        q.hit_slot = Q.hit_slot.p; q.slot_tri = Q.tri.p; q.slot_t = Q.t.p; q.slot_u = Q.u.p; q.slot_v = Q.v.p;
        q.split_base = Q.split_base.p; q.split_active = Q.split_active.p; q.split_occ = Q.split_occ.p;
        q.split_best = Q.split_best.p;
        q.items = Q.items.p; q.split_capacity = (uint32_t)split_cap; q.item_capacity = (uint32_t)item_cap;
        q.item_ready = Q.item_ready.p; q.split_pending = Q.split_pending.p; q.tag = 0;
        q.refl_idx = Q.refl_idx.p; q.refl_rgb = Q.refl_rgb.p; q.refl_cnt = Q.refl_cnt.p; q.capacity = (uint32_t)qcap;
        q.hit_sorted = nullptr; q.sort_mode = 0u; q.sort_slots = 0u;
        q.g_z = ssao ? ctx->d_gz.p : nullptr; q.g_n = ssao ? ctx->d_gn.p : nullptr;
    }
    for (int l = 1; l < n_lanes; l++) {
        if (ctx->lane_stream[l]) continue;
        RT_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->lane_stream[l], cudaStreamNonBlocking));
        RT_CUDA(ctx, cudaEventCreateWithFlags(&ctx->lane_join[l], cudaEventDisableTiming));
    }
    if (n_lanes > 1 && !ctx->lane_fork) RT_CUDA(ctx, cudaEventCreateWithFlags(&ctx->lane_fork, cudaEventDisableTiming));

    const cudaStream_t main_stream = ctx->stream;
    cudaStream_t st = main_stream;
    ctx->events_used = 0;
    ctx->timed.clear();
    uint32_t launches = 0;
    const bool count = ctx->opt_count_work || ctx->frame_work_map != nullptr;   // a work-map frame runs the instrumented kernels
    Pending& pd = ctx->pending;
    const size_t n_cnt = std::max<uint32_t>(n_chunks, 1);
    if (n_cnt > pd.host_cap) {
        if (pd.host_cnt) cudaFreeHost(pd.host_cnt);
        pd.host_cnt = nullptr; pd.host_cap = 0;
        RT_CUDA(ctx, cudaHostAlloc((void**)&pd.host_cnt, n_cnt * sizeof(ChunkCounters), cudaHostAllocDefault));
        pd.host_cap = n_cnt;
    }

    // ---- the frame as a graph.  Everything the launches below depend on is serialised into a key; a frame whose key
    // equals the previous frame's is captured (stream capture, the lanes' streams join through their fork / join events),
    // and from then on frames with that key are ONE cudaGraphLaunch: a tile shard's 40 short dependent launches otherwise
    // cost more host and launch latency than their kernels run (a 1/8 shard of the 4K frame: 2.2 ms, 0.5 ms of it the chain).
    static const bool trace_env = getenv("RTB200_TRACE") != nullptr;
    const bool graph_ok = ctx->opt_graph && !raster && !(tune.fused && tune.packets) && !trace_env && ctx->frame_work_map == nullptr;
    bool replay = false, capture = false;
    size_t graph_at = 0;
    std::string key;
    if (graph_ok) {
        auto put = [&](const void* ptr, size_t n) { key.append((const char*)ptr, n); };
        auto put64 = [&](unsigned long long v) { put(&v, sizeof(v)); };
        put(&sc, sizeof(sc)); put(&scp, sizeof(scp)); put(&fr, sizeof(fr)); put(&wk, sizeof(wk)); put(qv, sizeof(QueueView) * (size_t)n_lanes); put(&tune, sizeof(tune));
        put(&light_map, sizeof(light_map));
        if (!bounds.empty()) put(bounds.data(), bounds.size() * sizeof(uint32_t));
        put64((unsigned long long)tile_size); put64((unsigned long long)tile_mod); put64((unsigned long long)tile_rem); put64((unsigned long long)n_lanes);
        put64(n_chunks); put64(classify); put64(n_traced); put64(tl->count); put64((unsigned long long)(uintptr_t)tl->d); put64((unsigned long long)(uintptr_t)tl->d_split);
        put64(sort_hits); put64((unsigned long long)ctx->opt_shadow_sort); put64(tail); put64(psplit); put64(reflect); put64(ssao); put64(resolve); put64(count); put64(has_shapes);
        put64(ctx->opt_top_table); put64((unsigned long long)(uintptr_t)d_argb_out); put64((unsigned long long)(uintptr_t)super);
        put64((unsigned long long)(uintptr_t)ctx->d_counters.p); put64((unsigned long long)(uintptr_t)pd.host_cnt); put64(g_alloc_generation.load());
        put64((unsigned long long)(uintptr_t)main_stream); put64((unsigned long long)split_cap); put64((unsigned long long)item_cap); put64(px_per_tile);
        put64((unsigned long long)ctx->stack_limit_set); put64(ctx->opt_fan_lanes); put64(ctx->mask_generation); put64(ctx->cover_generation);
        if (ssao) { put(&ctx->proj, sizeof(ctx->proj)); put(&ctx->proj_fov, sizeof(float)); put(&ctx->proj_aspect, sizeof(float)); }
        for (size_t i = 0; i < ctx->graphs.size() && !replay; i++)
            if (ctx->graphs[i].key == key) { replay = true; graph_at = i; }
        if (!replay) {
            for (const std::string& k : ctx->seen_keys) capture |= (k == key);
            if (!capture) {
                if (ctx->seen_keys.size() >= 4) ctx->seen_keys.erase(ctx->seen_keys.begin());
                ctx->seen_keys.push_back(key);
            }
        }
    }
    cudaEvent_t ev_begin = next_event(ctx), ev_end = next_event(ctx);
    RT_CUDA(ctx, cudaEventRecord(ev_begin, st));
    if (rebuild_masks) if (int r = build_light_masks(ctx, st)) return r;
    auto enqueue = [&]() -> int {
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, sizeof(ChunkCounters) * std::max<uint32_t>(n_chunks, 1), st));
    if (ctx->frame_work_map) {                                                 // every chunk's counters point at the work map
        ctx->work_map_ptrs.assign(n_cnt, ctx->frame_work_map);
        RT_CUDA(ctx, cudaMemcpy2DAsync(&ctx->d_counters.p->work_map, sizeof(ChunkCounters), ctx->work_map_ptrs.data(), sizeof(unsigned long long*),
                                       sizeof(unsigned long long*), n_cnt, cudaMemcpyHostToDevice, st));
    }
    if (ssao) { k_gbuffer_clear<<<ctx->sm_count * 8, 256, 0, st>>>(ctx->d_gz.p, ctx->d_gn.p, (size_t)fr.rw * fr.rh); launches++; }

    int (&grids)[2][11] = ctx->grids;                                           // per context: its device's occupancy
    if (!grids[count][0]) {
        grids[count][3] = grid_for(ctx, count ? (const void*)k_primary_packet<true, true> : (const void*)k_primary_packet<false, true>, kPrimaryThreads);
        grids[count][4] = grid_for(ctx, count ? (const void*)k_shade_packet<true, true> : (const void*)k_shade_packet<false, true>, kQueueThreads);
        grids[count][5] = grid_for(ctx, count ? (const void*)k_shade_items<true> : (const void*)k_shade_items<false>, kQueueThreads);
        grids[count][7] = grid_for(ctx, count ? (const void*)k_primary_items<true> : (const void*)k_primary_items<false>, kPrimaryThreads);
        grids[count][8] = grid_for(ctx, (const void*)k_primary_finish, kPrimaryThreads);
        grids[count][6] = grid_for(ctx, count ? (const void*)k_shade_finish<true> : (const void*)k_shade_finish<false>, kQueueThreads);
        grids[count][9] = grid_for(ctx, count ? (const void*)k_primary_fused<true> : (const void*)k_primary_fused<false>, kPrimaryThreads);
        grids[count][10] = grid_for(ctx, count ? (const void*)k_shade_fused<true> : (const void*)k_shade_fused<false>, kQueueThreads);
        grids[count][0] = grid_for(ctx, count ? (const void*)k_primary<true> : (const void*)k_primary<false>, kPrimaryThreads);
        grids[count][1] = grid_for(ctx, count ? (const void*)k_reflect<true> : (const void*)k_reflect<false>, kQueueThreads);
        grids[count][2] = grid_for(ctx, count ? (const void*)k_shade<true> : (const void*)k_shade<false>, kQueueThreads);
    }
    const int grid_primary = grids[count][0], grid_reflect = grids[count][1], grid_shade = grids[count][2];
    const int grid_pp = grids[count][3], grid_sp = grids[count][4], grid_items = grids[count][5], grid_finish = grids[count][6], grid_pitems = grids[count][7], grid_pfinish = grids[count][8];
    // A fused kernel's CTAs all stay until the launch's last work item has completed, so two lanes' kernels only run side by
    // side if each takes its share of the SMs' CTA slots from the start: the persistent grid is divided among the lanes.
    const int grid_pf = std::max(ctx->sm_count, grids[count][9] / n_lanes), grid_sf = std::max(ctx->sm_count, grids[count][10] / n_lanes);
    if (n_lanes > 1) {                                                         // the other lanes start after everything enqueued so far
        RT_CUDA(ctx, cudaEventRecord(ctx->lane_fork, main_stream));
        for (int l = 1; l < n_lanes; l++) RT_CUDA(ctx, cudaStreamWaitEvent(ctx->lane_stream[l], ctx->lane_fork, 0));
    }
    for (uint32_t c = 0; c < n_chunks; c++) {
        wk.tile_begin = bounds[c];
        wk.tile_end = bounds[c + 1];
        ChunkCounters* cnt = ctx->d_counters.p + c;
        const int lane = (int)(c % (uint32_t)n_lanes);
        st = lane ? ctx->lane_stream[lane] : main_stream;
        const QueueView& q = qv[lane];
        {
            ScopedTimer tm(ctx, ST_PRIMARY, st);
            auto next_tag = [&]() { if (++ctx->frame_serial == 0u) ctx->frame_serial = 1u; return ctx->frame_serial; };
            if (tune.packets && tune.fused) {
                // one launch: the packet kernel's warps also consume the work items of the packets they split
                QueueView qf = q;
                qf.tag = next_tag();
                ScopedTimer t1(ctx, ST_PRIMARY, st, "  k_primary_fused");
                if (count) k_primary_fused<true><<<grid_pf, kPrimaryThreads, 0, st>>>(scp, fr, wk, qf, cnt, super, tune);
                else k_primary_fused<false><<<grid_pf, kPrimaryThreads, 0, st>>>(scp, fr, wk, qf, cnt, super, tune);
                launches++;
            } else {
            if (tune.packets) {
                ScopedTimer t1(ctx, ST_PRIMARY, st, "  k_primary_packet");
                const bool use_top = ctx->opt_top_table && scp.top_n > 0;
                if (count) {
                    if (use_top) k_primary_packet<true, true><<<grid_pp, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, super, tune);
                    else k_primary_packet<true, false><<<grid_pp, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, super, tune);
                } else if (use_top) k_primary_packet<false, true><<<grid_pp, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, super, tune);
                else k_primary_packet<false, false><<<grid_pp, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, super, tune);
            } else if (count) k_primary<true><<<grid_primary, kPrimaryThreads, 0, st>>>(sc, fr, wk, q, cnt, super, tune);
            else k_primary<false><<<grid_primary, kPrimaryThreads, 0, st>>>(sc, fr, wk, q, cnt, super, tune);
            launches++;
            if (psplit) {
                for (int pass = 0; pass < tune.item_passes; pass++) {
                    ScopedTimer t1(ctx, ST_PRIMARY, st, "  k_primary_items");
                    if (count) k_primary_items<true><<<grid_pitems, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, tune, pass);
                    else k_primary_items<false><<<grid_pitems, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, tune, pass);
                }
                k_primary_finish<<<grid_pfinish, kPrimaryThreads, 0, st>>>(scp, fr, wk, q, cnt, super);
                launches += tune.item_passes + 1;
            }
            }
            if (has_shapes) {                                                  // trace_ray's loop over the analytic shapes
                const uint32_t slots = (wk.tile_end - wk.tile_begin) * (uint32_t)px_per_tile;
                k_primary_shapes<<<ctx->sm_count * 8, 256, 0, st>>>(sc, fr, wk, q, slots, super);
                launches++;
            }
        }
        {
            ScopedTimer tm(ctx, ST_COMPACT, st);
            const uint32_t slots = (wk.tile_end - wk.tile_begin) * (uint32_t)px_per_tile;
            const uint32_t blocks = std::min<uint32_t>((slots + kCompactSlots - 1) / kCompactSlots, (uint32_t)ctx->sm_count * 8u);
            k_compact<<<blocks, kCompactThreads, 0, st>>>(sc, q, cnt, slots, reflect ? 1 : 0);
            launches++;
        }
        QueueView qsorted = q;                                                 // the shade stage's view of the queues
        if (sort_hits) {
            ScopedTimer tm(ctx, ST_COMPACT, st);
            QueueSet& Q = ctx->qs[lane];
            uint32_t* bins = Q.sort_bins.p;
            uint32_t* partial = bins + kSortBins;
            qsorted.hit_sorted = Q.hit_sorted.p;
            qsorted.sort_mode = (uint32_t)ctx->opt_shadow_sort;
            qsorted.sort_slots = (wk.tile_end - wk.tile_begin) * (uint32_t)px_per_tile;
            RT_CUDA(ctx, cudaMemsetAsync(bins, 0, sizeof(uint32_t) * kSortBins, st));
            k_sort_keys<<<ctx->sm_count * 4, 256, 0, st>>>(fr, wk, qsorted, cnt, light_map, Q.sort_keys.p, bins);
            k_sort_partial<<<kSortScanBlocks, kSortScanThreads, 0, st>>>(qsorted, cnt, bins, partial);
            k_sort_scan<<<kSortScanBlocks, kSortScanThreads, 0, st>>>(qsorted, cnt, bins, partial);
            k_sort_scatter<<<ctx->sm_count * 4, 256, 0, st>>>(qsorted, cnt, Q.sort_keys.p, bins);
            launches += 4;
        }
        if (reflect) {
            ScopedTimer tm(ctx, ST_REFLECT, st);
            // one lane per fan ray where the fan is a fixed point of its own hits (k_reflect_fan); else one thread per fan
            const bool fan_lanes = ctx->opt_fan_lanes && !count && s->max_recursion_depth == 1 && !s->enable_normal_mapping &&
                                   s->rough_reflections_sample_count >= 1 && s->rough_reflections_sample_count <= 32;
            if (fan_lanes) {
                if (!ctx->grid_fan) ctx->grid_fan = grid_for(ctx, (const void*)k_reflect_fan, kQueueThreads);
                k_reflect_fan<<<ctx->grid_fan, kQueueThreads, 0, st>>>(sc, fr, wk, q, cnt);
            } else if (count) k_reflect<true><<<grid_reflect, kQueueThreads, 0, st>>>(sc, fr, wk, q, cnt);
            else k_reflect<false><<<grid_reflect, kQueueThreads, 0, st>>>(sc, fr, wk, q, cnt);
            launches++;
        }
        {
            ScopedTimer tm(ctx, ST_SHADE, st);
            if (tune.packets && tune.fused) {
                QueueView qf = q;
                if (++ctx->frame_serial == 0u) ctx->frame_serial = 1u;
                qf.tag = ctx->frame_serial;
                ScopedTimer t1(ctx, ST_SHADE, st, "  k_shade_fused");
                if (count) k_shade_fused<true><<<grid_sf, kQueueThreads, 0, st>>>(scp, fr, wk, qf, cnt, super, tune);
                else k_shade_fused<false><<<grid_sf, kQueueThreads, 0, st>>>(scp, fr, wk, qf, cnt, super, tune);
                launches++;
            } else {
            if (tune.packets) {
                ScopedTimer t1(ctx, ST_SHADE, st, "  k_shade_packet");
                const bool use_top = ctx->opt_top_table && scp.top_n > 0;
                if (count) {
                    if (use_top) k_shade_packet<true, true><<<grid_sp, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super, tune);
                    else k_shade_packet<true, false><<<grid_sp, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super, tune);
                } else if (use_top) k_shade_packet<false, true><<<grid_sp, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super, tune);
                else k_shade_packet<false, false><<<grid_sp, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super, tune);
            } else if (count) k_shade<true><<<grid_shade, kQueueThreads, 0, st>>>(sc, fr, wk, qsorted, cnt, super, tune);
            else k_shade<false><<<grid_shade, kQueueThreads, 0, st>>>(sc, fr, wk, qsorted, cnt, super, tune);
            launches++;
            if (tail) {
                for (int pass = 0; pass < tune.item_passes; pass++) {
                    ScopedTimer t1(ctx, ST_SHADE, st, "  k_shade_items");
                    if (count) k_shade_items<true><<<grid_items, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, tune, pass);
                    else k_shade_items<false><<<grid_items, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, tune, pass);
                }
                if (count) k_shade_finish<true><<<grid_finish, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super);
                else k_shade_finish<false><<<grid_finish, kQueueThreads, 0, st>>>(scp, fr, wk, qsorted, cnt, super);
                launches += tune.item_passes + 1;
            }
            }
        }
    }
    st = main_stream;
    if (raster && !owned.empty()) {
        // Renderer::raster_trace (renderer.cpp:869-1006): depth pass, emit pass, shade pass (raster.cuh)
        const size_t npx = (size_t)fr.rw * fr.rh;
        RasterView rv;
        rv.world_to_cam = invert_matrix(ctx->cam_to_world);                    // Camera::_world_to_camera_mat, renderer.cpp:229
        rv.proj = ctx->proj;
        rv.clipping = s->enable_clipping;
        const size_t smem = ((size_t)fr.rw + kRasterBandRows) * sizeof(float);
        if (smem > 200 * 1024) return fail(ctx, RT_ERR_UNSUPPORTED, "hybrid_rasterization_tracing: frame wider than 51 000 supersampled pixels");
        if (smem > 48 * 1024 && smem > ctx->raster_smem_set) {
            RT_CUDA(ctx, cudaFuncSetAttribute(k_raster_units<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RT_CUDA(ctx, cudaFuncSetAttribute(k_raster_units<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ctx->raster_smem_set = smem;
        }
        const int shade_grid = ctx->sm_count * 8, shade_threads = 128;
        RT_CUDA(ctx, ctx->d_rkeys.ensure(npx)); RT_CUDA(ctx, ctx->d_rxy.ensure(npx)); RT_CUDA(ctx, ctx->d_rcount.ensure(1));
        RT_CUDA(ctx, ctx->d_rfrag.ensure((size_t)2 * shade_grid * shade_threads));
        if (ctx->d_runits.n == 0) RT_CUDA(ctx, ctx->d_runits.ensure(ctx->raster_units0));
        SceneView scf = sc;
        scf.frag_shade = ctx->d_rfrag.p;
        const int tri_grid = (int)std::min<uint64_t>(((uint64_t)ctx->n_tris + 127) / 128, (uint64_t)ctx->sm_count * 16), unit_grid = ctx->sm_count * 4;
        RasterBuffers rb;
        rb.keys = ctx->d_rkeys.p; rb.frag_xy = ctx->d_rxy.p; rb.n_units = ctx->d_rcount.p;
        {
            ScopedTimer tm(ctx, ST_PRIMARY, st);
            unsigned int n_units = 0;
            for (;;) {                                                         // depth pass; repeated once if the unit list was too short
                rb.units = ctx->d_runits.p;
                rb.unit_cap = (uint32_t)std::min<size_t>(ctx->d_runits.n, 0xffffffffu);
                RT_CUDA(ctx, cudaMemsetAsync(rb.keys, 0xff, npx * sizeof(unsigned long long), st));     // RT_RASTER_EMPTY = clear_z_buffer()
                RT_CUDA(ctx, cudaMemsetAsync(rb.n_units, 0, sizeof(unsigned int), st));
                if (ctx->n_tris) { k_raster_tris<false><<<tri_grid, 128, 0, st>>>(sc, fr, rv, rb); launches++; }
                // the number of work units says whether the list was long enough: a raster_trace frame waits for it here
                RT_CUDA(ctx, cudaMemcpyAsync(&n_units, rb.n_units, sizeof(n_units), cudaMemcpyDeviceToHost, st));
                RT_CUDA(ctx, cudaStreamSynchronize(st));
                if (n_units <= rb.unit_cap) break;
                RT_CUDA(ctx, ctx->d_runits.ensure((size_t)n_units + n_units / 4));
            }
            if (n_units) { k_raster_units<false><<<unit_grid, kRasterUnitThreads, smem, st>>>(sc, fr, rv, rb); launches++; }
            if (ctx->n_tris) { k_raster_tris<true><<<tri_grid, 128, 0, st>>>(sc, fr, rv, rb); launches++; }
            if (n_units) { k_raster_units<true><<<unit_grid, kRasterUnitThreads, smem, st>>>(sc, fr, rv, rb); launches++; }
        }
        {
            const uint32_t background = quantise_argb(col(135.0f / 255.0f, 206.0f / 255.0f, 235.0f / 255.0f));   // clear_image(), renderer.cpp:19,175-180
            ScopedTimer ts(ctx, ST_SHADE, st);
            if (count) k_raster_shade<true><<<shade_grid, shade_threads, 0, st>>>(scf, fr, rv, rb, ctx->d_rfrag.p, super, ssao ? ctx->d_gz.p : nullptr, ssao ? ctx->d_gn.p : nullptr, background, ctx->d_counters.p);
            else k_raster_shade<false><<<shade_grid, shade_threads, 0, st>>>(scf, fr, rv, rb, ctx->d_rfrag.p, super, ssao ? ctx->d_gz.p : nullptr, ssao ? ctx->d_gn.p : nullptr, background, ctx->d_counters.p);
            launches++;
        }
    }
    for (int l = 1; l < n_lanes; l++) {                                        // the frame continues when all lanes are done
        RT_CUDA(ctx, cudaEventRecord(ctx->lane_join[l], ctx->lane_stream[l]));
        RT_CUDA(ctx, cudaStreamWaitEvent(main_stream, ctx->lane_join[l], 0));
    }
    // the tiles that cannot contain a hit: miss colour only.  With a ray-independent miss colour and a resolve pass the
    // resolved pixel IS that colour: k_resolve writes it and the samples of those tiles are never produced.
    const bool const_fill = resolve && !(s->enable_skysphere || s->enable_skybox);
    if (classify && n_traced < tl->count && !const_fill) {
        wk.tile_begin = n_traced;
        wk.tile_end = tl->count;
        ScopedTimer tm(ctx, ST_PRIMARY);
        k_fill_miss<<<ctx->sm_count * 8, 256, 0, st>>>(sc, fr, wk, super);
        launches++;
    }
    if (ssao && !owned.empty()) {
        // Renderer::post_process: SSAO on the supersampled image, then the SSAA resolve (renderer.cpp:1118-1124)
        SsaoView sv;
        sv.rw = fr.rw; sv.rh = fr.rh; sv.z = ctx->d_gz.p; sv.n = ctx->d_gn.p;
        sv.proj = ctx->proj;
        sv.aspect = ctx->proj_aspect;
        sv.fov_mult_simd = (float)std::tan(ctx->proj_fov / 2 / 180 * M_PI);                  // renderer.cpp:1249
        sv.fov_mult_scalar = std::tan(((float)M_PI / 180) * (ctx->proj_fov / 2));            // radians(), mat.cpp:13-16, std::tan(float)
        sv.samples = s->ssao_sample_count; sv.radius = s->ssao_radius; sv.amount = s->ssao_amount;
        sv.rng_seed = s->rng_seed;
        ScopedTimer tm(ctx, ST_RESOLVE);
        k_ssao_occlusion<<<ctx->sm_count * 16, 128, 0, st>>>(sv, ctx->d_ao.p);
        k_ssao_apply<<<ctx->sm_count * 8, 256, 0, st>>>(sv, ctx->d_ao.p, super);
        launches += 2;
    }
    if (resolve && !owned.empty()) {
        wk.tile_begin = 0;
        wk.tile_end = tl->count;                                               // all owned tiles, traced or not
        const uint32_t background = quantise_argb(col(135.0f / 255.0f, 206.0f / 255.0f, 235.0f / 255.0f));   // renderer.cpp:19, as shade_miss
        ScopedTimer tm(ctx, ST_RESOLVE);
        k_resolve<<<ctx->sm_count * 8, 256, 0, st>>>(super, d_argb_out, wk, tile_size, fr.factor, s->image_width, s->image_height,
                                                     (classify && const_fill) ? n_traced : tl->count, background);
        launches++;
    }
    // the counters come back in the same stream order and are read by rt_render_device_end
    RT_CUDA(ctx, cudaMemcpyAsync(pd.host_cnt, ctx->d_counters.p, sizeof(ChunkCounters) * n_cnt, cudaMemcpyDeviceToHost, st));
    return RT_OK;
    };
    if (replay) {
        RT_CUDA(ctx, cudaGraphLaunch(ctx->graphs[graph_at].exec, main_stream));
        launches = ctx->graphs[graph_at].launches;
    } else if (capture) {
        if (ctx->graphs.size() >= 4) { cudaGraphExecDestroy(ctx->graphs.front().exec); ctx->graphs.erase(ctx->graphs.begin()); }
        RT_CUDA(ctx, cudaStreamBeginCapture(main_stream, cudaStreamCaptureModeRelaxed));
        ctx->capturing = true;
        const int rc = enqueue();
        ctx->capturing = false;
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(main_stream, &graph);
        if (rc != RT_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess || !graph) {
            // the sequence cannot be captured: run this frame and the following ones the ordinary way
            (void)cudaGetLastError();
            if (graph) cudaGraphDestroy(graph);
            ctx->opt_graph = false;
            launches = 0;
            st = main_stream;
            if (int r = enqueue()) return r;
        } else {
            cudaGraphExec_t exec = nullptr;
            const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) return fail(ctx, RT_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie));
            RtContext::FrameGraph fg;
            fg.key = key; fg.exec = exec; fg.launches = launches;
            ctx->graphs.push_back(fg);
            RT_CUDA(ctx, cudaGraphLaunch(exec, main_stream));
        }
    } else if (int r = enqueue()) return r;
    st = main_stream;
    RT_CUDA(ctx, cudaEventRecord(ev_end, st));
    RT_CUDA(ctx, cudaGetLastError());

    // everything is enqueued
    pd.n_chunks = raster ? 1u : n_chunks;
    pd.raster = raster;
    pd.launches = launches;
    pd.count = count;
    pd.ev_begin = ev_begin; pd.ev_end = ev_end;
    pd.shadow = s->shading_method == RT_SHADING && s->compute_shadows;
    pd.has_key = !raster;
    pd.key[0] = s->image_width; pd.key[1] = s->image_height; pd.key[2] = tile_size; pd.key[3] = tile_mod; pd.key[4] = tile_rem;
    pd.traced_slots = (uint64_t)n_traced * px_per_tile;
    pd.primary_rays = 0;                                  // supersampled pixels of the owned tiles that lie inside the frame
    for (uint32_t tile : owned) {
        int tx = (int)(tile % (uint32_t)tiles_x), ty = (int)(tile / (uint32_t)tiles_x);
        int w = std::min(tile_size, s->image_width - tx * tile_size), h = std::min(tile_size, s->image_height - ty * tile_size);
        pd.primary_rays += (uint64_t)w * h * fr.factor * fr.factor;
    }
    pd.active = true;
    return RT_OK;
}

int rt_render_device_end(RtContext* ctx, RtRenderStats* stats)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    Pending& pd = ctx->pending;
    if (!pd.active) return fail(ctx, RT_ERR_STATE, "rt_render_device_end without rt_render_device_begin");
    pd.active = false;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const ChunkCounters* host_cnt = pd.host_cnt;
    const uint32_t n_chunks = pd.n_chunks;
    const bool count = pd.count;
    const cudaEvent_t ev_begin = pd.ev_begin, ev_end = pd.ev_end;

    RtRenderStats rs;
    memset(&rs, 0, sizeof(rs));
    bool overflow = false;
    for (uint32_t c = 0; c < n_chunks; c++) {
        rs.primary_hits += host_cnt[c].n_hits;
        rs.reflection_rays += host_cnt[c].refl_rays;
        rs.reflection_shadow_rays += host_cnt[c].refl_shadow_rays;
        rs.primary_volume_tests += host_cnt[c].primary_vol; rs.primary_triangle_tests += host_cnt[c].primary_tri;
        rs.shadow_volume_tests += host_cnt[c].shadow_vol; rs.shadow_triangle_tests += host_cnt[c].shadow_tri;
        rs.reflection_volume_tests += host_cnt[c].refl_vol; rs.reflection_triangle_tests += host_cnt[c].refl_tri;
        rs.primary_fetched_bytes += host_cnt[c].primary_fetch; rs.shadow_fetched_bytes += host_cnt[c].shadow_fetch;
        rs.reflection_fetched_bytes += host_cnt[c].refl_fetch;
        rs.traced_primary_rays += host_cnt[c].traced_primary;
        overflow |= host_cnt[c].stack_overflow != 0;
    }
    if (pd.has_key) {
        auto it = ctx->tile_lists.find(TileKey(pd.key[0], pd.key[1], pd.key[2], pd.key[3], pd.key[4]));
        if (it != ctx->tile_lists.end()) it->second.last_hit_fraction = pd.traced_slots ? (float)((double)rs.primary_hits / (double)pd.traced_slots) : 0.0f;
    }
    rs.primary_rays = pd.raster ? rs.traced_primary_rays : pd.primary_rays;
    rs.shadow_rays = pd.shadow ? rs.primary_hits : 0;
    rs.kernel_launches = pd.launches;
    cudaEventElapsedTime(&rs.device_ms, ev_begin, ev_end);
    static const bool trace = getenv("RTB200_TRACE") != nullptr;       // per-launch CUDA-event times on stderr
    for (const TimedLaunch& tl : ctx->timed) {
        float ms = 0;
        cudaEventElapsedTime(&ms, tl.a, tl.b);
        if (trace) fprintf(stderr, "[rtb200] %s %.3f ms\n", tl.label ? tl.label : tl.stage == ST_PRIMARY ? "k_primary" : tl.stage == ST_COMPACT ? "k_compact" : tl.stage == ST_REFLECT ? "k_reflect" : tl.stage == ST_SHADE ? "k_shade" : "k_resolve", ms);
        if (tl.label) continue;
        if (tl.stage == ST_PRIMARY) rs.trace_primary_ms += ms;
        else if (tl.stage == ST_COMPACT) rs.compact_ms += ms;
        else if (tl.stage == ST_REFLECT) rs.reflect_ms += ms;
        else if (tl.stage == ST_SHADE) rs.shade_ms += ms;
        else rs.resolve_ms += ms;
    }
    if (trace && count && ctx->tune.packets) {
        for (int w = 0; w < 2; w++) {
            unsigned hist[16] = {0}, mx = 0;
            unsigned long long mns = 0, sns = 0, packets = 0;
            for (uint32_t c = 0; c < n_chunks; c++) {
                for (int b = 0; b < 16; b++) hist[b] += host_cnt[c].rounds_hist[w][b];
                mx = std::max(mx, host_cnt[c].max_rounds[w]);
                mns = std::max(mns, host_cnt[c].max_packet_ns[w]);
                sns += host_cnt[c].sum_packet_ns[w];
            }
            for (int b = 0; b < 16; b++) packets += hist[b];
            if (w) {
                unsigned long long ns = 0, ni[kItemPasses] = {0};
                for (uint32_t c = 0; c < n_chunks; c++) { ns += host_cnt[c].n_split; for (int p = 0; p < kItemPasses; p++) ni[p] += host_cnt[c].items_n[p]; }
                fprintf(stderr, "[rtb200] split shadow packets %llu, work items per pass:", ns);
                for (int p = 0; p < kItemPasses; p++) fprintf(stderr, " %llu", ni[p]);
                ns = 0;
                for (int p = 0; p < kItemPasses; p++) ni[p] = 0;
                for (uint32_t c = 0; c < n_chunks; c++) { ns += host_cnt[c].p_split; for (int p = 0; p < kItemPasses; p++) ni[p] += host_cnt[c].p_items_n[p]; }
                fprintf(stderr, "\n[rtb200] split primary packets %llu, work items per pass:", ns);
                for (int p = 0; p < kItemPasses; p++) fprintf(stderr, " %llu", ni[p]);
                fprintf(stderr, "\n");
            }
            fprintf(stderr, "[rtb200] %s packets %llu  max rounds %u  max packet %.3f ms  mean packet %.1f us  log2(rounds) histogram:",
                    w ? "shadow" : "primary", packets, mx, mns * 1e-6, packets ? sns * 1e-3 / packets : 0.0);
            for (int b = 0; b < 16; b++) fprintf(stderr, " %u", hist[b]);
            fprintf(stderr, "\n");
        }
    }
    if (stats) *stats = rs;
    if (overflow) return fail(ctx, RT_ERR_STATE, "traversal stack overflow (tree deeper than RT_MAX_TREE_DEPTH)");
    return RT_OK;
}

int rt_render_device(RtContext* ctx, const RtSettings* s, uint32_t* d_argb_out, int tile_size, int tile_mod, int tile_rem,
                     RtRenderStats* stats)
{
    if (int r = rt_render_device_begin(ctx, s, d_argb_out, tile_size, tile_mod, tile_rem)) return r;
    return rt_render_device_end(ctx, stats);
}

// Device frame -> the caller's pageable buffer.  The caller's buffer is ordinary memory (the adapter hands a std::vector,
// the GUI a QImage): a device-to-host copy straight into it is staged by the driver in small pieces.  Frames of a
// megapixel and more go through a pinned buffer of the context instead, in up to 8 slices: every slice's copy is enqueued
// behind the frame's kernels with an event, and while slice i+1 crosses PCIe the host threads move slice i into the
// caller's buffer.
static int frame_to_host(RtContext* ctx, const uint32_t* d_frame, uint32_t* host_out, size_t n)
{
    if (n == 0) return RT_OK;
    const bool staged = n >= ((size_t)1 << 20);
    if (staged && n > ctx->h_frame_cap) {
        if (ctx->h_frame) cudaFreeHost(ctx->h_frame);
        ctx->h_frame = nullptr; ctx->h_frame_cap = 0;
        if (cudaHostAlloc((void**)&ctx->h_frame, n * sizeof(uint32_t), cudaHostAllocDefault) == cudaSuccess) ctx->h_frame_cap = n;
        else { ctx->h_frame = nullptr; (void)cudaGetLastError(); }             // no pinned memory to be had: copy directly
    }
    if (!staged || !ctx->h_frame) {
        RT_CUDA(ctx, cudaMemcpyAsync(host_out, d_frame, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    }
    const int n_slices = (int)std::min<size_t>(8, std::max<size_t>(1, n >> 20));
    const size_t per = ((n + n_slices - 1) / n_slices + 1023) & ~(size_t)1023;
    for (int i = 0; i < n_slices; i++) {
        const size_t b = std::min(n, per * i), e = std::min(n, b + per);
        if (!ctx->copy_ev[i]) RT_CUDA(ctx, cudaEventCreateWithFlags(&ctx->copy_ev[i], cudaEventDisableTiming));
        if (e > b) RT_CUDA(ctx, cudaMemcpyAsync(ctx->h_frame + b, d_frame + b, (e - b) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        RT_CUDA(ctx, cudaEventRecord(ctx->copy_ev[i], ctx->stream));
    }
    for (int i = 0; i < n_slices; i++) {
        const size_t b = std::min(n, per * i), e = std::min(n, b + per);
        RT_CUDA(ctx, cudaEventSynchronize(ctx->copy_ev[i]));
        const long long chunks = (long long)((e - b + 65535) / 65536);
#pragma omp parallel for schedule(static)
        for (long long c = 0; c < chunks; c++) {
            const size_t cb = b + (size_t)c * 65536, ce = std::min(e, cb + 65536);
            memcpy(host_out + cb, ctx->h_frame + cb, (ce - cb) * sizeof(uint32_t));
        }
    }
    return RT_OK;
}

int rt_frame_to_host(RtContext* ctx, const uint32_t* d_frame, uint32_t* host_out, size_t n_pixels)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (n_pixels && (!d_frame || !host_out)) return fail(ctx, RT_ERR_INVALID, "NULL buffer");
    return frame_to_host(ctx, d_frame, host_out, n_pixels);
}

int rt_render(RtContext* ctx, const RtSettings* s, uint32_t* argb_out, RtRenderStats* stats)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (!argb_out) return fail(ctx, RT_ERR_INVALID, "argb_out is NULL");
    const size_t n = (size_t)s->image_width * s->image_height;
    RT_CUDA(ctx, ctx->d_frame.ensure(n));
    if (int r = rt_render_device_begin(ctx, s, ctx->d_frame.p, 64, 1, 0)) return r;
    const int rc = frame_to_host(ctx, ctx->d_frame.p, argb_out, n);           // enqueued behind the kernels; returns when argb_out is complete
    if (int r = rt_render_device_end(ctx, stats)) return r;
    return rc;
}

int rt_render_work_map(RtContext* ctx, const RtSettings* s, uint32_t* argb_out, RtPixelWork* work_out, RtRenderStats* stats)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (!work_out) return fail(ctx, RT_ERR_INVALID, "work_out is NULL");
    const size_t n = (size_t)s->image_width * s->image_height;
    RT_CUDA(ctx, ctx->d_frame.ensure(n));
    if (n > ctx->work_map_pixels) {
        if (ctx->d_work_map) RT_CUDA(ctx, cudaFree(ctx->d_work_map));
        ctx->d_work_map = nullptr;
        ctx->work_map_pixels = 0;
        RT_CUDA(ctx, cudaMalloc((void**)&ctx->d_work_map, n * sizeof(RtPixelWork)));
        ctx->work_map_pixels = n;
    }
    static_assert(sizeof(RtPixelWork) == 6 * sizeof(unsigned long long), "credit_work (kernels.cuh) addresses six words per pixel");
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_work_map, 0, n * sizeof(RtPixelWork), ctx->stream));
    ctx->frame_work_map = ctx->d_work_map;
    const int rb = rt_render_device_begin(ctx, s, ctx->d_frame.p, 64, 1, 0);
    ctx->frame_work_map = nullptr;                                              // only this frame: the next one is what it would have been
    if (rb) return rb;
    int rc = argb_out ? frame_to_host(ctx, ctx->d_frame.p, argb_out, n) : RT_OK;
    if (rc == RT_OK) {
        const cudaError_t e = cudaMemcpyAsync(work_out, ctx->d_work_map, n * sizeof(RtPixelWork), cudaMemcpyDeviceToHost, ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, RT_ERR_CUDA, "work map copy: %s", cudaGetErrorString(e));
    }
    if (int r = rt_render_device_end(ctx, stats)) return r;                    // waits for the stream: the map copy is complete
    return rc;
}

int rt_set_host_threads(int n)
{
    if (n <= 0) {
        cpu_set_t set;
        CPU_ZERO(&set);
        n = sched_getaffinity(0, sizeof(set), &set) == 0 ? CPU_COUNT(&set) : omp_get_num_procs();
    }
    omp_set_num_threads(std::max(1, n));
    return RT_OK;
}

// ---- frame buffers shared between the ranks of a box (CUDA IPC; see rtb200.h) ----------------------------------------
int rt_frame_alloc(RtContext* ctx, size_t bytes, void** d_ptr_out, unsigned char handle_out[RT_FRAME_HANDLE_BYTES])
{
    if (!ctx || !d_ptr_out || !handle_out) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    static_assert(sizeof(cudaIpcMemHandle_t) == RT_FRAME_HANDLE_BYTES, "handle size");
    void* p = nullptr;
    RT_CUDA(ctx, cudaMalloc(&p, std::max<size_t>(bytes, 4)));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(ctx, RT_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle_out, &h, sizeof(h));
    *d_ptr_out = p;
    return RT_OK;
}

int rt_frame_open(RtContext* ctx, const unsigned char handle[RT_FRAME_HANDLE_BYTES], void** d_ptr_out)
{
    if (!ctx || !handle || !d_ptr_out) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(ctx, RT_ERR_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e));
    }
    *d_ptr_out = p;
    return RT_OK;
}

int rt_frame_close(RtContext* ctx, void* d_ptr)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (!d_ptr) return RT_OK;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    RT_CUDA(ctx, cudaIpcCloseMemHandle(d_ptr));
    return RT_OK;
}

int rt_frame_free(RtContext* ctx, void* d_ptr)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (!d_ptr) return RT_OK;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    RT_CUDA(ctx, cudaFree(d_ptr));
    return RT_OK;
}

static int pack_unpack(RtContext* ctx, const RtSettings* s, const uint32_t* d_frame_in, uint32_t* d_frame_out, uint32_t* d_staging,
                       int tile_size, int tile_mod, int tile_rem, int unpack)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (int r = check_tile_args(ctx, tile_size, tile_mod, tile_rem)) return r;
    TileList* tl = nullptr;
    if (int r = get_tile_list(ctx, s, tile_size, tile_mod, tile_rem, &tl)) return r;
    if (tl->count == 0) return RT_OK;
    WorkView wk = {};
    wk.tiles = tl->d;
    wk.tile_begin = 0;
    wk.tile_end = tl->count;
    wk.tiles_x = tl->tiles_x;
    k_pack_tiles<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_frame_in, d_staging, wk, tile_size, s->image_width, s->image_height, unpack, d_frame_out);
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;                                                  // stream-ordered: no host synchronisation
}

int rt_pack_tiles(RtContext* ctx, const RtSettings* s, const uint32_t* d_frame, uint32_t* d_staging, int tile_size, int tile_mod, int tile_rem)
{
    return pack_unpack(ctx, s, d_frame, nullptr, d_staging, tile_size, tile_mod, tile_rem, 0);
}

int rt_unpack_tiles(RtContext* ctx, const RtSettings* s, uint32_t* d_frame, const uint32_t* d_staging, int tile_size, int tile_mod, int tile_rem)
{
    return pack_unpack(ctx, s, nullptr, d_frame, const_cast<uint32_t*>(d_staging), tile_size, tile_mod, tile_rem, 1);
}

int rt_unpack_gathered(RtContext* ctx, const RtSettings* s, uint32_t* d_frame, const uint32_t* d_gathered, int tile_size, int tile_mod, int self_rem)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (int r = check_tile_args(ctx, tile_size, tile_mod, self_rem < 0 ? 0 : self_rem)) return r;
    if (!d_frame || !d_gathered) return fail(ctx, RT_ERR_INVALID, "NULL buffer");
    TileList* tl = nullptr;
    if (int r = get_tile_list(ctx, s, tile_size, tile_mod, -1, &tl)) return r;
    if (tl->count == 0) return RT_OK;
    k_unpack_gathered<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_gathered, d_frame, tl->d, tl->count / (uint32_t)tile_mod, tile_mod, self_rem, tl->tiles_x,
                                                                  tile_size, s->image_width, s->image_height);
    RT_CUDA(ctx, cudaGetLastError());
    return RT_OK;
}

int rt_intersect(RtContext* ctx, const float* o3, const float* d3, size_t n, int32_t* tri_id, float* t, float* u, float* v)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (!ctx->bvh_valid) return fail(ctx, RT_ERR_STATE, "rt_build_bvh has not been called for the current triangles");
    if (n == 0) return RT_OK;
    if (!o3 || !d3) return fail(ctx, RT_ERR_INVALID, "ray arrays are NULL");
    cudaStream_t st = ctx->stream;
    RT_CUDA(ctx, ctx->b_a.ensure(3 * n)); RT_CUDA(ctx, ctx->b_b.ensure(3 * n));
    RT_CUDA(ctx, ctx->b_id.ensure(n)); RT_CUDA(ctx, ctx->b_t.ensure(n)); RT_CUDA(ctx, ctx->b_u.ensure(n)); RT_CUDA(ctx, ctx->b_v.ensure(n));
    RT_CUDA(ctx, ctx->d_flag.ensure(1));
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->b_a.p, o3, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->b_b.p, d3, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_flag.p, 0, sizeof(unsigned int), st));
    if (!ctx->grid_intersect) ctx->grid_intersect = grid_for(ctx, (const void*)k_intersect, kQueueThreads);
    int blocks = (int)std::min<size_t>((size_t)ctx->grid_intersect, (n + kQueueThreads - 1) / kQueueThreads);
    k_intersect<<<blocks, kQueueThreads, 0, st>>>(scene_view(ctx), ctx->b_a.p, ctx->b_b.p, n, ctx->d_orig.p, ctx->b_id.p, ctx->b_t.p, ctx->b_u.p,
                                                 ctx->b_v.p, ctx->d_flag.p);
    RT_CUDA(ctx, cudaGetLastError());
    unsigned int flag = 0;
    if (tri_id) RT_CUDA(ctx, cudaMemcpyAsync(tri_id, ctx->b_id.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (t) RT_CUDA(ctx, cudaMemcpyAsync(t, ctx->b_t.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (u) RT_CUDA(ctx, cudaMemcpyAsync(u, ctx->b_u.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (v) RT_CUDA(ctx, cudaMemcpyAsync(v, ctx->b_v.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag.p, sizeof(flag), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    if (flag) return fail(ctx, RT_ERR_STATE, "traversal stack overflow");
    return RT_OK;
}

int rt_occluded(RtContext* ctx, const float* p3, const float* n3, size_t n, uint8_t* occluded)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (!ctx->bvh_valid) return fail(ctx, RT_ERR_STATE, "rt_build_bvh has not been called for the current triangles");
    if (n == 0) return RT_OK;
    if (!p3 || !n3 || !occluded) return fail(ctx, RT_ERR_INVALID, "arrays are NULL");
    cudaStream_t st = ctx->stream;
    RT_CUDA(ctx, ctx->b_a.ensure(3 * n)); RT_CUDA(ctx, ctx->b_b.ensure(3 * n)); RT_CUDA(ctx, ctx->b_occ.ensure(n));
    RT_CUDA(ctx, ctx->d_flag.ensure(1));
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->b_a.p, p3, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->b_b.p, n3, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    RT_CUDA(ctx, cudaMemsetAsync(ctx->d_flag.p, 0, sizeof(unsigned int), st));
    if (!ctx->grid_occluded) ctx->grid_occluded = grid_for(ctx, (const void*)k_occluded, kQueueThreads);
    int blocks = (int)std::min<size_t>((size_t)ctx->grid_occluded, (n + kQueueThreads - 1) / kQueueThreads);
    k_occluded<<<blocks, kQueueThreads, 0, st>>>(scene_view(ctx), ctx->light, ctx->b_a.p, ctx->b_b.p, n, ctx->b_occ.p, ctx->d_flag.p);
    RT_CUDA(ctx, cudaGetLastError());
    unsigned int flag = 0;
    RT_CUDA(ctx, cudaMemcpyAsync(occluded, ctx->b_occ.p, n, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag.p, sizeof(flag), cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    if (flag) return fail(ctx, RT_ERR_STATE, "traversal stack overflow");
    return RT_OK;
}

int rt_generate_primary_rays(RtContext* ctx, const RtSettings* s, float* o3, float* d3)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (int r = validate_settings(ctx, s)) return r;
    if (!ctx->camera_set) return fail(ctx, RT_ERR_STATE, "rt_set_camera has not been called");
    if (!o3 || !d3) return fail(ctx, RT_ERR_INVALID, "arrays are NULL");
    FrameView fr = frame_view(ctx, s);
    size_t n = (size_t)fr.rw * fr.rh;
    RT_CUDA(ctx, ctx->b_a.ensure(3 * n)); RT_CUDA(ctx, ctx->b_b.ensure(3 * n));
    k_raygen<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(fr, ctx->b_a.p, ctx->b_b.p);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(o3, ctx->b_a.p, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(ctx, cudaMemcpyAsync(d3, ctx->b_b.p, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_resolve_ssaa(RtContext* ctx, const uint32_t* argb_in, int width, int height, int factor, uint32_t* argb_out)
{
    if (!ctx) return RT_ERR_INVALID;
    if (int r = bind(ctx)) return r;
    if (!argb_in || !argb_out || factor < 1 || width <= 0 || height <= 0) return fail(ctx, RT_ERR_INVALID, "bad resolve arguments");
    if (width % factor || height % factor) return fail(ctx, RT_ERR_INVALID, "image size not divisible by the factor (imageUtils.h:100-112)");
    const int w = width / factor, h = height / factor;
    RtSettings s;
    rt_default_settings(&s);
    s.image_width = w; s.image_height = h;
    const int tile = 64;
    TileList* tl = nullptr;
    if (int r = get_tile_list(ctx, &s, tile, 1, 0, &tl)) return r;
    RT_CUDA(ctx, ctx->d_super.ensure((size_t)width * height));
    RT_CUDA(ctx, ctx->d_frame.ensure((size_t)w * h));
    cudaStream_t st = ctx->stream;
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->d_super.p, argb_in, (size_t)width * height * 4, cudaMemcpyHostToDevice, st));
    WorkView wk = {};
    wk.tiles = tl->d; wk.tile_begin = 0; wk.tile_end = tl->count; wk.tiles_x = tl->tiles_x;
    k_resolve<<<ctx->sm_count * 8, 256, 0, st>>>(ctx->d_super.p, ctx->d_frame.p, wk, tile, factor, w, h, tl->count, 0u);
    RT_CUDA(ctx, cudaGetLastError());
    RT_CUDA(ctx, cudaMemcpyAsync(argb_out, ctx->d_frame.p, (size_t)w * h * 4, cudaMemcpyDeviceToHost, st));
    RT_CUDA(ctx, cudaStreamSynchronize(st));
    return RT_OK;
}

} // extern "C"
