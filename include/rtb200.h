/*
 * rtb200.h -- C ABI of the B200-native ray-tracing hot path (librtb200.so).
 *
 * This is the drop-in boundary for ONE path of TomClabault/RayTracerCPP: everything that sits behind
 * `Renderer::ray_trace()` / `Renderer::raster_trace()` + `Renderer::post_process()` (SSAO, SSAA), `BVH::BVH` and
 * `BVH::intersect()`, plus the OBJ / MTL loader that feeds it.
 * The reference has no FFI of its own; the seam is the public section of `class Renderer`
 * (tp2/projets/renderer/renderer.h:38-169) and `class BVH` (tp2/projets/bvh.h:302,307).  Each entry
 * point below names the reference member it replaces.  A header-only C++ adapter with the reference's
 * method names lives in `rtb200_renderer.hpp`; INTEGRATION.md shows how a maintainer swaps it in.
 *
 * Conventions
 *  - plain pointers and sizes only; all host buffers are caller-owned and copied during the call;
 *  - every function returns RT_OK (0) or a negative RtStatus; rt_last_error() gives the message;
 *  - a handle is bound to one CUDA device and is NOT thread-safe (one caller thread, like the
 *    reference's RenderThread, QT/mainWindowThreads.cpp:39-65);
 *  - there is no CPU fallback: without a usable CUDA device rt_create() fails with RT_ERR_CUDA.
 */
#ifndef RTB200_H
#define RTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct RtContext RtContext;

typedef enum RtStatus {
    RT_OK = 0,
    RT_ERR_INVALID = -1,      /* bad argument / unsupported setting            */
    RT_ERR_CUDA = -2,         /* CUDA runtime error (message in rt_last_error) */
    RT_ERR_STATE = -3,        /* call order (e.g. render before set_triangles) */
    RT_ERR_UNSUPPORTED = -4   /* a combination the path cannot serve (see rt_render) */
} RtStatus;

/* Blinn-Phong material: the fields of `Material` (tp2/src/materials.h:14-38) that the path reads. */
typedef struct RtMaterial {
    float ambient_coeff[3];
    float diffuse[3];
    float specular[3];
    float emission[3];
    float reflection;
    float roughness;
    float ns;
    float specular_threshold; /* set by MainWindow::precompute_materials, QT/mainwindow.cpp:240-249 */
} RtMaterial;

/* Shading modes: RenderSettings::ShadingMethod, tp2/projets/renderer/rendererSettings.h:8-26. */
enum {
    RT_SHADING = 0,
    RT_ABS_NORMALS_SHADING = 1,
    RT_PASTEL_NORMALS_SHADING = 2,
    RT_BARYCENTRIC_COORDINATES_SHADING = 3,
    RT_VISUALIZE_AO = 4
};

/* POD mirror of `RenderSettings` (tp2/projets/renderer/rendererSettings.h:6-105), same defaults via
 * rt_default_settings(). */
typedef struct RtSettings {
    int32_t image_width;
    int32_t image_height;
    int32_t enable_ssaa;
    int32_t ssaa_factor;
    int32_t hybrid_rasterization_tracing; /* 1: Renderer::raster_trace() instead of ray_trace() (renderer.cpp:869-1006): primary
                                             visibility by rasterisation + z-buffer, shading / shadow / reflection rays as before;
                                             needs rt_set_projection; whole frame on one GPU */
    int32_t shading_method;
    int32_t compute_shadows;
    int32_t max_recursion_depth;
    int32_t enable_bvh;                   /* must be 1 */
    int32_t bvh_max_depth;
    int32_t bvh_leaf_object_count;
    int32_t enable_ssao;                  /* screen-space ambient occlusion post-process (renderer.cpp:1229-1434), see rt_set_projection */
    int32_t enable_ambient;
    int32_t enable_diffuse;
    int32_t enable_specular;
    int32_t enable_emissive;
    int32_t rough_reflections_sample_count;
    int32_t enable_ao_mapping;
    int32_t enable_diffuse_mapping;
    int32_t enable_normal_mapping;
    int32_t enable_displacement_mapping;  /* parallax occlusion mapping, renderer.cpp:518-554,567-568 */
    int32_t enable_roughness_mapping;
    int32_t enable_skysphere;
    int32_t enable_skybox;                /* cube-map miss shader (Skybox::sample, skybox.cpp:12-51); the skysphere wins */
    /* Seed of the per-pixel xorshift32 streams used by rough reflections.  The reference owns one
     * generator per OpenMP thread seeded from std::rand() (renderer.cpp:51-61), which is not
     * reproducible; the shared stream is state(px,py) = rt_pixel_seed(py*W'+px, rng_seed). */
    uint32_t rng_seed;
    /* RenderSettings::displacement_mapping_strength / parallax_mapping_steps, rendererSettings.h:94-95 (0.02, 32). */
    float displacement_mapping_strength;
    int32_t parallax_mapping_steps;
    /* RenderSettings::ssao_sample_count / ssao_radius / ssao_amount, rendererSettings.h:69-73 (64, 0.5, 1.0). */
    int32_t ssao_sample_count;
    float ssao_radius;
    float ssao_amount;
    /* RenderSettings::enable_clipping, rendererSettings.h:40 (true): hybrid_rasterization_tracing clips every triangle against
     * the six planes of the view volume in clip space (renderer.cpp:837-853) before it is rasterised. */
    int32_t enable_clipping;
} RtSettings;

/* Texture slots: Renderer::set_{ao,diffuse,normal,roughness}_map / set_skysphere / set_skybox, renderer.cpp:194-201.
 * The six faces of the cube-map skybox are six slots, in the order of Skybox::Skybox(const Image faces[6])
 * (renderer/skybox.h:13-17): right, left, top, bottom, back, front. */
enum {
    RT_TEX_AO = 0,
    RT_TEX_DIFFUSE = 1,
    RT_TEX_NORMAL = 2,
    RT_TEX_ROUGHNESS = 3,
    RT_TEX_SKYSPHERE = 4,
    RT_TEX_SKYBOX_RIGHT = 5,
    RT_TEX_SKYBOX_LEFT = 6,
    RT_TEX_SKYBOX_TOP = 7,
    RT_TEX_SKYBOX_BOTTOM = 8,
    RT_TEX_SKYBOX_BACK = 9,
    RT_TEX_SKYBOX_FRONT = 10,
    RT_TEX_DISPLACEMENT = 11, /* Renderer::set_displacement_map: the depth map of parallax occlusion mapping (.r) */
    RT_TEX_COUNT = 12
};

/* Per-render counters (rays actually traced + what the pipeline did). */
typedef struct RtRenderStats {
    uint64_t primary_rays;
    uint64_t shadow_rays;      /* depth-0 shadow rays                                       */
    uint64_t reflection_rays;  /* closest-hit rays of reflection fans (all depths)          */
    uint64_t reflection_shadow_rays;
    uint64_t primary_hits;
    uint32_t kernel_launches;  /* launches of this library's kernels during the call        */
    float    device_ms;        /* CUDA-event time of the kernels (excludes the D2H copy)    */
    float    trace_primary_ms; /* per-stage CUDA-event times, summed over chunks            */
    float    shade_ms;
    float    reflect_ms;
    float    compact_ms;       /* ordered compaction of the hit records into the ray queues */
    float    resolve_ms;
    /* Filled only when RT_OPT_COUNT_WORK is on (instrumented kernel instantiations, never the timed ones):
     * 7-slab volume tests and ray/triangle tests the traversal performed, per ray class -- the V and T of
     * the bytes-per-ray metric 56*V + 36*T (DESIGN.md).  Reflection = fan rays and their shadow rays. */
    uint64_t primary_volume_tests, primary_triangle_tests;
    uint64_t shadow_volume_tests, shadow_triangle_tests;
    uint64_t reflection_volume_tests, reflection_triangle_tests;
    /* Primary rays that were really traced: `primary_rays` counts every sample of the frame, also those of tiles and
     * packets outside the screen-space bound of the scene, which are written as misses without a ray (RT_OPT_SCREEN_CULL).
     * Always filled. */
    uint64_t traced_primary_rays;
    /* RT_OPT_COUNT_WORK only: bytes of child records (64 each) and triangles (48 each) the kernels fetched for the tests
     * above.  A 32-ray packet fetches a record once per warp and tests it in every lane; a single ray fetches per test. */
    uint64_t primary_fetched_bytes, shadow_fetched_bytes, reflection_fetched_bytes;
} RtRenderStats;

/* Flattened-tree facts, for tests and DESIGN.md (the reference tree has the same node/leaf counts). */
typedef struct RtBvhInfo {
    uint64_t triangles;
    uint64_t nodes;            /* all octree cells, empty leaves included (bvh.h:153-167)   */
    uint64_t leaves;
    uint64_t empty_leaves;
    uint64_t interior;
    uint32_t max_depth_reached;
    uint32_t max_leaf_size;
    uint64_t child_records;    /* 64-byte slab records resident in HBM                      */
    uint64_t device_bytes;     /* records + triangles + shading side arrays                 */
    double   build_ms;         /* host octree build + flatten                               */
    double   upload_ms;
} RtBvhInfo;

void rt_default_settings(RtSettings* s);
uint32_t rt_pixel_seed(uint32_t pixel_index, uint32_t rng_seed);

/* Renderer::Renderer() -- renderer.cpp:80.  `device` is a CUDA ordinal. */
int rt_create(int device, RtContext** out);
void rt_destroy(RtContext* ctx);
const char* rt_last_error(const RtContext* ctx); /* ctx may be NULL for rt_create failures */

/* Library knobs (no reference counterpart). */
enum {
    RT_OPT_COUNT_WORK = 0,    /* 1: run the instrumented kernels and fill the *_tests counters of RtRenderStats */
    RT_OPT_CHUNK_PIXELS = 1,  /* supersampled pixels per wavefront chunk (bounds ray-queue memory)             */
    RT_OPT_REFILL_PRIMARY = 3,/* a warp of k_primary / k_shade fetches new rays once this many of its 32 lanes are idle  */
    RT_OPT_REFILL_SHADE = 4,  /* (default 16)                                                                          */
    RT_OPT_TRI_BATCH = 5,     /* a warp runs a round of triangle tests once this many lanes wait for one (default 8)   */
    RT_OPT_PACKETS = 6,       /* 1 (default): primary and shadow rays are traced as 32-ray packets (one traversal per
                                 warp); 0: every lane runs its own traversal state machine with lane refill.  Results do
                                 not depend on it                                                                       */
    /* Round budgets of the 32-ray packets.  A packet that needs more cell/leaf rounds than its budget is SPLIT: each cell
       it has not visited becomes a work item that another warp traces for the same 32 rays (items can be split again, 6
       generations deep, the last without a limit); answers are merged (shadow: OR, primary: 64-bit atomicMin on
       (t, original index)).  n > 0: n rounds; 0: never split; n < 0 (the defaults): adaptive -- split after 8 |n| rounds
       at the latest, and after |n| / 4 rounds (items: |n|) as soon as the launch's queue has been handed out completely,
       i.e. when the packet has become the tail of its launch and other warps are free to take its cells.  Results do not
       depend on any of them. */
    RT_OPT_PACKET_ROUNDS = 7, /* shadow packets (default -256)                                                           */
    RT_OPT_PRIMARY_ROUNDS = 11,/* primary packets (default -256; negative additionally means: not split in long launches,
                                 256 and more packets per resident warp)                                                  */
    RT_OPT_ITEM_ROUNDS = 10,  /* work items of all generations but the last (default -16; 0 is invalid)                 */
    RT_OPT_ITEM_PASSES = 16,  /* generations of work items per stage = launches of the item kernels (1..6, default 6)        */
    RT_OPT_FUSED_ITEMS = 12,  /* 0 (default): the work items of split packets are traced generation by generation in separate
                                 launches (six item passes and a finish kernel per stage); 1: the packet kernels consume the
                                 items themselves through 32 ticket queues, the last item of a record stores its pixels -- one
                                 launch per stage, but items of a record run concurrently and prune each other less: measured
                                 slower on B200 (DESIGN.md), kept for experiments.  Results do not depend on it             */
    RT_OPT_TOP_TABLE = 13,    /* 1: every CTA of the packet kernels loads the child blocks of the first tree levels (<= 72 records,
                                 4.6 KB) into shared memory with one bulk asynchronous copy (cp.async.bulk + mbarrier) and takes
                                 those cells from there instead of fetching them; 0 (default): they are fetched like any other
                                 cell -- they never leave the L1, and the extra address select costs 2 % of the frame on B200
                                 (measured, DESIGN.md).  Results do not depend on it                                       */
    RT_OPT_DEVICE_BUILD = 15, /* 1 (default): rt_build_bvh / rt_transform_triangles build the octree ON THE GPU (per-triangle path
                                 through the reference's subdivision -> stable radix sort -> cells level by level): same cells,
                                 leaf contents and order, slab extents and rt_bvh_info statistics as the host builder, hence as
                                 the reference's BVH::BVH; the caller's arrays stay resident, so a transform + rebuild moves no
                                 triangle data.  0: the host builder (C++/OpenMP) + upload.  Results do not depend on it  */
    RT_OPT_SHADOW_SORT = 14,  /* before the shadow packets are formed the hit queue is put in LIGHT-SPACE order (Morton code of
                                 the hit point's direction from the light, one counting sort), so a packet's 32 shadow rays run
                                 through the same cells whatever the depth of their hits.  0: never (queue order = pixel order);
                                 1: always; 2 (default): when fewer than a quarter of a chunk's ray slots are hits -- sparse
                                 hits (thin strands) lie at unrelated depths, whereas the neighbouring pixels of a closed
                                 surface already are neighbours from the light (measured: hair scene shadow stage 18.0 ->
                                 6.8 ms with it, 10 M-triangle sphere 7.3 -> 9.6 ms).  Not used with reflection fans.
                                 Results do not depend on it                                                              */
    RT_OPT_SCREEN_CULL = 8,   /* 1 (default): primary packets whose 8x4 sample block no ray can take into the boxes of the
                                 tree's upper levels, and tiles of only such blocks, are written as misses without
                                 tracing.  Results do not depend on it                                                  */
    RT_OPT_LANES = 9,         /* wavefront chunks in flight at a time, each on its own stream with its own queues, so one
                                 chunk's kernels fill the SMs the others leave idle while their longest packets finish; the
                                 per-stage times of RtRenderStats then overlap.  0: one chunk at a time; 1 (default): 2 chunks;
                                 n in [2,6]: n chunks.  Results do not depend on it                                     */
    RT_OPT_PACKET_CULL = 19,  /* bounding-pyramid cull of the packet kernels: the rays of a packet leave from (primary: the camera) or
                                 arrive at (shadow: the point light) one point, so they lie in a thin pyramid; the children of a cell
                                 whose boxes lie outside one of its four side planes are dropped in one pass, 4 lanes per child, before
                                 the per-ray slab tests.  Bit 0: primary packets, bit 1: shadow packets (default 3).  Results do not
                                 depend on it                                                                                 */
    RT_OPT_FAN_LANES = 20,    /* 1 (default): with max_recursion_depth 1 and no normal mapping a rough-reflection fan runs with one LANE
                                 per fan ray (k_reflect_fan: the stream offsets and the stale hit record of the reference's sequential
                                 walk are found as a fixed point); 0: one thread walks the fan (k_reflect).  Results do not depend on it */
    RT_OPT_GRAPH = 18,        /* 1 (default): a frame whose launch sequence equals the previous frame's (same settings, camera, light,
                                 buffers, options) is captured as a CUDA graph and replayed with one cudaGraphLaunch from then on;
                                 the per-stage times of RtRenderStats are 0 for such frames.  0: every frame is enqueued launch by
                                 launch.  Results do not depend on it                                                       */
    RT_OPT_RASTER_UNITS = 17, /* hybrid raster path: first size of the list of work units (row bands of the pieces too large for one
                                 thread); a frame that needs more grows the list and repeats its depth pass.  Default 2^18       */
    RT_OPT_LIGHT_CULL = 21,   /* 1 (default): shadow packets skip the triangles, and the subtrees holding only triangles, that have the
                                 point light strictly on their front side: back-face culling rejects every crossing of such a triangle
                                 on the way to the light.  Per-light masks, rebuilt at the first frame after the light, the tree or
                                 this option changes.  0: masks with every bit set.  Results do not depend on it            */
    RT_OPT_LEAF_SPLIT = 2     /* n > 0 (default 8): when flattening, octree leaves with more than n triangles get a
                                 device-side median-split sub-hierarchy of groups of <= n triangles; 0 = flatten the
                                 reference's cells and leaves exactly as they are.  Applies to the next rt_build_bvh.
                                 Results do not depend on it (tests/test_gpu_parity.py)                               */
};
int rt_set_option(RtContext* ctx, int option, int64_t value);
/* Threads the library's host-side loops may use (octree build, the copy into the caller's frame buffer): OpenMP's
 * omp_set_num_threads for this process.  A launcher that exports OMP_NUM_THREADS=1 for every rank (torchrun does) would
 * otherwise serialise rt_build_bvh.  n <= 0: all the cores this process may run on. */
int rt_set_host_threads(int n);
/* Run all of the context's work on the caller's CUDA stream (a cudaStream_t; NULL = back to the context's own
 * non-blocking stream), so a host that already orders work on a stream -- or times it with events -- can do so. */
int rt_set_stream(RtContext* ctx, void* cuda_stream);

/* Renderer::set_triangles(const std::vector<Triangle>&) -- renderer.cpp:137-144.
 * xyz9: n*9 floats (a,b,c); uv6: n*6 floats (u_a,u_b,u_c,v_a,v_b,v_c) as Triangle::_tex_coords_u/_v
 * (triangle.h:99-103) or NULL for the default (-1,-1,-1); mat: n material indices or NULL (-1).
 * Does not build the tree: rt_build_bvh() is separate, as reconstruct_bvh_new() is in the reference. */
int rt_set_triangles(RtContext* ctx, const float* xyz9, const float* uv6, const int32_t* mat, size_t n);

/* BVH::BVH(std::vector<Triangle>*, int max_depth, int leaf_max_obj_count) -- bvh.cpp:19-43;
 * Renderer::reconstruct_bvh_new -- renderer.cpp:243-246.  Builds the same octree as the reference's
 * sequential insertion, flattens it, uploads it. */
int rt_build_bvh(RtContext* ctx, int max_depth, int leaf_max_obj_count);
int rt_bvh_info(const RtContext* ctx, RtBvhInfo* out);

/* Renderer::set_object_transform(const Transform&) -- renderer.cpp:214-224: re-transforms every triangle
 * by `m` (row-major 4x4, applied as Transform::operator()(Point), mat.cpp:83-100) and rebuilds the tree.
 * The caller composes object_transform * previous^-1 exactly as the reference does. */
int rt_transform_triangles(RtContext* ctx, const float m[16], int max_depth, int leaf_max_obj_count);

/* ---- load -> upload: Wavefront OBJ + MTL (host side, csrc/scene_io.cpp) --------------------------------------------------
 * rt_obj_load = read_meshio_data(path) (tp2/src/mesh_io.cpp:426-591, with read_materials_mtl :213-304) followed by
 * MeshIOUtils::create_triangles(data, current_material_count, transform) (tp2/projets/utils/meshIOUtils.cpp:4-33): what
 * MainWindow::load_obj does before Renderer::set_triangles (QT/mainwindow.cpp:251-282).  The arrays of the returned mesh have
 * the layout rt_set_triangles / rt_set_materials take: a maintainer's load_obj becomes rt_obj_load -> (edit the materials) ->
 * rt_precompute_materials -> rt_set_triangles -> rt_set_materials.  transform: row-major 4x4 or NULL (identity).
 * err (may be NULL): receives the message when the call fails (RT_ERR_INVALID: file missing, parse error, no geometry). */
typedef struct RtObjMesh RtObjMesh;
int rt_obj_load(const char* path, const float transform[16], int32_t current_material_count, RtObjMesh** out, char* err, size_t err_cap);
void rt_obj_free(RtObjMesh* mesh);
size_t rt_obj_triangle_count(const RtObjMesh* mesh);
size_t rt_obj_material_count(const RtObjMesh* mesh);             /* materials of the .mtl (+ "default" when a face needed it)  */
const float* rt_obj_xyz9(const RtObjMesh* mesh);
const float* rt_obj_uv6(const RtObjMesh* mesh);                  /* NULL when the file has no texture coordinates              */
const int32_t* rt_obj_material_indices(const RtObjMesh* mesh);   /* already offset by current_material_count                   */
const RtMaterial* rt_obj_materials(const RtObjMesh* mesh);       /* specular_threshold = 0 until rt_precompute_materials       */
const char* rt_obj_material_name(const RtObjMesh* mesh, size_t i);
/* MainWindow::precompute_materials -- QT/mainwindow.cpp:240-249: specular_threshold = pow(1e-3 / luminance(specular), 1 / ns),
 * in the reference's mixed float / double arithmetic. */
void rt_precompute_materials(RtMaterial* mats, size_t n);

/* Renderer::set_materials / get_materials().materials -- renderer.cpp:150-152. */
int rt_set_materials(RtContext* ctx, const RtMaterial* mats, size_t n);

/* Renderer::add_analytic_shape(Sphere(center, radius, mat_index)) / (Plane(point, normal, mat_index)) -- renderer.cpp:146,
 * analyticShape.h:22-55; rt_clear_analytic_shapes: the shapes half of Renderer::clear_geometry (renderer.cpp:182-186).
 * Shapes are tested after the BVH, in the order they were added, by trace_ray (renderer.cpp:1029-1037) and is_shadowed
 * (:376-397).  A frame with shapes refuses the texture-mapping switches and the barycentric / AO debug modes: the
 * reference reads HitInfo::triangle there, which a shape hit leaves stale or null.  `normal` is used as given
 * (the reference expects it normalised). */
int rt_add_sphere(RtContext* ctx, const float center[3], float radius, int32_t mat_index);
int rt_add_plane(RtContext* ctx, const float point[3], const float normal[3], int32_t mat_index);
int rt_clear_analytic_shapes(RtContext* ctx);

/* Renderer::set_*_map(const Image&) / set_skysphere -- renderer.cpp:194-201.  Texels are RGBA, row 0 first
 * (no Y flip, QT/mainwindow.cpp:285).  f32 is the reference's `Image` storage; u8 is the on-disk form,
 * decoded on the device as u8 * (1/255.f) exactly like read_image (image_io.cpp:115-121). */
int rt_set_texture_f32(RtContext* ctx, int slot, const float* rgba, int width, int height);
int rt_set_texture_u8(RtContext* ctx, int slot, const uint8_t* rgba, int width, int height);
int rt_clear_texture(RtContext* ctx, int slot); /* Renderer::clear_*_map -- renderer.cpp:203-207 */

/* Camera state: Camera::_perspective_proj_mat_inv, _camera_to_world_mat, _position
 * (scene/camera.h:9-33; set by change_camera_fov/aspect_ratio + set_camera_transform, renderer.cpp:189-233).
 * Matrices are row-major (Transform::m[row][col], mat.h). */
int rt_set_camera(RtContext* ctx, const float proj_inv[16], const float cam_to_world[16], const float position[3]);
/* Host helpers with the reference's float arithmetic, for callers that hold (fov, aspect) or a transform rather
 * than the derived matrices: Perspective(fov, aspect, znear, zfar).inverse() (mat.cpp:307-319,378-447; the
 * reference's Camera uses znear 0.1, zfar 1000, scene/camera.h:11) and Transform::inverse().  Row-major. */
void rt_perspective_inverse(float fov, float aspect, float znear, float zfar, float proj_inv_out[16]);
void rt_invert_transform(const float m[16], float out[16]);
/* Transform::operator()(const Point&) -- mat.cpp:83-100 (e.g. Camera::_position = transform(Point(0,0,0))). */
void rt_transform_point(const float m[16], const float p[3], float out[3]);

/* Camera::_perspective_proj_mat, _fov, _aspect_ratio (scene/camera.cpp:5-19): what Renderer::post_process_ssao_SIMD reads
 * (renderer.cpp:1249,1283-1326).  Needed only with RtSettings::enable_ssao; the matrix is Perspective(fov, aspect, znear,
 * zfar) in the reference's float arithmetic (mat.cpp:307-319).  fov in degrees. */
int rt_set_projection(RtContext* ctx, float fov, float aspect, float znear, float zfar);

/* Renderer::set_light_position -- renderer.cpp:191. */
int rt_set_light(RtContext* ctx, const float position[3]);

/* Renderer::ray_trace() + Renderer::post_process() -- renderer.cpp:1068-1135 (what render() times,
 * utils/mainUtils.cpp:6-21).  argb_out: image_width*image_height ARGB32 words, row 0 = bottom row, exactly
 * the layout of Renderer::get_image() (renderer.cpp:1086).  Host pointer; includes the D2H copy. */
int rt_render(RtContext* ctx, const RtSettings* settings, uint32_t* argb_out, RtRenderStats* stats);

/* Same frame, result left in device memory (`d_argb_out` is a device pointer on the context's device).
 * Tile sharding for the multi-GPU path: the frame is cut into tile_size x tile_size final-resolution
 * tiles; this call renders only tiles with (tile_index % tile_mod) == tile_rem (tile_mod = 1 -> all)
 * and leaves the other pixels of d_argb_out untouched. */
int rt_render_device(RtContext* ctx, const RtSettings* settings, uint32_t* d_argb_out,
                     int tile_size, int tile_mod, int tile_rem, RtRenderStats* stats);

/* The same call in two halves, for hosts that put more work (pack, a collective, unpack, a copy) on the context's stream
 * behind the frame without a host synchronisation in between: _begin enqueues every kernel of the frame and returns;
 * _end waits for the stream, fills `stats` (may be NULL) and reports device-side errors.  One frame at a time. */
int rt_render_device_begin(RtContext* ctx, const RtSettings* settings, uint32_t* d_argb_out,
                           int tile_size, int tile_mod, int tile_rem);
int rt_render_device_end(RtContext* ctx, RtRenderStats* stats);

/* ---- Frame buffers shared between the ranks of one box (one process per GPU) -------------------------------------------
 * The gather of the sharded frame is fused into the kernels that produce the pixels: rank 0 allocates the frame with
 * rt_frame_alloc and hands the 64-byte handle to its peers (any byte transport: the Python side uses torch.distributed);
 * a peer maps it with rt_frame_open and passes the mapped pointer as `d_argb_out` of rt_render_device_begin -- its resolve
 * (or shading) kernel then stores the final pixels of its tiles straight into rank 0's memory over NVLink.  No pack, no
 * collective, no unpack; the only cross-rank step left is one barrier per frame, which the host enqueues.
 * (CUDA IPC: cudaIpcGetMemHandle / cudaIpcOpenMemHandle with peer access.)  rt_frame_close unmaps, rt_frame_free frees. */
#define RT_FRAME_HANDLE_BYTES 64
int rt_frame_alloc(RtContext* ctx, size_t bytes, void** d_ptr_out, unsigned char handle_out[RT_FRAME_HANDLE_BYTES]);
int rt_frame_open(RtContext* ctx, const unsigned char handle[RT_FRAME_HANDLE_BYTES], void** d_ptr_out);
int rt_frame_close(RtContext* ctx, void* d_ptr);
int rt_frame_free(RtContext* ctx, void* d_ptr);

/* The last step of rt_render for a frame that already is (or is about to be, in stream order) in device memory: copies
 * n_pixels ARGB32 words from d_frame to the caller's ordinary (pageable) host buffer, behind everything enqueued on the
 * context's stream so far, and returns when host_out is complete.  The copy runs in slices through a pinned staging
 * buffer; while one slice crosses PCIe the previous one is moved into host_out by the host threads. */
int rt_frame_to_host(RtContext* ctx, const uint32_t* d_frame, uint32_t* host_out, size_t n_pixels);

/* Pack / unpack the tiles owned by (tile_mod, tile_rem) between the row-major frame and a tile-major
 * staging buffer -- the operand of the framebuffer all-gather.  rt_tile_count gives how many tiles the
 * shard owns; every tile occupies tile_size*tile_size words in the staging buffer (edge tiles padded). */
int rt_tile_count(const RtSettings* settings, int tile_size, int tile_mod, int tile_rem);
int rt_pack_tiles(RtContext* ctx, const RtSettings* settings, const uint32_t* d_frame, uint32_t* d_staging,
                  int tile_size, int tile_mod, int tile_rem);
int rt_unpack_tiles(RtContext* ctx, const RtSettings* settings, uint32_t* d_frame, const uint32_t* d_staging,
                    int tile_size, int tile_mod, int tile_rem);

/* The receiving side of the all-gather in one launch: d_gathered holds the staging buffers of all tile_mod shards
 * back to back, each max_r(rt_tile_count(r)) * tile_size^2 words; the tiles of every shard but self_rem are
 * written into d_frame (self_rem = -1: all shards).  Stream-ordered like rt_pack_tiles (no host synchronisation). */
int rt_unpack_gathered(RtContext* ctx, const RtSettings* settings, uint32_t* d_frame, const uint32_t* d_gathered,
                       int tile_size, int tile_mod, int self_rem);

/* Batched bool BVH::intersect(const Ray&, HitInfo&) const -- bvh.h:307, bvh.cpp:68-71.
 * o3/d3: n*3 floats.  Outputs (any may be NULL): tri_id = index into the rt_set_triangles array or -1
 * (HitInfo::triangle - triangles.data()), t/u/v = HitInfo::t,u,v (hitInfo.h:8-29; t = -1 on a miss). */
int rt_intersect(RtContext* ctx, const float* o3, const float* d3, size_t n,
                 int32_t* tri_id, float* t, float* u, float* v);

/* Batched Renderer::is_shadowed -- renderer.cpp:340-402.  p3 = inter_point, n3 = shading normal,
 * light = the context's light.  occluded[i] = 1 iff the reference returns true (BVH, then the analytic shapes).
 * rt_intersect above is BVH::intersect alone: the shapes are Renderer state, not part of the BVH. */
int rt_occluded(RtContext* ctx, const float* p3, const float* n3, size_t n, uint8_t* occluded);

/* Primary-ray generation only (renderer.cpp:1083-1098) for the supersampled frame of `settings`:
 * o3/d3 receive (W*f)*(H*f)*3 floats, pixel-major, row 0 = bottom row.  For parity tests. */
int rt_generate_primary_rays(RtContext* ctx, const RtSettings* settings, float* o3, float* d3);

/* Quantise + SSAA resolve only (imageUtils.h:98-152) on a host ARGB32 image; for parity tests. */
int rt_resolve_ssaa(RtContext* ctx, const uint32_t* argb_in, int width, int height, int factor, uint32_t* argb_out);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
