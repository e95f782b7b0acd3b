// raster.cuh -- Renderer::raster_trace (tp2/projets/renderer/renderer.cpp:869-1006) as CUDA kernels: the hybrid path
// (RenderSettings::hybrid_rasterization_tracing), SURVEY.md section 8(f)4.  The arithmetic is raster_device.h's; this file
// is the scheduling.
//
//   k_raster_tris<EMIT>   one thread per triangle (leaf order; the reference's order is carried in the z-key): clip, set up
//                         every piece, rasterise the pieces whose bounding box holds at most kRasterSmallArea pixels right
//                         there; a larger piece is cut into bands of kRasterBandRows rows, one work unit each (cover pass)
//   k_raster_units<EMIT>  one CTA per unit: the piece's pixel-point sequences (image_x += increment, renderer.cpp:926-937)
//                         are one dependent chain of float additions each, so two threads lay them out in shared memory
//                         once and the CTA's threads then test the band's pixels independently
//   k_raster_shade        one thread per pixel: the winner's piece is re-derived from the key and shaded (shadow ray and
//                         reflection fan through the octree with the single-ray traversal of rt_device.h); uncovered
//                         pixels get the colour of clear_image(); with SSAO the G-buffers are the reference's
//                         (z = the fragment's depth, normal = the ORIGINAL triangle's un-normalised normal)
// EMIT = false: depth pass, atomicMin on the 64-bit z-keys.  EMIT = true: the same walk again; the fragment that owns a
// pixel's key stores its pixel point.  SSAO and the SSAA resolve follow as for ray_trace() (ssao.cuh, k_resolve).
#pragma once

#include <cuda_runtime.h>
#include "raster_device.h"
#include "kernels.cuh"

namespace rtb {

constexpr int kRasterSmallArea = 1024;       // bounding-box pixels a triangle's own thread still walks
constexpr int kRasterBandRows = 16;          // rows per work unit of a larger piece
constexpr int kRasterUnitThreads = 256;

struct RasterUnit {
    uint32_t tri;                            // leaf-order triangle
    uint32_t piece_band;                     // piece | band << 4
};

struct RasterBuffers {
    unsigned long long* keys;                // per pixel of the supersampled frame
    float2* frag_xy;                         // per pixel: the winner's pixel point
    RasterUnit* units;
    unsigned int* n_units;                   // units written (may exceed unit_cap: the host then grows the list and repeats the pass)
    uint32_t unit_cap;
};

template <bool EMIT>
RT_DEV void raster_visit(const RasterBuffers& rb, size_t pix, unsigned long long key, float ppx, float ppy)
{
    if (!EMIT) atomicMin(rb.keys + pix, key);
    else if (rb.keys[pix] == key) rb.frag_xy[pix] = make_float2(ppx, ppy);
}

template <bool EMIT>
__global__ void __launch_bounds__(128)
k_raster_tris(SceneView sc, FrameView fr, RasterView rv, RasterBuffers rb)
{
    const float sx = raster_scale(fr.rw), sy = raster_scale(fr.rh);
    for (uint32_t tri = blockIdx.x * blockDim.x + threadIdx.x; tri < sc.n_tris; tri += gridDim.x * blockDim.x) {
        const RasterSource src = raster_source(sc, tri);
        Tri4 scratch[RT_CLIP_MAX], clipped[RT_CLIP_MAX];
        const int n_pieces = raster_clip(rv, src.a, src.b, src.c, src.tu, src.tv, scratch, clipped);
        for (int pi = 0; pi < n_pieces; pi++) {
            const RasterPiece pc = raster_piece(fr, clipped[pi]);
            if (pc.max_x < pc.min_x || pc.max_y < pc.min_y) continue;
            const long long area = (long long)(pc.max_x - pc.min_x + 1) * (long long)(pc.max_y - pc.min_y + 1);
            if (area > kRasterSmallArea) {
                if (!EMIT) {
                    const uint32_t bands = (uint32_t)(pc.max_y - pc.min_y + kRasterBandRows) / (uint32_t)kRasterBandRows;
                    const uint32_t at = atomicAdd(rb.n_units, bands);
                    for (uint32_t b = 0; b < bands && at + b < rb.unit_cap; b++) {
                        RasterUnit u;
                        u.tri = tri; u.piece_band = (uint32_t)pi | (b << 4);
                        rb.units[at + b] = u;
                    }
                }
                continue;
            }
            const uint32_t order = (uint32_t)src.orig * 16u + (uint32_t)pi;
            float image_y = raster_start(pc.min_y, sy);
            for (int py = pc.min_y; py <= pc.max_y; py++, image_y += sy) {
                float image_x = raster_start(pc.min_x, sx);
                for (int px = pc.min_x; px <= pc.max_x; px++, image_x += sx) {
                    float ppx, ppy, u, v, w, z;
                    if (!raster_fragment(pc, image_x, image_y, sx, sy, ppx, ppy, u, v, w, z)) continue;
                    unsigned long long key;
                    if (!raster_key(z, order, key)) continue;
                    raster_visit<EMIT>(rb, (size_t)py * fr.rw + px, key, ppx, ppy);
                }
            }
        }
    }
}

// Dynamic shared memory: (columns of the widest possible piece = fr.rw) + kRasterBandRows floats.
template <bool EMIT>
__global__ void __launch_bounds__(kRasterUnitThreads)
k_raster_units(SceneView sc, FrameView fr, RasterView rv, RasterBuffers rb)
{
    extern __shared__ float seq[];                           // xs[0 .. width), then ys[0 .. kRasterBandRows)
    __shared__ RasterPiece s_piece;
    __shared__ uint32_t s_order;
    const uint32_t n_units = min(*rb.n_units, rb.unit_cap);
    const float sx = raster_scale(fr.rw), sy = raster_scale(fr.rh);
    float* xs = seq;
    float* ys = seq + fr.rw;
    for (uint32_t ui = blockIdx.x; ui < n_units; ui += gridDim.x) {
        const RasterUnit unit = rb.units[ui];
        const int band = (int)(unit.piece_band >> 4);
        __syncthreads();                                     // the previous unit's tables are no longer read
        if (threadIdx.x == 0) {
            const RasterSource src = raster_source(sc, unit.tri);
            Tri4 scratch[RT_CLIP_MAX], clipped[RT_CLIP_MAX];
            raster_clip(rv, src.a, src.b, src.c, src.tu, src.tv, scratch, clipped);
            s_piece = raster_piece(fr, clipped[unit.piece_band & 15u]);
            s_order = (uint32_t)src.orig * 16u + (unit.piece_band & 15u);
        }
        __syncthreads();
        const RasterPiece pc = s_piece;
        const int width = pc.max_x - pc.min_x + 1;
        const int y0 = pc.min_y + band * kRasterBandRows;
        const int rows = min(kRasterBandRows, pc.max_y - y0 + 1);
        if (threadIdx.x == 0) {
            float image_x = raster_start(pc.min_x, sx);
            for (int i = 0; i < width; i++, image_x += sx) xs[i] = image_x;
        } else if (threadIdx.x == 32) {
            float image_y = raster_start(pc.min_y, sy);
            for (int py = pc.min_y; py < y0; py++) image_y += sy;
            for (int i = 0; i < rows; i++, image_y += sy) ys[i] = image_y;
        }
        __syncthreads();
        const uint32_t order = s_order;
        const long long total = (long long)width * rows;
        for (long long i = threadIdx.x; i < total; i += kRasterUnitThreads) {
            const int r = (int)(i / width), cidx = (int)(i % width);
            float ppx, ppy, u, v, w, z;
            if (!raster_fragment(pc, xs[cidx], ys[r], sx, sy, ppx, ppy, u, v, w, z)) continue;
            unsigned long long key;
            if (!raster_key(z, order, key)) continue;
            raster_visit<EMIT>(rb, (size_t)(y0 + r) * fr.rw + (size_t)(pc.min_x + cidx), key, ppx, ppy);
        }
    }
}

// Tallies go to the frame's ChunkCounters (kernels.cuh): traced_primary = fragments whose ray was tested against their piece,
// n_hits = those that hit it (each casts one shadow ray), refl_* = the fans' rays, shadow_vol / shadow_tri = tests of all of them
// (and so does the work map of rt_render_work_map: a fragment's tests are all shadow tests of its pixel).
template <bool COUNT>
__global__ void __launch_bounds__(128)
k_raster_shade(SceneView sc, FrameView fr, RasterView rv, RasterBuffers rb, rt_f4* frag_slots, uint32_t* super, float* g_z, V3* g_n,
               uint32_t background, ChunkCounters* tallies)
{
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    rt_f4* slot = frag_slots + 2 * (size_t)tid;
    const size_t npx = (size_t)fr.rw * fr.rh;
    unsigned long long shaded = 0, hits = 0, refl = 0, refl_shadow = 0, vol = 0, tri = 0;
    unsigned overflow = 0;
    for (size_t pix = tid; pix < npx; pix += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long key = rb.keys[pix];
        if (key == RT_RASTER_EMPTY) { super[pix] = background; continue; }         // clear_image(), renderer.cpp:175-180
        const uint32_t order = (uint32_t)(key & 0xffffffffull);
        const float2 pp = rb.frag_xy[pix];
        TraceCounters tc = zero_counters();
        const RasterShadeOut o = raster_shade<COUNT>(sc, fr, rv, (uint32_t)sc.leaf_of[order >> 4], (int)(order & 15u), (uint32_t)pix, pp.x, pp.y, slot, tid, &tc);
        super[pix] = quantise_argb(o.colour);
        if (g_z != nullptr) { g_z[pix] = raster_key_depth(key); g_n[pix] = o.normal; }   // renderer.cpp:976-979
        shaded += o.shaded; hits += o.hit; refl += tc.refl_rays; refl_shadow += tc.refl_shadow_rays;
        if (COUNT) {
            vol += tc.vol_tests; tri += tc.tri_tests;
            credit_work(tallies, fr, (uint32_t)pix, kWorkShadow, tc.vol_tests, tc.tri_tests);   // all of a fragment's rays, as the totals
        }
        overflow |= tc.stack_overflow;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        shaded += __shfl_down_sync(0xffffffffu, shaded, d); hits += __shfl_down_sync(0xffffffffu, hits, d);
        refl += __shfl_down_sync(0xffffffffu, refl, d); refl_shadow += __shfl_down_sync(0xffffffffu, refl_shadow, d);
        if (COUNT) { vol += __shfl_down_sync(0xffffffffu, vol, d); tri += __shfl_down_sync(0xffffffffu, tri, d); }
    }
    if ((threadIdx.x & 31u) == 0u) {
        if (shaded) atomicAdd(&tallies->traced_primary, shaded);
        if (hits) atomicAdd(&tallies->n_hits, (unsigned int)hits);
        if (refl) atomicAdd(&tallies->refl_rays, refl);
        if (refl_shadow) atomicAdd(&tallies->refl_shadow_rays, refl_shadow);
        if (COUNT) { atomicAdd(&tallies->shadow_vol, vol); atomicAdd(&tallies->shadow_tri, tri); }
    }
    if (overflow) atomicOr(&tallies->stack_overflow, 1u);
}

} // namespace rtb
