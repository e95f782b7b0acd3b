// hostsim_work_map.cpp -- TEST INFRASTRUCTURE ONLY: the kernel emulation of tests/hostsim plus rt_render_work_map.
//
// Built by tests/test_work_map.py into a library of its own (hostsim.cpp + this entry point, octree_build.cpp, scene_io.cpp).
// rt_render_work_map renders the frame and its RtRenderStats with the emulation's rt_render, then walks the same rays again
// serially with the counting traversal of rt_device.h -- primary ray, analytic shapes and the min_t gate, the reflection fan
// of a reflective hit (same random stream), the depth-0 shadow ray; in a hybrid_rasterization_tracing frame the shading of
// each pixel's winning fragment -- and credits each ray tree's TraceCounters to the final pixel of its sample.  The serial
// traversal is deterministic, so the map's sums must equal the emulation's counters: the tests check exactly that.
#include "hostsim/hostsim.cpp"

namespace {

void credit(RtPixelWork* map, const FrameView& fr, uint32_t pix, int cls, const TraceCounters& tc)
{
    const uint32_t rw = (uint32_t)fr.rw, f = (uint32_t)fr.factor;
    uint64_t* w = &map[(size_t)((pix / rw) / f) * (rw / f) + (pix % rw) / f].primary_volume_tests + 2 * cls;
    w[0] += tc.vol_tests;
    w[1] += tc.tri_tests;
}

// the depth pass and the emit pass of raster_trace (hostsim.cpp): the winning fragment's key and pixel point per sample
void raster_keys(const RtContext* c, const SceneView& sc, const FrameView& fr, const RasterView& rv, std::vector<unsigned long long>& keys,
                 std::vector<float>& fx, std::vector<float>& fy)
{
    const size_t npx = (size_t)fr.rw * fr.rh;
    keys.assign(npx, RT_RASTER_EMPTY);
    fx.assign(npx, 0.0f);
    fy.assign(npx, 0.0f);
    const float sx = raster_scale(fr.rw), sy = raster_scale(fr.rh);
    for (int pass = 0; pass < 2; pass++)
        for (uint32_t tri = 0; tri < sc.n_tris; tri++) {
            const RasterSource src = raster_source(sc, tri);
            Tri4 scratch[RT_CLIP_MAX], clipped[RT_CLIP_MAX];
            const int np = raster_clip(rv, src.a, src.b, src.c, src.tu, src.tv, scratch, clipped);
            for (int pi = 0; pi < np; pi++) {
                const RasterPiece pc = raster_piece(fr, clipped[pi]);
                float image_y = raster_start(pc.min_y, sy);
                for (int py = pc.min_y; py <= pc.max_y; py++, image_y += sy) {
                    float image_x = raster_start(pc.min_x, sx);
                    for (int px = pc.min_x; px <= pc.max_x; px++, image_x += sx) {
                        float ppx, ppy, u, v, w, z;
                        if (!raster_fragment(pc, image_x, image_y, sx, sy, ppx, ppy, u, v, w, z)) continue;
                        unsigned long long key;
                        if (!raster_key(z, (uint32_t)src.orig * 16u + (uint32_t)pi, key)) continue;
                        const size_t pix = (size_t)py * fr.rw + px;
                        if (pass == 0) keys[pix] = std::min(keys[pix], key);
                        else if (keys[pix] == key) { fx[pix] = ppx; fy[pix] = ppy; }
                    }
                }
            }
        }
    (void)c;
}

} // namespace

extern "C" int rt_render_work_map(RtContext* c, const RtSettings* s, uint32_t* argb_out, RtPixelWork* work_out, RtRenderStats* stats)
{
    if (!work_out) return fail(c, RT_ERR_INVALID, "work_out is NULL");
    std::string why;
    if (int r = check_settings(s, why)) return fail(c, r, why);
    std::vector<uint32_t> frame((size_t)s->image_width * s->image_height);
    if (int r = rt_render(c, s, frame.data(), stats)) return r;
    if (argb_out) memcpy(argb_out, frame.data(), frame.size() * sizeof(uint32_t));
    memset(work_out, 0, frame.size() * sizeof(RtPixelWork));
    const FrameView fr = frame_view(c, s);
    const SceneView sc = scene_view(c);
    if (s->hybrid_rasterization_tracing) {
        RasterView rv;
        rv.world_to_cam = invert_matrix(c->cam_to_world);
        rv.proj = c->proj;
        rv.clipping = s->enable_clipping;
        std::vector<unsigned long long> keys;
        std::vector<float> fx, fy;
        raster_keys(c, sc, fr, rv, keys, fx, fy);
        std::vector<int32_t> leaf_of(sc.n_tris);
        for (uint32_t i = 0; i < sc.n_tris; i++) leaf_of[(size_t)sc.orig[i]] = (int32_t)i;
        F4 frag_slot[2];
        SceneView scf = sc;
        scf.frag_shade = frag_slot;
        for (size_t pix = 0; pix < keys.size(); pix++) {
            if (keys[pix] == RT_RASTER_EMPTY) continue;
            const uint32_t order = (uint32_t)(keys[pix] & 0xffffffffull);
            TraceCounters tc = zero_counters();
            raster_shade<true>(scf, fr, rv, (uint32_t)leaf_of[order >> 4], (int)(order & 15u), (uint32_t)pix, fx[pix], fy[pix], frag_slot, 0u, &tc);
            credit(work_out, fr, (uint32_t)pix, 1, tc);                       // every test of a fragment's rays is a shadow test
        }
        return RT_OK;
    }
    const bool reflect = c->any_reflective && s->shading_method == RT_SHADING;
    for (int py = 0; py < fr.rh; py++)
        for (int px = 0; px < fr.rw; px++) {
            const uint32_t pix = (uint32_t)py * (uint32_t)fr.rw + (uint32_t)px;
            V3 o, d;
            primary_ray(fr, px, py, o, d);
            HitRec hr;
            TraceCounters tc = zero_counters();
            bool found = trace_closest<true>(sc, o, d, hr, &tc);
            credit(work_out, fr, pix, 0, tc);
            float final_t = found ? hr.t : -1.0f;                             // the analytic shapes, then the min_t gate
            for (int i = 0; i < sc.n_shapes; i++) {
                float t;
                V3 sn;
                int32_t sm;
                if (shape_intersect(sc, i, o, d, t, sn, sm) && (t < final_t || final_t == -1.0f)) { final_t = t; hr.tri = -2 - i; hr.t = t; found = true; }
            }
            if (!(found && hr.t > 0.1f) || s->shading_method != RT_SHADING) continue;
            const int32_t mat = hr.tri >= 0 ? load_tri_shade(sc, hr.tri).mat : shape_material(sc, -2 - hr.tri);
            if (reflect && load_material(sc, mat).reflection > 0.0f) {
                Hit hit = make_hit(sc, hr, o, d);
                V3 p;
                MatView m;
                shade_direct(sc, fr, o, d, hit, p, m);
                XorShift32 rng;
                rng.state = pixel_seed(pix, fr.s.rng_seed);
                TraceCounters tr = zero_counters();
                compute_reflection<true>(sc, fr, d, p, hit, m, 0, rng, &tr);
                credit(work_out, fr, pix, 2, tr);
            }
            if (fr.s.compute_shadows) {
                Hit hit = make_hit(sc, hr, o, d);
                V3 p;
                MatView m;
                shade_direct(sc, fr, o, d, hit, p, m);
                TraceCounters ts = zero_counters();
                trace_occluded<true>(sc, p, hit.normal, fr.light, &ts);
                credit(work_out, fr, pix, 1, ts);
            }
        }
    return RT_OK;
}
