"""Per-pixel traversal work maps (rt_render_work_map): the six work counters of RtRenderStats split over the final pixels
whose samples issued the rays.

CPU part (the kernel emulation of tests/hostsim with the entry point of tests/hostsim_work_map.cpp): the map sums to the
frame's counters, the frame is render()'s, pixels whose samples all miss carry no shadow or reflection work, the ABI refuses
a NULL map, and a library without the entry point refuses the call.  GPU part: the same over a matrix of scenes
and options (packets, split packets, fused items, top table, leaf split, light cull, lanes, tiny chunks), the single-ray
kernels' maps against the emulation pixel for pixel, where the screen cull leaves its zeros, and the context state the call
must not touch (RT_OPT_COUNT_WORK, the captured frame graphs).

Test tallies of the packet kernels are not reproducible from frame to frame wherever the work of a ray depends on which rays
share its packet or on the timing of split packets: shadow packets are formed from a hit queue whose block order is set by
atomics, and work items prune each other while they run.  So a map's sums are compared with the counters of the SAME call,
and the counters with rt_render's only where they are reproducible."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np
import pytest

import raytracercpp_b200 as rt
from raytracercpp_b200 import api, scenes
from tests import common

FIELDS = [n for n, _ in api.RtPixelWork._fields_]
RAY_COUNTS = ("primary_rays", "shadow_rays", "reflection_rays", "reflection_shadow_rays", "primary_hits", "traced_primary_rays")
FETCHED = ("primary_fetched_bytes", "shadow_fetched_bytes", "reflection_fetched_bytes")
SPHERE_MATS = rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def emu_lib(tmp_path_factory):
    """The kernel emulation (tests/hostsim/hostsim.cpp) with rt_render_work_map (tests/hostsim_work_map.cpp), built for the CPU
    with the flags of tests/hostsim/Makefile."""
    out = tmp_path_factory.mktemp("work_map_emulation") / "librtb200_work_map_emulation.so"
    csrc = ROOT / "raytracercpp_b200" / "csrc"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-o", str(out),
                    str(ROOT / "tests" / "hostsim_work_map.cpp"), str(csrc / "octree_build.cpp"), str(csrc / "scene_io.cpp")], check=True)
    return api.bind(ctypes.CDLL(str(out)), require_all=True)


def settings(r, hybrid=False):
    s = r.render_settings().copy()
    s.hybrid_rasterization_tracing = int(hybrid)
    return s


def factor(s):
    return s.ssaa_factor if s.enable_ssaa else 1


def assert_sums(work, stats, what=""):
    for k in FIELDS:
        assert int(work[k].sum(dtype=np.uint64)) == getattr(stats, k), (what, k, int(work[k].sum(dtype=np.uint64)), getattr(stats, k))


def all_miss_pixels(r, s):
    """Final pixels none of whose samples' primary rays hits a triangle (BVH::intersect of the generated primary rays)."""
    o, d = r.ctx.generate_primary_rays(s)
    tri, _, _, _ = r.ctx.intersect(o, d)
    f = factor(s)
    miss = (tri < 0).reshape(s.image_height, f, s.image_width, f)
    return miss.all(axis=(1, 3))


def host_cases(robot):
    tab = common.config_table(robot["materials"])
    ss = dict(enable_ssaa=1, ssaa_factor=2)
    return {
        "cfg1": (robot, dict(tab["cfg1"][0], image_width=96, image_height=54, **ss), tab["cfg1"][1], tab["cfg1"][2], False),
        "cfg3": (robot, dict(tab["cfg3"][0], image_width=64, image_height=36, **ss), tab["cfg3"][1], tab["cfg3"][2], False),
        "shapes": (robot, dict(tab["cfg3_shapes"][0], image_width=80, image_height=45, **ss), tab["cfg3_shapes"][1], tab["cfg3_shapes"][2], False),
        "raster": (robot, dict(tab["cfg1"][0], image_width=96, image_height=54, **ss), tab["cfg1"][1], tab["cfg1"][2], True),
    }


# ---- CPU: the host emulation -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg1", "cfg3", "shapes", "raster"])
def test_host_map_sums_frame_and_misses(emu_lib, robot, name):
    scene, kw, mats, tex, hybrid = host_cases(robot)[name]
    r = common.product_renderer(emu_lib, scene, kw, mats, tex)
    s = settings(r, hybrid)
    img, work, st = r.ctx.render_work_map(s)
    ref, _ = r.ctx.render(s)
    assert work.shape == (s.image_height, s.image_width)
    assert np.array_equal(img, ref)
    assert_sums(work, st, name)
    assert st.shadow_volume_tests > 0
    if hybrid:                                         # raster_trace: every test of a fragment's rays is a shadow test
        assert st.primary_volume_tests == 0 and not work["primary_volume_tests"].any()
    else:
        assert (work["primary_volume_tests"] > 0).all()     # the emulation traces every sample
    if name in ("cfg1", "cfg3"):                       # (a primary ray that misses the BVH may hit an analytic shape)
        miss = all_miss_pixels(r, s)
        assert miss.any() and not miss.all()
        for k in FIELDS[2:]:
            assert not work[k][miss].any(), k
    if name == "cfg3":
        assert st.reflection_volume_tests > 0 and work["reflection_volume_tests"].any()
    r.close()


def test_pixel_work_layout():
    assert ctypes.sizeof(api.RtPixelWork) == 48
    assert api.PIXEL_WORK_DTYPE.itemsize == 48 and list(api.PIXEL_WORK_DTYPE.names) == FIELDS
    assert FIELDS == [n for n, _ in api.RtRenderStats._fields_ if n.endswith("_tests")]


def test_null_arguments(emu_lib, robot):
    kw, mats, tex = common.config_table(robot["materials"])["cfg1"]
    r = common.product_renderer(emu_lib, robot, dict(kw, image_width=48, image_height=27), mats, tex)
    s = settings(r)
    lib, h = r.ctx.lib, r.ctx.h
    work = np.zeros((27, 48), api.PIXEL_WORK_DTYPE)
    wp = work.ctypes.data_as(ctypes.POINTER(api.RtPixelWork))
    assert lib.rt_render_work_map(h, ctypes.byref(s), None, None, None) == api.RT_ERR_INVALID
    assert lib.rt_render_work_map(h, ctypes.byref(s), None, wp, None) == api.RT_OK
    _, full, st = r.ctx.render_work_map(s)
    assert np.array_equal(work, full)
    assert_sums(work, st)
    r.close()


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
def gpu_scenes(robot):
    tab = common.config_table(robot["materials"])
    rtab = common.raster_table(robot)
    sx, suv, smat = scenes.displaced_sphere(*scenes.sphere_grid_for(200_000))
    hx, huv, hmat = scenes.hair_ball(n_strands=3000, segments=8)
    ssao = common.ssao_table(robot["materials"])["ssao_ssaa2"]
    return {
        "cfg1": (robot, tab["cfg1"][0], tab["cfg1"][1], tab["cfg1"][2], None, False),
        "cfg2": (robot, tab["cfg2"][0], tab["cfg2"][1], tab["cfg2"][2], None, False),
        "cfg3": (robot, tab["cfg3"][0], tab["cfg3"][1], tab["cfg3"][2], None, False),
        "sphere_ssaa4": (dict(xyz9=sx, uv6=suv, mat=smat), dict(image_width=96, image_height=64, enable_ssaa=1, ssaa_factor=4, compute_shadows=1),
                         SPHERE_MATS, {}, None, False),
        "hair": (dict(xyz9=hx, uv6=huv, mat=hmat), dict(image_width=192, image_height=108, compute_shadows=1), SPHERE_MATS, {}, None, False),
        "shapes": (robot, tab["cfg3_shapes"][0], tab["cfg3_shapes"][1], tab["cfg3_shapes"][2], None, False),
        "raster_clip": (robot, rtab["r_inside"][1], rtab["r_inside"][2], rtab["r_inside"][3], rtab["r_inside"][4], True),
        "raster_noclip": (robot, rtab["r_inside_noclip"][1], rtab["r_inside_noclip"][2], rtab["r_inside_noclip"][3], rtab["r_inside_noclip"][4], True),
        "ssao": (robot, ssao[0], ssao[1], ssao[2], None, False),
    }


SPLIT = {api.RT_OPT_PACKET_ROUNDS: 2, api.RT_OPT_ITEM_ROUNDS: 2, api.RT_OPT_PRIMARY_ROUNDS: 2}
VARIANTS = [
    {},
    {api.RT_OPT_PACKETS: 0},
    {api.RT_OPT_FUSED_ITEMS: 1},
    SPLIT,
    {**SPLIT, api.RT_OPT_FUSED_ITEMS: 1},
    {**SPLIT, api.RT_OPT_ITEM_PASSES: 2},
    {api.RT_OPT_TOP_TABLE: 1},
    {api.RT_OPT_LEAF_SPLIT: 0},
    {api.RT_OPT_LEAF_SPLIT: 8, api.RT_OPT_PRIMARY_ROUNDS: 0},
    {api.RT_OPT_LIGHT_CULL: 0},
    {api.RT_OPT_LANES: 0},
    {api.RT_OPT_LANES: 2},
    {api.RT_OPT_CHUNK_PIXELS: 4096},
]


def reproducible(opts, cls):
    """Whether the test tallies of class `cls` repeat from one frame to the next under `opts` (module docstring)."""
    if cls == "reflection" or opts.get(api.RT_OPT_PACKETS) == 0:
        return True                      # reflection fans (and every ray with RT_OPT_PACKETS 0) run the single-ray traversal
    if cls == "primary":                 # primary packets are fixed 8x4 blocks: reproducible unless they are split
        return opts.get(api.RT_OPT_PRIMARY_ROUNDS) == 0
    return False


def make_renderer(lib, scene, kw, mats, tex, cam, opts):
    r = common.product_renderer(lib, scene, kw, mats, tex, cam=cam)
    for k, v in opts.items():
        r.ctx.set_option(k, v)
    if api.RT_OPT_LEAF_SPLIT in opts:
        r.reconstruct_bvh_new()
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "sphere_ssaa4", "hair", "shapes", "raster_clip", "raster_noclip", "ssao"])
def test_map_sums_stats_and_frame_across_options(cuda_lib, robot, name):
    scene, kw, mats, tex, cam, hybrid = gpu_scenes(robot)[name]
    for opts in VARIANTS:
        r = make_renderer(cuda_lib, scene, kw, mats, tex, cam, opts)
        s = settings(r, hybrid)
        img, work, st = r.ctx.render_work_map(s)
        assert_sums(work, st, (name, opts))
        assert st.shadow_volume_tests > 0, (name, opts)
        plain, _ = r.ctx.render(s)                                        # RT_OPT_COUNT_WORK 0: the timed kernels
        assert np.array_equal(img, plain), (name, opts)
        r.ctx.set_option(api.RT_OPT_COUNT_WORK, 1)
        counted, cst = r.ctx.render(s)
        assert np.array_equal(img, counted), (name, opts)
        for k in RAY_COUNTS:
            assert getattr(st, k) == getattr(cst, k), (name, opts, k)
        for cls in ("primary", "shadow", "reflection"):
            keys = [f"{cls}_volume_tests", f"{cls}_triangle_tests", f"{cls}_fetched_bytes"]
            if reproducible(opts, cls):
                for k in keys:
                    assert getattr(st, k) == getattr(cst, k), (name, opts, k)
            else:
                for k in keys:
                    assert (getattr(st, k) > 0) == (getattr(cst, k) > 0), (name, opts, k)
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "cfg3"])
def test_single_ray_maps_equal_the_host_emulation(cuda_lib, emu_lib, robot, name):
    """RT_OPT_PACKETS 0: the GPU's per-lane state machines do exactly the emulation's tests, pixel by pixel."""
    kw, mats, tex = common.config_table(robot["materials"])[name]
    maps = []
    for lib in (cuda_lib, emu_lib):
        r = common.product_renderer(lib, robot, kw, mats, tex)
        r.ctx.set_option(api.RT_OPT_PACKETS, 0)
        img, work, st = r.ctx.render_work_map(settings(r))
        assert_sums(work, st, name)
        maps.append((img, work))
        r.close()
    assert np.array_equal(maps[0][0], maps[1][0])
    for k in FIELDS:
        assert np.array_equal(maps[0][1][k], maps[1][1][k]), (name, k)


@pytest.mark.gpu
def test_screen_cull_leaves_culled_pixels_without_primary_work(cuda_lib):
    """Primary packets are fixed 8x4 sample blocks, so with no packet split a block's work does not depend on the cull: with the
    cull on every pixel carries its cull-off primary work or none, and the pixels that lose it are the culled samples."""
    sx, suv, smat = scenes.displaced_sphere(*scenes.sphere_grid_for(100_000), radius=0.5)
    scene = dict(xyz9=sx, uv6=suv, mat=smat)
    kw = dict(image_width=256, image_height=144, enable_ssaa=1, ssaa_factor=2, compute_shadows=1)
    res = []
    for cull in (0, 1):
        r = make_renderer(cuda_lib, scene, kw, SPHERE_MATS, {}, None, {api.RT_OPT_SCREEN_CULL: cull, api.RT_OPT_PRIMARY_ROUNDS: 0})
        img, work, st = r.ctx.render_work_map(settings(r))
        assert_sums(work, st)
        res.append((img, work, st))
        r.close()
    (img0, w0, st0), (img1, w1, st1) = res
    assert np.array_equal(img0, img1)
    for k in ("primary_volume_tests", "primary_triangle_tests"):
        assert ((w1[k] == 0) | (w1[k] == w0[k])).all(), k
    culled = (w1["primary_volume_tests"] == 0) & (w0["primary_volume_tests"] > 0)
    untraced = st1.primary_rays - st1.traced_primary_rays
    assert untraced > 0 and int(culled.sum()) * 4 == untraced
    for k in FIELDS[2:]:
        assert not w1[k][culled].any(), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "cfg3"])
def test_missed_pixels_carry_no_shadow_or_reflection_work(cuda_lib, robot, name):
    kw, mats, tex = common.config_table(robot["materials"])[name]
    r = common.product_renderer(cuda_lib, robot, dict(kw, enable_ssaa=1, ssaa_factor=2), mats, tex)
    s = settings(r)
    _, work, st = r.ctx.render_work_map(s)
    miss = all_miss_pixels(r, s)
    assert miss.any() and not miss.all()
    for k in FIELDS[2:]:
        assert not work[k][miss].any(), (name, k)
    assert work["shadow_volume_tests"][~miss].any()
    r.close()


@pytest.mark.gpu
def test_primary_map_does_not_depend_on_the_light_cull(cuda_lib, robot):
    kw, mats, tex = common.config_table(robot["materials"])["cfg2"]
    maps = []
    for cull in (0, 1):
        r = make_renderer(cuda_lib, robot, kw, mats, tex, None, {api.RT_OPT_LIGHT_CULL: cull, api.RT_OPT_PRIMARY_ROUNDS: 0})
        img, work, _ = r.ctx.render_work_map(settings(r))
        maps.append((img, work))
        r.close()
    assert np.array_equal(maps[0][0], maps[1][0])
    for k in FIELDS[:2]:
        assert np.array_equal(maps[0][1][k], maps[1][1][k]), k


@pytest.mark.gpu
def test_context_state_is_left_alone(cuda_lib, robot):
    """A map call between frames replayed from a captured graph: the replay goes on (stage times 0, as for every replayed
    frame) with the same frame, RT_OPT_COUNT_WORK stays what it was, and after a transform + rebuild the map still sums up."""
    kw, mats, tex = common.config_table(robot["materials"])["cfg1"]
    r = common.product_renderer(cuda_lib, robot, kw, mats, tex)
    s = settings(r)
    frames = [r.ctx.render(s) for _ in range(3)]                           # enqueued, captured, replayed
    assert frames[2][1].trace_primary_ms == 0 and frames[2][1].shade_ms == 0
    img, work, st = r.ctx.render_work_map(s)
    assert_sums(work, st)
    assert np.array_equal(img, frames[2][0])
    after, ast = r.ctx.render(s)
    assert np.array_equal(after, frames[2][0])
    assert ast.trace_primary_ms == 0 and ast.shade_ms == 0                 # still the replayed graph
    for k in FIELDS:
        assert getattr(ast, k) == 0, k                                      # RT_OPT_COUNT_WORK is still 0
    r.ctx.set_option(api.RT_OPT_COUNT_WORK, 1)
    r.ctx.render_work_map(s)
    _, cst = r.ctx.render(s)
    assert cst.primary_volume_tests > 0 and cst.shadow_volume_tests > 0     # ... and 1 stays 1
    r.ctx.set_option(api.RT_OPT_COUNT_WORK, 0)
    m = np.eye(4, dtype=np.float32)
    m[:3, 3] = (0.3, -0.2, -0.5)
    r.set_object_transform(m)
    img2, work2, st2 = r.ctx.render_work_map(s)
    assert_sums(work2, st2)
    assert np.array_equal(img2, r.ctx.render(s)[0])
    assert not np.array_equal(img2, img)
    r.close()


def test_a_library_without_the_entry_point_refuses_the_call(hostsim_lib, robot):
    """The emulation of tests/hostsim alone does not export rt_render_work_map: it still binds (every other symbol), and the
    call raises instead of rendering anything else."""
    assert not hasattr(hostsim_lib, "rt_render_work_map")
    kw, mats, tex = common.config_table(robot["materials"])["cfg1"]
    r = common.product_renderer(hostsim_lib, robot, dict(kw, image_width=48, image_height=27), mats, tex)
    with pytest.raises(api.RtError) as e:
        r.ctx.render_work_map(settings(r))
    assert e.value.code == api.RT_ERR_UNSUPPORTED
    r.close()
