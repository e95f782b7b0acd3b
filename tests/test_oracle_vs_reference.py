"""The oracle against the compiled reference itself (oracle/_ref), live: skipped unless RTB200_REFERENCE named the
original sources when oracle/_ref was built (tests/conftest.py).  Pins, among others, the argument evaluation order of renderer.cpp:313."""
import numpy as np
import pytest

from tests import common


@pytest.mark.parametrize("params", [(12, 40), (10, 8), (4, 3), (0, 8)])
def test_random_rays(oracle, ref_strict, robot, params):
    o, d = common.random_rays(40000, 99, (-1.5, -2.5, -5.5), (1.5, 0.5, -2.5))
    a = ref_strict.bvh(robot["xyz9"], *params)
    b = oracle.bvh(robot["xyz9"], *params)
    assert a.stats() == b.stats()
    for x, y in zip(a.intersect(o, d), b.intersect(o, d)):
        assert np.array_equal(x, y)


def test_triangle_soup(oracle, ref_strict):
    soup = common.triangle_soup(5000, 3)
    o, d = common.random_rays(20000, 4, (-1.5, -1.5, -5.5), (1.5, 1.5, -2.5))
    for params in ((12, 40), (6, 2)):
        a, b = ref_strict.bvh(soup, *params), oracle.bvh(soup, *params)
        assert a.stats() == b.stats()
        for x, y in zip(a.intersect(o, d), b.intersect(o, d)):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg3_mirror5"])
def test_images(oracle, ref_strict, robot, name):
    kw, mats, tex = common.config_table(robot["materials"])[name]
    kw = dict(kw, image_width=kw["image_width"] // 2, image_height=kw["image_height"] // 2, rng_seed=11)
    assert np.array_equal(common.oracle_image(oracle, robot, kw, mats, tex), common.oracle_image(ref_strict, robot, kw, mats, tex))


def test_rough_reflection_depth2_and_normal_mapping(oracle, ref_strict, robot):
    kw, mats, tex = common.config_table(robot["materials"])["cfg3"]
    tex = dict(tex)
    tex[2] = common.scenes.normal_map_texture((64, 64), 8)
    kw = dict(kw, image_width=96, image_height=54, max_recursion_depth=2, rough_reflections_sample_count=5, enable_normal_mapping=1)
    assert np.array_equal(common.oracle_image(oracle, robot, kw, mats, tex), common.oracle_image(ref_strict, robot, kw, mats, tex))


@pytest.mark.parametrize("name", ["ssao_ssaa2", "ssao_normal_mapped"])
@pytest.mark.parametrize("seed", [1234, 77])
def test_ssao_reference_order(oracle, ref_strict, robot, name, seed):
    """Renderer::post_process_ssao_SIMD (renderer.cpp:1229-1434) on one thread after srand(seed) against the oracle's
    restatement drawing from the same nine generator seeds in the same order: bit-exact, G-buffers (z, normal-mapped
    normals) included.  The per-pixel stream differs from it only as two samplings of the same estimator do."""
    kw, mats, tex = common.ssao_table(robot["materials"])[name]
    want, rand_values = common.oracle_renderer(ref_strict, robot, kw, mats, tex).render_ssao(srand_seed=seed)
    plain, _ = common.oracle_renderer(ref_strict, robot, dict(kw, enable_ssao=0), mats, tex).render()
    assert (want != plain).mean() > 0.05                                  # the pass really darkens a good part of the frame
    orc = common.oracle_renderer(oracle, robot, kw, mats, tex)
    got, _ = orc.render_ssao(ref_seeds9=common.ssao_reference_seeds(rand_values))
    assert np.array_equal(got, want)
    per_pixel, _ = orc.render_ssao()
    diff = np.abs(common.channels(per_pixel).astype(int) - common.channels(want).astype(int))
    assert diff.mean() < 0.5 and (per_pixel != plain).mean() > 0.05


@pytest.mark.parametrize("name", ["r_inside", "r_big", "r_ssao"])
def test_raster_trace_live(oracle, ref_strict, robot, name):
    """The oracle's restatement of Renderer::raster_trace (clipping, rasterisation, z-buffer, trace_triangle) against the
    compiled reference run here on one thread: bit-exact, also with SSAO on the rasterizer's G-buffers."""
    scene, kw, mats, tex, cam = common.raster_table(robot)[name]
    ref_img, rand_values = common.oracle_renderer(ref_strict, scene, kw, mats, tex, cam=cam).raster(srand_seed=7)
    seeds = common.ssao_reference_seeds(rand_values) if kw.get("enable_ssao") else None
    img, _ = common.oracle_renderer(oracle, scene, kw, mats, tex, cam=cam).raster(ref_seeds9=seeds)
    assert np.array_equal(img, ref_img)
