"""The light cull of the shadow packets (csrc/light_cull.cuh, RT_OPT_LIGHT_CULL): triangles with the point light strictly on
their front side, and subtrees of only such triangles, are skipped by the any-hit packet traversal.

The CPU test restates tri_test (rt_device.h, the reference's back-face-culled Moeller-Trumbore) with the shadow predicate
of renderer.cpp:351-354 and the mask rule in numpy float32, in the kernels' operation order, and checks that no triangle
the rule prunes is ever accepted -- on tiny, huge, sliver and degenerate triangles, lights on, near and far from their
planes, shadow rays built as the kernels build them (origin EPSILON off the hit point along a shading normal that is not
the geometric one, direction taken from the hit point).  The GPU tests render with the cull on and off: frames and ray /
hit counters must be identical."""
import numpy as np
import pytest

import raytracercpp_b200 as rt
from raytracercpp_b200 import api, scenes
from tests import common

F = np.float32
ABS_MARGIN, REL_MARGIN = F(2.5e-4), F(2.0 ** -16)


def dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def cross(u, v):
    return np.stack([u[..., 1] * v[..., 2] - u[..., 2] * v[..., 1], u[..., 2] * v[..., 0] - u[..., 0] * v[..., 2],
                     u[..., 0] * v[..., 1] - u[..., 1] * v[..., 0]], -1)


def normalize(v):
    with np.errstate(divide="ignore", invalid="ignore"):
        kk = F(1) / np.sqrt(dot(v, v))
    return kk[..., None] * v


def norm1(v):
    return (np.abs(v[..., 0]) + np.abs(v[..., 1])) + np.abs(v[..., 2])


def tri_test(a, b, c, n, o, md):
    """rt_device.h: tri_test, vectorised; returns (accepted, t)."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        det = dot(n, md)
        ok = det > 0
        ab, ac, oa = b - a, c - a, o - a
        mdxoa = cross(md, oa)
        inv = F(1) / det
        u = dot(mdxoa, ac) * inv
        ok &= ~((u < 0) | (u > 1))
        v = dot(mdxoa, -ab) * inv
        ok &= ~((v < 0) | (u + v > 1))
        t = dot(n, oa) * inv
        ok &= ~(t < 0)
    return ok, t


def may_occlude(a, b, c, n, light, span):
    """light_cull.cuh: may_occlude, vectorised."""
    with np.errstate(invalid="ignore", over="ignore"):
        ha, hb, hc = dot(n, light - a), dot(n, light - b), dot(n, light - c)
        ext = (np.maximum(norm1(a), np.maximum(norm1(b), norm1(c))) + norm1(light)) + span
        margin = norm1(n) * (ABS_MARGIN + REL_MARGIN * ext)
        return ~((ha > margin) & (hb > margin) & (hc > margin))


def random_cases(rng, m):
    """m triangles, lights and shadow rays, in float32."""
    centre = rng.uniform(-3, 3, (m, 1, 3))
    size = 10.0 ** rng.uniform(-4, 1.5, (m, 1, 1))                   # a refined leaf of 10 M triangles .. a ground quad
    tri = centre + size * rng.normal(size=(m, 3, 3))
    kind = rng.integers(0, 4, m)
    w = rng.uniform(0, 1, (m, 1))
    tri[kind == 1, 2] = (w * tri[:, 0] + (1 - w) * tri[:, 1])[kind == 1] + size[kind == 1, 0] * 1e-4 * rng.normal(size=(int((kind == 1).sum()), 3))  # sliver
    tri[kind == 2, 2] = tri[kind == 2, 1]                               # degenerate: two equal vertices
    tri[kind == 3, 2] = (w * tri[:, 0] + (1 - w) * tri[:, 1])[kind == 3]   # degenerate: collinear
    tri = tri.astype(F)
    a, b, c = tri[:, 0], tri[:, 1], tri[:, 2]
    n = cross(b - a, c - a)                                             # the cached normal (k_ob_triangles)
    with np.errstate(divide="ignore", invalid="ignore"):
        nhat = np.nan_to_num(n / np.linalg.norm(n.astype(np.float64), axis=-1, keepdims=True)).astype(np.float64)
    # the light: on the plane, near it (either side) or far from it, somewhere above the triangle or off to the side
    x_on = (a + rng.uniform(0, 1, (m, 1)) * (b - a) + rng.uniform(0, 1, (m, 1)) * (c - a)).astype(np.float64)
    lateral = rng.normal(size=(m, 3)) * 10.0 ** rng.uniform(-3, 1, (m, 1))
    lateral -= (lateral * nhat).sum(-1, keepdims=True) * nhat
    height = rng.choice([0.0, 1.0], (m, 1)) * rng.choice([-1.0, 1.0], (m, 1)) * 10.0 ** rng.uniform(-8, 1, (m, 1))
    light = (x_on + lateral + height * nhat).astype(F)
    # hit points: on the line from the light through a point of the triangle, beyond it (the ray crosses the triangle), on
    # the triangle itself (its own shadow ray), or anywhere near
    x = (a + rng.uniform(0, 0.6, (m, 1)) * (b - a) + rng.uniform(0, 0.4, (m, 1)) * (c - a)).astype(np.float64)
    s = 1.0 + rng.choice([0.0, 1.0], (m, 1)) * 10.0 ** rng.uniform(-7, 1, (m, 1))
    p = light + s * (x - light)
    stray = rng.uniform(0, 1, m) < 0.2
    p[stray] += rng.normal(size=(int(stray.sum()), 3)) * size[stray, 0]
    p = p.astype(F)
    # shading normals: the geometric one (either way round), a perturbed one, or any direction
    g = nhat * rng.choice([-1.0, 1.0], (m, 1))
    nrm = np.where(rng.uniform(0, 1, (m, 1)) < 0.5, g + 0.3 * rng.normal(size=(m, 3)), rng.normal(size=(m, 3)))
    nrm = normalize(nrm.astype(F))
    return a, b, c, n, light, p, nrm


@pytest.mark.parametrize("seed", range(8))
def test_pruned_triangles_are_never_accepted_by_a_shadow_ray(seed):
    rng = np.random.default_rng(1000 + seed)
    a, b, c, n, light, p, nrm = random_cases(rng, 200_000)
    so = p + F(1.0e-4) * nrm                                            # k_shade_packet: L.p + 1.0e-4f * L.nrm
    sd = normalize(light - p)
    dist2 = dot(p - light, p - light)
    ok, t = tri_test(a, b, c, n, so, -sd)
    with np.errstate(invalid="ignore", over="ignore"):
        q = so + t[:, None] * sd                                        # renderer.cpp:351
        accepted = ok & (t > 0) & (dot(p - q, p - q) < dist2)           # renderer.cpp:354
    # span: at least the shadow ray's length and the light's distance to the triangle (plan_light_masks bounds both)
    far = np.sqrt(np.maximum(dist2, np.maximum(dot(light - a, light - a), np.maximum(dot(light - b, light - b), dot(light - c, light - c)))))
    span = (F(1.01) * far + F(1e-3)).astype(F)
    pruned = ~may_occlude(a, b, c, n, light, span)
    assert not np.any(pruned & accepted), np.flatnonzero(pruned & accepted)[:10]
    assert pruned.mean() > 0.05 and accepted.sum() > 2000               # the rule prunes, and the rays do hit
    # near-miss cases exist: the light within 10 margins of the plane of a triangle that is still kept
    assert np.any(~pruned & accepted & (np.abs(dot(n, light - a)) < 10 * norm1(n) * ABS_MARGIN))


def test_degenerate_and_nan_triangles_are_kept():
    light = np.array([[0.0, 0.0, 5.0]], F)
    a = np.array([[0, 0, 0]], F)
    for b, c in (([1, 0, 0], [1, 0, 0]), ([1, 0, 0], [2, 0, 0]), ([np.nan, 0, 0], [0, 1, 0]), ([np.inf, 0, 0], [0, 1, 0])):
        b, c = np.array([b], F), np.array([c], F)
        with np.errstate(invalid="ignore"):
            n = cross(b - a, c - a)
        assert may_occlude(a, b, c, n, light, F(10)).all()
    b, c = np.array([[1, 0, 0]], F), np.array([[0, 1, 0]], F)               # n = +z: the light is in front ...
    n = cross(b - a, c - a)
    assert not may_occlude(a, b, c, n, light, F(10)).any()
    assert may_occlude(a, b, c, n, np.array([[0, 0, 1e-5]], F), F(10)).all()   # ... but not by the margin
    assert may_occlude(a, c, b, cross(c - a, b - a), light, F(10)).all()      # the other winding faces away


# ---------------------------------------------------------------------------------------------------------------- GPU

COUNTS = ("primary_rays", "shadow_rays", "primary_hits", "reflection_rays", "reflection_shadow_rays")
MATS = rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
KW = dict(image_width=160, image_height=90, compute_shadows=1)


def one_material(xyz9):
    return dict(xyz9=np.ascontiguousarray(xyz9, np.float32), uv6=None, mat=np.zeros(len(xyz9), np.int32))


def with_ground(xyz9, y):
    """xyz9 plus a large two-triangle ground quad at height y, facing up."""
    quad = np.float32([[-20, y, 10, 20, y, 10, 20, y, -30], [-20, y, 10, 20, y, -30, -20, y, -30]])
    return one_material(np.concatenate([xyz9, quad]))


def cull_scenes(robot=None):
    sx, suv, smat = scenes.displaced_sphere(*scenes.sphere_grid_for(300_000))
    hx, huv, hmat = scenes.hair_ball(n_strands=3000, segments=8)
    soup = common.triangle_soup(4000, 8, size=0.1)
    out = {
        "sphere": (dict(xyz9=sx, uv6=suv, mat=smat), KW, MATS, {}, {}),
        "hair": (dict(xyz9=hx, uv6=huv, mat=hmat), KW, MATS, {}, {}),
        # camera and light inside the soup's root cell
        "inside": (one_material(soup), KW, MATS, {}, dict(cam=np.float32([[1, 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, -4.0], [0, 0, 0, 1]]),
                                                         light=(0.3, 0.2, -3.8))),
        # the light exactly in the plane of the ground quad's two large triangles
        "light_on_plane": (with_ground(soup, -1.0), KW, MATS, {}, dict(light=(2.0, -1.0, -1.0))),
        # an analytic sphere (the masks' span grows to cover its hit points) and a plane (masks with every bit set)
        "sphere_shape": (one_material(soup), KW, MATS + rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL]),
                         {"shapes": [("sphere", (0.6, 0.3, -3.0), 0.5, 1)]}, {}),
        "plane_shape": (one_material(soup), KW, MATS + rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL]),
                        {"shapes": [("plane", (0, -1.5, 0), (0, 1, 0), 1), ("sphere", (0.6, 0.3, -3.0), 0.5, 1)]}, {}),
    }
    if robot is not None:                                                   # normal mapping moves the shadow rays' origins
        kw, mats, tex = common.config_table(robot["materials"])["cfg2"]
        out["normal_mapped"] = (dict(xyz9=robot["xyz9"], uv6=robot["uv6"], mat=robot["mat"]), kw, mats, tex, {})
    return out


def render(lib, scene, kw, mats, tex, where, opts, frames=1):
    r = common.product_renderer(lib, scene, kw, mats, tex, **where)
    for k, v in opts.items():
        r.ctx.set_option(k, v)
    r.reconstruct_bvh_new()
    for _ in range(frames):
        r.ray_trace()
    img, st = r.get_image().copy(), r.last_stats().as_dict()
    r.close()
    return img, st


VARIANTS = [
    {},
    {api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_LEAF_SPLIT: 0},
    {api.RT_OPT_LEAF_SPLIT: 1},
    {api.RT_OPT_LEAF_SPLIT: 0, api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_TOP_TABLE: 1},
    # split packets: work items start at links the masks have already filtered
    {api.RT_OPT_PACKET_ROUNDS: 1, api.RT_OPT_ITEM_ROUNDS: 1},
    {api.RT_OPT_PACKET_ROUNDS: 2, api.RT_OPT_ITEM_ROUNDS: 2, api.RT_OPT_TOP_TABLE: 1},
    {api.RT_OPT_PACKET_ROUNDS: 2, api.RT_OPT_ITEM_ROUNDS: 2, api.RT_OPT_FUSED_ITEMS: 1},
]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere", "hair", "inside", "light_on_plane", "sphere_shape", "plane_shape", "normal_mapped"])
def test_light_cull_changes_no_frame_and_no_count(cuda_lib, robot, name):
    scene, kw, mats, tex, where = cull_scenes(robot)[name]
    for opts in VARIANTS:
        off, off_st = render(cuda_lib, scene, kw, mats, tex, where, {**opts, api.RT_OPT_LIGHT_CULL: 0})
        on, on_st = render(cuda_lib, scene, kw, mats, tex, where, opts)
        assert off_st["shadow_rays"] > 0
        assert np.array_equal(on, off), (name, opts)
        for k in COUNTS:
            assert on_st[k] == off_st[k], (name, opts, k)


@pytest.mark.gpu
def test_light_cull_skips_work(cuda_lib):
    """The instrumented kernels test fewer triangles with the cull on, for the same frame."""
    scene, kw, mats, tex, where = cull_scenes()["sphere"]
    res = [render(cuda_lib, scene, kw, mats, tex, where, {api.RT_OPT_COUNT_WORK: 1, api.RT_OPT_LIGHT_CULL: on}) for on in (0, 1)]
    (off, off_st), (on, on_st) = res
    assert np.array_equal(on, off)
    assert on_st["shadow_triangle_tests"] < 0.8 * off_st["shadow_triangle_tests"], (on_st["shadow_triangle_tests"], off_st["shadow_triangle_tests"])


@pytest.mark.gpu
def test_masks_follow_light_moves_tree_changes_and_the_option_through_frame_graphs(cuda_lib):
    """Light 1 -> 2 -> 1, a transform + rebuild and the option toggled between frames that replay captured frame graphs,
    against the same sequence without graphs and without the cull."""
    scene = one_material(common.triangle_soup(4000, 9, size=0.1))
    m = np.eye(4, dtype=np.float32)
    c, s_ = np.float32(np.cos(0.7)), np.float32(np.sin(0.7))
    m[0, 0], m[0, 2], m[2, 0], m[2, 2] = c, s_, -s_, c
    m[:3, 3] = (4.0 * s_ + 0.4, -0.2, -4.0 * (1 - c))
    steps = [("light", (3.0, 3.0, 2.0)), ("light", (-2.0, 1.0, -1.0)), ("light", (3.0, 3.0, 2.0)), ("cull", 0), ("cull", 1),
             ("transform", m), ("light", (-2.0, 1.0, -1.0)), ("light", (3.0, 3.0, 2.0))]
    runs = []
    for graph, cull in ((1, 1), (0, 1), (0, 0)):
        r = common.product_renderer(cuda_lib, scene, KW, MATS, {})
        r.ctx.set_option(api.RT_OPT_GRAPH, graph)
        r.ctx.set_option(api.RT_OPT_LIGHT_CULL, cull)
        frames = []
        for what, v in steps:
            if what == "light":
                r.set_light_position(v)
            elif what == "transform":
                r.set_object_transform(v)
            elif cull:
                r.ctx.set_option(api.RT_OPT_LIGHT_CULL, v)
            for _ in range(3):                                              # the third frame replays the second's graph
                r.ray_trace()
            frames.append((r.get_image().copy(), r.last_stats().as_dict()))
        r.close()
        runs.append(frames)
    for frames in runs[1:]:
        for (a, sa), (b, sb) in zip(runs[0], frames):
            assert np.array_equal(a, b)
            for k in COUNTS:
                assert sa[k] == sb[k], k
    assert not np.array_equal(runs[0][0][0], runs[0][1][0])                # the light did move
