"""The wide copy of the tree that the packet kernels traverse (wrecs[], octree_device.cuh: k_wb_*): blocks of up to 8
records collapsed from the reference-shaped recs[], which the single-ray kernels keep.  Frames and ray / hit counts of
the packet kernels must equal those of the single-ray kernels bit for bit, and the oracle's frame within the shading
tolerance, on scenes whose trees stress the collapse, with either builder, every leaf refinement, the top table, split
packets (work items carry links into wrecs[]) and a rebuild replayed through frame graphs."""
import numpy as np
import pytest

import raytracercpp_b200 as rt
from raytracercpp_b200 import api, scenes
from tests import common

pytestmark = pytest.mark.gpu

COUNTS = ("primary_rays", "shadow_rays", "primary_hits", "reflection_rays", "reflection_shadow_rays")
MATS = rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
KW = dict(image_width=128, image_height=72, compute_shadows=1)


def one_material(xyz9):
    return dict(xyz9=np.ascontiguousarray(xyz9, np.float32), uv6=None, mat=np.zeros(len(xyz9), np.int32))


def wide_scenes():
    tri = np.float32([[-0.6, -0.5, -3, 0.7, -0.4, -3.2, 0.1, 0.6, -2.9]])
    hx, huv, hmat = scenes.hair_ball(n_strands=1500, segments=8)
    return {
        # a chain of single-child cells down to max_depth, then one leaf of 60 that cannot be refined
        "coincident": (one_material(np.repeat(tri, 60, 0)), KW, {}),
        # max_depth 2: leaves of hundreds of triangles, refined below the reference's leaves
        "depth_capped": (one_material(common.triangle_soup(3000, 4, size=0.05)), dict(KW, bvh_max_depth=2, bvh_leaf_object_count=4), {}),
        "hair": (dict(xyz9=hx, uv6=huv, mat=hmat), KW, {}),
        "soup": (one_material(common.triangle_soup(4000, 7, size=0.1)), KW, {}),
        # camera and light inside the soup's root cell
        "inside": (one_material(common.triangle_soup(4000, 8, size=0.1)), KW, dict(cam=np.float32([[1, 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, -4.0], [0, 0, 0, 1]]),
                                                                                   light=(0.3, 0.2, -3.8))),
    }


def render(lib, scene, kw, where, opts):
    r = common.product_renderer(lib, scene, kw, MATS, {}, **where)
    for k, v in opts.items():
        r.ctx.set_option(k, v)
    r.reconstruct_bvh_new()
    r.ray_trace()
    img, st = r.get_image().copy(), r.last_stats().as_dict()
    r.close()
    return img, st


VARIANTS = [
    {},
    {api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_TOP_TABLE: 1},
    {api.RT_OPT_TOP_TABLE: 1, api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_LEAF_SPLIT: 0},
    {api.RT_OPT_LEAF_SPLIT: 1},
    {api.RT_OPT_LEAF_SPLIT: 3, api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_LEAF_SPLIT: 16},
] + [
    {api.RT_OPT_PACKET_ROUNDS: n, api.RT_OPT_PRIMARY_ROUNDS: n, api.RT_OPT_ITEM_ROUNDS: n, api.RT_OPT_FUSED_ITEMS: fused, api.RT_OPT_TOP_TABLE: n & 1}
    for n in (1, 2, 3) for fused in (0, 1)
]


@pytest.mark.parametrize("name", ["coincident", "depth_capped", "hair", "soup", "inside"])
def test_packets_on_the_wide_tree_equal_single_rays(cuda_lib, oracle, name):
    scene, kw, where = wide_scenes()[name]
    base, base_st = render(cuda_lib, scene, kw, where, {api.RT_OPT_PACKETS: 0})
    assert base_st["primary_hits"] > 0
    for opts in VARIANTS:
        img, st = render(cuda_lib, scene, kw, where, opts)
        assert np.array_equal(img, base), (name, opts)
        for k in COUNTS:
            assert st[k] == base_st[k], (name, opts, k)
    common.assert_image_close(base, common.oracle_image(oracle, scene, kw, MATS, {}, **where), what=name)


def test_rebuild_replayed_through_frame_graphs(cuda_lib):
    """Transform + rebuild between frames that replay a captured frame graph: the graph of the old tree must not be
    replayed on the new one."""
    scene = one_material(common.triangle_soup(4000, 9, size=0.1))
    m = np.eye(4, dtype=np.float32)
    c, s_ = np.float32(np.cos(0.7)), np.float32(np.sin(0.7))
    m[0, 0], m[0, 2], m[2, 0], m[2, 2] = c, s_, -s_, c
    m[:3, 3] = (4.0 * s_ + 0.4, -0.2, -4.0 * (1 - c))                          # about the soup's centre, moved a little
    frames = []
    for packets in (1, 0):
        r = common.product_renderer(cuda_lib, scene, KW, MATS, {})
        r.ctx.set_option(api.RT_OPT_PACKETS, packets)
        r.ctx.set_option(api.RT_OPT_GRAPH, packets)
        for _ in range(3):                                                     # the third frame replays the second's graph
            r.ray_trace()
        before = r.get_image().copy()
        r.set_object_transform(m)
        for _ in range(3):
            r.ray_trace()
        frames.append((before, r.get_image().copy(), r.last_stats().as_dict()))
        r.close()
    (b1, a1, s1), (b0, a0, s0) = frames
    assert np.array_equal(b1, b0) and np.array_equal(a1, a0) and not np.array_equal(a1, b1)
    for k in COUNTS:
        assert s1[k] == s0[k], k
