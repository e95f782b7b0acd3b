"""Blocks of up to 16 records in the wide tree (octree_device.cuh: k_wb_collapse, rt_device.h: kWideBlock): the packet
cull, the staging of a cell round and the light-cull masks must cover every member of a block, and the packet stack must
hold the deepest tree the builders allow.  Frames and ray / hit counts of the packet kernels are compared with those of
the single-ray kernels bit for bit, and with the oracle's frame within the shading tolerance."""
import numpy as np
import pytest

import raytracercpp_b200 as rt
from raytracercpp_b200 import api, scenes
from tests import common

pytestmark = pytest.mark.gpu

COUNTS = ("primary_rays", "shadow_rays", "primary_hits", "reflection_rays", "reflection_shadow_rays")
MATS = rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
KW = dict(image_width=160, image_height=90, compute_shadows=1)


def one_material(xyz9):
    return dict(xyz9=np.ascontiguousarray(xyz9, np.float32), uv6=None, mat=np.zeros(len(xyz9), np.int32))


def two_clusters():
    """Two dense soups in opposite octants of the root cell: the root has two children of eight children each, so its
    block holds 16 records, and the dense cells below collapse into blocks of 15."""
    a = common.triangle_soup(3000, 21, size=0.03, center=(-0.8, -0.5, -4.6), spread=0.6)
    b = common.triangle_soup(3000, 22, size=0.03, center=(0.8, 0.5, -3.4), spread=0.6)
    return one_material(np.concatenate([a, b]))


def nested(levels=22):
    """A chain of octree cells down to max_depth 20 and below (leaf size 1).  At every level the cell [0, h]^3 has a
    single triangle in each of its octants 1..6, a cluster of eight triangles (one per sub-octant) in octant 7 and the
    next level in octant 0: eight children per cell on every level of the chain, and the leaf at the depth cap refined
    below it.  Blocks of 16 absorb a cluster or the next level beside the chain's cells, and the packet stack bound of the
    tree comes within a few entries of RT_STACK_SIZE."""
    shape = np.float32([[-1.0, -0.5, 0.0], [1.0, -0.5, 0.2], [0.0, 1.0, -0.2]])      # faces +z, towards the camera
    tris = []
    for k in range(levels):
        h = 0.5 ** k
        for o in range(1, 7):
            c = np.float32([(0.5 + ((o >> a) & 1)) * 0.5 * h for a in range(3)])
            tris.append(c + 0.1 * h * shape)
        for o in range(8):
            c = np.float32([0.5 * h + (0.5 + ((o >> a) & 1)) * 0.25 * h for a in range(3)])
            tris.append(c + 0.45 * 0.25 * h * shape)
    tris.append(np.float32([[0, 0, 0], [1e-7, 0, 0], [0, 1e-7, 0]]))                # pins the root cell to [0, 1]^3
    tris.append(np.float32([[1, 1, 1], [1 - 1e-3, 1, 1], [1, 1 - 1e-3, 1]]))
    xyz = 2.0 * np.stack(tris).astype(np.float64) + np.float64([0.0, 0.0, -4.0])   # corner of the chain at (0, 0, -4)
    return one_material(xyz.reshape(-1, 9))


def render(lib, scene, kw, opts, frames=1, **where):
    r = common.product_renderer(lib, scene, kw, MATS, {}, **where)
    for k, v in opts.items():
        r.ctx.set_option(k, v)
    r.reconstruct_bvh_new()
    for _ in range(frames):
        r.ray_trace()
    img, st = r.get_image().copy(), r.last_stats().as_dict()
    r.close()
    return img, st


# work items of split packets start at links into 16-wide blocks; the top table holds whole 16-wide blocks
VARIANTS = [
    {},
    {api.RT_OPT_DEVICE_BUILD: 0},
    {api.RT_OPT_TOP_TABLE: 1},
    {api.RT_OPT_LIGHT_CULL: 0},
    {api.RT_OPT_SCREEN_CULL: 0},
] + [
    {api.RT_OPT_PACKET_ROUNDS: n, api.RT_OPT_PRIMARY_ROUNDS: n, api.RT_OPT_ITEM_ROUNDS: n, api.RT_OPT_FUSED_ITEMS: fused, api.RT_OPT_TOP_TABLE: n & 1}
    for n in (1, 2, 3) for fused in (0, 1)
]

SCENES = {
    "two_clusters": (two_clusters, KW, {}),
    # the camera close to the chain's corner, so that rays pass through its deepest cells
    "nested": (nested, dict(KW, bvh_max_depth=20, bvh_leaf_object_count=1),
               dict(cam=np.float32([[1, 0, 0, 0.05], [0, 1, 0, 0.05], [0, 0, 1, -2.5], [0, 0, 0, 1]]), light=(1.5, 2.5, 0.0))),
}


@pytest.mark.parametrize("name", sorted(SCENES))
def test_full_blocks_and_deep_trees_equal_single_rays(cuda_lib, oracle, name):
    make, kw, where = SCENES[name]
    scene = make()
    base, base_st = render(cuda_lib, scene, kw, {api.RT_OPT_PACKETS: 0}, **where)
    assert base_st["primary_hits"] > 0 and base_st["shadow_rays"] > 0
    for opts in VARIANTS:
        img, st = render(cuda_lib, scene, kw, opts, **where)
        assert np.array_equal(img, base), (name, opts)
        for k in COUNTS:
            assert st[k] == base_st[k], (name, opts, k)
    common.assert_image_close(base, common.oracle_image(oracle, scene, kw, MATS, {}, **where), what=name)


def test_sixteen_bit_masks_follow_light_moves_through_frame_graphs(cuda_lib):
    """Light moves between frames that replay captured frame graphs, over blocks of 16 records: the same frames and counts
    as single rays, and as packets without the light cull."""
    scene = two_clusters()
    lights = [(3.0, 3.0, 2.0), (-2.0, 1.0, -1.0), (0.0, -3.0, -4.0), (3.0, 3.0, 2.0)]
    runs = []
    for packets, graph, cull in ((1, 1, 1), (1, 0, 0), (0, 0, 1)):
        r = common.product_renderer(cuda_lib, scene, KW, MATS, {})
        r.ctx.set_option(api.RT_OPT_PACKETS, packets)
        r.ctx.set_option(api.RT_OPT_GRAPH, graph)
        r.ctx.set_option(api.RT_OPT_LIGHT_CULL, cull)
        frames = []
        for light in lights:
            r.set_light_position(light)
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
