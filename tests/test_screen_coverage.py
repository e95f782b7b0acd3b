"""The screen coverage of the primary packets (rtb200.cu: screen_coverage, RT_OPT_SCREEN_CULL): one bit per 8x4 block of the
supersampled frame, set when the block's rays can reach a box of a set whose union holds the scene (the upper levels of the
wide tree).  Blocks without the bit, and tiles without any, are written as misses without a ray.

The CPU test restates primary_ray (rt_device.h) in numpy float32, in the kernels' operation order, and checks the library's
bitmap (rt_screen_coverage, a host-only entry point) against exact float64 ray/box tests of those float32 rays: no sample whose
ray meets a box may lie in an uncovered block -- for random cameras near and far from scenes translated up to 1e5, tiny boxes,
boxes that straddle the camera plane or hold the camera, frame widths that are not multiples of 8 and SSAA factors 1-4.  With
the margin scaled to zero the same check fails.  The GPU tests render with the cull on and off: frames and ray / hit counters
must be identical."""
import ctypes as C

import numpy as np
import pytest

import raytracercpp_b200 as rt
from raytracercpp_b200 import api, build, scenes
from tests import common

F = np.float32


@pytest.fixture(scope="module")
def covlib():
    build.build()
    lib = C.CDLL(str(api.LIB_PATH))
    FP = C.POINTER(C.c_float)
    lib.rt_screen_coverage.restype = C.c_int
    lib.rt_screen_coverage.argtypes = [FP, FP, FP, C.c_int, C.c_int, FP, C.c_size_t, C.c_double, C.POINTER(C.c_uint32), C.c_size_t]
    lib.rt_perspective_inverse.restype = None
    lib.rt_perspective_inverse.argtypes = [C.c_float, C.c_float, C.c_float, C.c_float, FP]
    return lib


def perspective_inverse(lib, fov, aspect, near=0.1, far=1000.0):
    out = np.zeros(16, F)
    lib.rt_perspective_inverse(fov, aspect, near, far, out.ctypes.data_as(C.POINTER(C.c_float)))
    return out.reshape(4, 4)


def coverage(lib, pinv, c2w, pos, rw, rh, boxes, margin_scale=1.0):
    words = (((rw + 7) // 8) + 31) // 32
    bits = np.zeros(words * ((rh + 3) // 4), np.uint32)
    fp = lambda a: np.ascontiguousarray(a, F).ctypes.data_as(C.POINTER(C.c_float))
    pinv, c2w, pos, boxes = (np.ascontiguousarray(a, F) for a in (pinv, c2w, pos, boxes))
    rc = lib.rt_screen_coverage(fp(pinv), fp(c2w), fp(pos), rw, rh, fp(boxes), len(boxes), margin_scale,
                                bits.ctypes.data_as(C.POINTER(C.c_uint32)), bits.size)
    assert rc in (0, 1)
    return rc == 1, bits.reshape(-1, words)


def block_bits(bits, px, py):
    w = bits[py >> 2, px >> 8]
    return ((w >> ((px >> 3) & 31).astype(np.uint32)) & 1).astype(bool)


def xform_point(m, p):
    """rt_math.h: xform_point, vectorised, float32, left to right without FMA."""
    out = [((m[i, 0] * p[..., 0] + m[i, 1] * p[..., 1]) + m[i, 2] * p[..., 2]) + m[i, 3] for i in range(4)]
    wt = out[3]
    with np.errstate(divide="ignore", invalid="ignore"):
        w = np.where(wt == F(1), F(1), F(1) / wt)
    return np.stack([np.where(wt == F(1), out[i], out[i] * w) for i in range(3)], -1)


def primary_rays(pinv, c2w, pos, rw, rh, px, py):
    """rt_device.h: primary_ray, vectorised, float32."""
    yw = (py.astype(F) + F(0.5)) / F(rh) * F(2) - F(1)
    xw = (px.astype(F) + F(0.5)) / F(rw) * F(2) - F(1)
    vs = xform_point(pinv, np.stack([xw, yw, np.full_like(xw, F(-1))], -1))
    ws = xform_point(c2w, vs)
    v = ws - pos
    kk = F(1) / np.sqrt((v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]) + v[..., 2] * v[..., 2])
    return kk[..., None] * v


def ray_meets_box(o, d, lo, hi):
    """Exact (float64) slab test of the rays o + t d, t >= 0, against the closed box [lo, hi]."""
    o, d = o.astype(np.float64), d.astype(np.float64)
    tn = np.zeros(d.shape[:-1])
    tf = np.full(d.shape[:-1], np.inf)
    for k in range(3):
        with np.errstate(divide="ignore", invalid="ignore"):
            a, b = (float(lo[k]) - o[k]) / d[..., k], (float(hi[k]) - o[k]) / d[..., k]
        par = d[..., k] == 0
        inside = (lo[k] <= o[k]) & (o[k] <= hi[k])
        a = np.where(par, -np.inf if inside else np.inf, a)
        b = np.where(par, np.inf, b)                                     # outside the slab: tn = inf
        tn = np.maximum(tn, np.minimum(a, b))
        tf = np.minimum(tf, np.maximum(a, b))
    return tn <= tf


def rotation(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def random_case(lib, rng, offset, far):
    """A camera looking at a cluster of boxes around `offset` from near (a few units) or far (hundreds)."""
    factor = int(rng.integers(1, 5))
    w, h = int(rng.integers(40, 97)), int(rng.integers(30, 71))
    rw, rh = w * factor, h * factor
    R = rotation(rng)
    centre = np.asarray(offset, np.float64) + rng.normal(size=3)
    dist = 10.0 ** rng.uniform(2, 2.7) if far else 10.0 ** rng.uniform(-0.3, 0.8)
    cam = centre + R[:, 2] * dist                                      # the camera looks down its -z axis
    c2w = np.eye(4)
    c2w[:3, :3], c2w[:3, 3] = R, cam
    c2w = c2w.astype(F)
    pos = c2w[:3, 3].copy()
    pinv = perspective_inverse(lib, float(rng.uniform(30, 80)), rw / rh)
    n = int(rng.integers(1, 24))
    kind = rng.choice(4, n, p=[0.6, 0.04, 0.16, 0.2])
    scale = dist * 10.0 ** rng.uniform(-4, -0.5, (n, 1))
    c = centre + rng.normal(size=(n, 3)) * dist * 0.3
    half = scale * rng.uniform(0.05, 1.0, (n, 3))
    c[kind == 1] = cam + rng.normal(size=(int((kind == 1).sum()), 3)) * 1e-3 * dist   # around the camera
    c[kind == 2] = cam - R[:, 2] * dist * 0.5 + rng.normal(size=(int((kind == 2).sum()), 3)) * 0.05 * dist
    half[kind == 3] = dist * 1e-6                                        # tiny
    lo, hi = (c - half).astype(F), (c + half).astype(F)
    straddle = rng.uniform(size=n) < 0.05                                 # crosses the camera plane off to the side
    if straddle.any():
        side = cam + R[:, 0] * dist * 0.5
        lo[straddle] = np.minimum(lo[straddle], (side - R[:, 2] * dist).astype(F))
        hi[straddle] = np.maximum(hi[straddle], (side + R[:, 2] * dist).astype(F))
    boxes = np.concatenate([lo, hi], 1)
    return pinv, c2w, pos, rw, rh, boxes


def violations(lib, case, margin_scale):
    pinv, c2w, pos, rw, rh, boxes = case
    bound, bits = coverage(lib, pinv, c2w, pos, rw, rh, boxes, margin_scale)
    if not bound:
        return None, 0, 1.0
    py, px = np.mgrid[0:rh, 0:rw]
    px, py = px.ravel(), py.ravel()
    d = primary_rays(pinv, c2w, pos, rw, rh, px, py)
    o = pos.astype(np.float64)
    hit = np.zeros(px.size, bool)
    for b in boxes:
        hit |= ray_meets_box(o, d, b[:3], b[3:])
    cov = block_bits(bits, px, py)
    return bound, int((hit & ~cov).sum()), float(cov.mean())


@pytest.mark.parametrize("offset", [0.0, 1e3, 1e4, 1e5])
@pytest.mark.parametrize("far", [False, True])
def test_no_ray_that_meets_a_box_lands_in_an_uncovered_block(covlib, offset, far):
    rng = np.random.default_rng(int(offset) % 997 + 31 * far)
    bounded, partial = 0, 0
    for _ in range(16):
        case = random_case(covlib, rng, (offset, -0.5 * offset, 0.25 * offset), far)
        bound, bad, frac = violations(covlib, case, 1.0)
        assert bad == 0, (offset, far, case[3:5])
        bounded += bool(bound)
        partial += bool(bound) and frac < 0.9
    # a bound exists for most cameras ...  (not 1e5 from the origin: there a float32 direction built from a near plane 0.1 away
    # is off by more than the rounding bounds allow, and every block is traced)
    assert bounded >= 8 or offset >= 1e5
    if offset <= 1e3:
        assert partial >= 4                                             # ... and it culls where the rounding allows it


def test_the_margin_is_needed(covlib):
    """With the margin scaled to zero, float32 rays that meet a box land in blocks the bitmap leaves out."""
    rng = np.random.default_rng(5)
    bad = 0
    for offset, far in ((1e4, False), (1e5, False), (1e5, True), (0.0, False)):
        for _ in range(12):
            bound, v, _ = violations(covlib, random_case(covlib, rng, (offset, -0.5 * offset, 0.25 * offset), far), 0.0)
            bad += v
    assert bad > 0


def test_bitmap_layout_and_special_cases(covlib):
    lib = covlib
    pinv = perspective_inverse(lib, 45.0, 1.5)
    c2w, pos = np.eye(4, dtype=F), np.zeros(3, F)
    # nothing to hit: a bound, no bit
    bound, bits = coverage(lib, pinv, c2w, pos, 123, 77, np.zeros((0, 6), F))
    assert bound and bits.shape == (20, 1) and not bits.any()
    # a box that holds the camera, or straddles its plane: every block
    for box in ([-1, -1, -1, 1, 1, 1], [5, -1, -1, 6, 1, 1]):
        bound, bits = coverage(lib, pinv, c2w, pos, 123, 77, np.float32([box]))
        py, px = np.mgrid[0:77, 0:123]
        assert bound and block_bits(bits, px.ravel(), py.ravel()).all()
    # a box straight ahead: a block rectangle around the centre, nothing else
    bound, bits = coverage(lib, pinv, c2w, pos, 123, 77, np.float32([[-0.1, -0.1, -5.1, 0.1, 0.1, -4.9]]))
    py, px = np.mgrid[0:77, 0:123]
    cov = block_bits(bits, px.ravel(), py.ravel()).reshape(77, 123)
    assert bound and cov[38, 61] and not cov[0, 0] and not cov[76, 122] and 0.001 < cov.mean() < 0.2
    # the empty boxes the builder writes for the nodes it leaves out of the set, (+inf, -inf), hold nothing ...
    inf = np.inf
    empty = [inf, inf, inf, -inf, -inf, -inf]
    bound2, bits2 = coverage(lib, pinv, c2w, pos, 123, 77, np.float32([empty, [-0.1, -0.1, -5.1, 0.1, 0.1, -4.9], empty]))
    assert bound2 and np.array_equal(bits, bits2)
    # ... while a box with an infinite bound may hold anything: every block
    bound3, bits3 = coverage(lib, pinv, c2w, pos, 123, 77, np.float32([[-0.1, -0.1, -inf, 0.1, 0.1, -4.9]]))
    assert bound3 and block_bits(bits3, px.ravel(), py.ravel()).all()
    # an orthographic projection_inverse: its rays do not leave from the camera, no bound
    ortho = np.eye(4, dtype=F)
    assert not coverage(lib, ortho, c2w, pos, 123, 77, np.float32([[-0.1, -0.1, -5.1, 0.1, 0.1, -4.9]]))[0]


# ---- GPU: frames and counters with the cull on and off ------------------------------------------------------------------

KEYS = ("primary_rays", "primary_hits", "shadow_rays", "reflection_rays")


def render_both(lib, scene, kw, mats, tex, cams, transform=None, **k):
    """Frames and stats of one renderer per cull setting over a sequence of cameras (graphs get captured and replayed)."""
    out = {}
    for cull in (1, 0):
        r = common.product_renderer(lib, scene, kw, mats, tex, **k)
        r.ctx.set_option(api.RT_OPT_SCREEN_CULL, cull)
        seq = []
        for i, cam in enumerate(cams):
            if transform is not None and i == transform[0]:
                r.ctx.transform_triangles(transform[1])
            if cam is not None:
                r.set_camera_transform(cam)
            r.ray_trace()
            seq.append((r.get_image().copy(), r.last_stats().as_dict()))
        r.close()
        out[cull] = seq
    for i, ((a, sa), (b, sb)) in enumerate(zip(out[1], out[0])):
        assert np.array_equal(a, b), i
        for key in KEYS:
            assert sa[key] == sb[key], (i, key)
    return out


def cam_at(x, y, z, yaw=0.0):
    c, s = np.cos(yaw), np.sin(yaw)
    return np.float32([[c, 0, s, x], [0, 1, 0, y], [-s, 0, c, z], [0, 0, 0, 1]])


@pytest.mark.gpu
def test_robot_cameras_and_camera_moves(cuda_lib, robot):
    table = common.config_table(robot["materials"])
    cams = [cam_at(0, 0, 0), cam_at(1.5, -0.5, -1.0, 0.9), cam_at(0, -1.5, -3.9), cam_at(0, 0, 2.0, np.pi), cam_at(3, 2, 4),
            cam_at(0, 0, 0), cam_at(0, 0, 0), cam_at(0, 0, 0), cam_at(3, 2, 4), cam_at(3, 2, 4), cam_at(3, 2, 4), cam_at(0, 0, 0)]
    for name in ("cfg1", "cfg3", "cfg3_skybox"):
        kw, mats, tex = table[name]
        render_both(cuda_lib, robot, dict(kw, image_width=160, image_height=90), mats, tex, cams)


@pytest.mark.gpu
def test_robot_far_from_the_origin_with_a_close_camera(cuda_lib, robot):
    table = common.config_table(robot["materials"])
    kw, mats, tex = table["cfg1"]
    off = np.float32([1e4, -3e3, 5e3])
    scene = dict(robot, xyz9=(robot["xyz9"].reshape(-1, 3) + off).reshape(robot["xyz9"].shape).astype(F))
    cams = [cam_at(*(off + np.float32([0.0, -1.0, -2.5]))), cam_at(*(off + np.float32([0.3, -1.2, -3.0])), 0.4),
            cam_at(*(off + np.float32([0.0, -1.5, -3.9])))]
    render_both(cuda_lib, scene, dict(kw, image_width=200, image_height=120), mats, tex, cams, light=tuple(off + np.float32([3, 3, 2])))


@pytest.mark.gpu
def test_sphere_and_hair_and_fewer_traced_rays_than_the_root_rectangle(cuda_lib):
    mats = rt.precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
    kw = dict(image_width=320, image_height=180, enable_ssaa=1, ssaa_factor=2, compute_shadows=1)
    xyz9, uv6, mat = scenes.displaced_sphere(200, 400)
    sphere = dict(xyz9=xyz9, uv6=uv6, mat=mat)
    out = render_both(cuda_lib, sphere, kw, mats, {}, [None, cam_at(0.4, 0.2, 0.5, 0.1), None])
    # the root box's screen rectangle, without any margin, holds fewer samples than the cull traces with it
    v = xyz9.reshape(-1, 3).astype(np.float64)
    lo, hi = v.min(0), v.max(0)
    corners = np.array([[hi[0] if c & 1 else lo[0], hi[1] if c & 2 else lo[1], hi[2] if c & 4 else lo[2]] for c in range(8)])
    t = np.tan(np.radians(common.FOV) / 2)
    rw, rh = 640, 360
    x = (-corners[:, 0] / corners[:, 2]) / (t * rw / rh)
    y = (-corners[:, 1] / corners[:, 2]) / t
    rect = ((min(1, x.max()) - max(-1, x.min())) / 2 * rw) * ((min(1, y.max()) - max(-1, y.min())) / 2 * rh)
    st = out[1][0][1]
    assert 0 < st["primary_hits"] <= st["traced_primary_rays"] < rect, (st["traced_primary_rays"], rect)
    xyz9, uv6, mat = scenes.hair_ball(n_strands=2000, segments=8, width=4.0e-3)
    render_both(cuda_lib, dict(xyz9=xyz9, uv6=uv6, mat=mat), kw, mats, {}, [None, cam_at(0.2, 0.1, -1.0, 0.2)])


@pytest.mark.gpu
def test_transform_then_rebuild(cuda_lib, robot):
    table = common.config_table(robot["materials"])
    kw, mats, tex = table["cfg1"]
    m = np.float32([[1, 0, 0, 0.7], [0, 1, 0, 0.3], [0, 0, 1, -0.5], [0, 0, 0, 1]])
    render_both(cuda_lib, robot, dict(kw, image_width=160, image_height=90), mats, tex, [None, None, None, None], transform=(2, m))


@pytest.mark.gpu
def test_tile_shards(cuda_lib, robot):
    import torch
    table = common.config_table(robot["materials"])
    kw, mats, tex = table["cfg1"]
    kw = dict(kw, image_width=200, image_height=120)
    frames = {}
    for cull in (1, 0):
        r = common.product_renderer(cuda_lib, robot, kw, mats, tex, cam=cam_at(0.8, -0.5, -1.0, 0.5))
        r.ctx.set_option(api.RT_OPT_SCREEN_CULL, cull)
        r.ray_trace()
        s = r.render_settings()
        got = []
        for mod in (3, 4):
            for rem in range(mod):
                for _ in range(3):                                       # the third frame replays a graph
                    shard = torch.full((120, 200), 0x5a5a5a5a, dtype=torch.int32, device="cuda")
                    st = r.ctx.render_device(s, shard.data_ptr(), 24, mod, rem)
                torch.cuda.synchronize()
                got.append((shard.cpu().numpy().copy(), tuple(getattr(st, k) for k in KEYS)))
        r.close()
        frames[cull] = got
    for (a, sa), (b, sb) in zip(frames[1], frames[0]):
        assert np.array_equal(a, b) and sa == sb
