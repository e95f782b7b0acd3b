"""ctypes binding of the C ABI in include/rtb200.h (librtb200.so).

`load_library()` opens the CUDA library built by `raytracercpp_b200.build` and nothing else: if the shared
object is missing it raises, and `Context()` raises when no CUDA device is usable -- there is no CPU path.
(Tests may hand `Context` another handle that exports the same ABI -- the kernel emulation under tests/hostsim --
but the package itself never looks for one.)
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "librtb200.so"

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_STATE, RT_ERR_UNSUPPORTED = 0, -1, -2, -3, -4
RT_SHADING, RT_ABS_NORMALS_SHADING, RT_PASTEL_NORMALS_SHADING, RT_BARYCENTRIC_COORDINATES_SHADING, RT_VISUALIZE_AO = range(5)
RT_TEX_AO, RT_TEX_DIFFUSE, RT_TEX_NORMAL, RT_TEX_ROUGHNESS, RT_TEX_SKYSPHERE = range(5)
RT_TEX_SKYBOX_RIGHT, RT_TEX_SKYBOX_LEFT, RT_TEX_SKYBOX_TOP, RT_TEX_SKYBOX_BOTTOM, RT_TEX_SKYBOX_BACK, RT_TEX_SKYBOX_FRONT = range(5, 11)
RT_TEX_DISPLACEMENT = 11
RT_OPT_COUNT_WORK, RT_OPT_CHUNK_PIXELS, RT_OPT_LEAF_SPLIT, RT_OPT_REFILL_PRIMARY, RT_OPT_REFILL_SHADE, RT_OPT_TRI_BATCH, RT_OPT_PACKETS = 0, 1, 2, 3, 4, 5, 6
RT_OPT_PACKET_ROUNDS, RT_OPT_SCREEN_CULL, RT_OPT_LANES, RT_OPT_ITEM_ROUNDS, RT_OPT_PRIMARY_ROUNDS, RT_OPT_FUSED_ITEMS, RT_OPT_TOP_TABLE, RT_OPT_SHADOW_SORT, RT_OPT_DEVICE_BUILD, RT_OPT_ITEM_PASSES = 7, 8, 9, 10, 11, 12, 13, 14, 15, 16
RT_OPT_RASTER_UNITS, RT_OPT_GRAPH, RT_OPT_PACKET_CULL, RT_OPT_FAN_LANES, RT_OPT_LIGHT_CULL = 17, 18, 19, 20, 21


class RtError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rtb200 error {code}: {message}")
        self.code = code
        self.message = message


class RtMaterial(C.Structure):
    _fields_ = [("ambient_coeff", C.c_float * 3), ("diffuse", C.c_float * 3), ("specular", C.c_float * 3),
                ("emission", C.c_float * 3), ("reflection", C.c_float), ("roughness", C.c_float), ("ns", C.c_float),
                ("specular_threshold", C.c_float)]


SETTINGS_FIELDS = [
    "image_width", "image_height", "enable_ssaa", "ssaa_factor", "hybrid_rasterization_tracing", "shading_method",
    "compute_shadows", "max_recursion_depth", "enable_bvh", "bvh_max_depth", "bvh_leaf_object_count", "enable_ssao",
    "enable_ambient", "enable_diffuse", "enable_specular", "enable_emissive", "rough_reflections_sample_count",
    "enable_ao_mapping", "enable_diffuse_mapping", "enable_normal_mapping", "enable_displacement_mapping",
    "enable_roughness_mapping", "enable_skysphere", "enable_skybox",
]


class RtSettings(C.Structure):
    _fields_ = [(n, C.c_int32) for n in SETTINGS_FIELDS] + [("rng_seed", C.c_uint32), ("displacement_mapping_strength", C.c_float),
                                                              ("parallax_mapping_steps", C.c_int32),
                                                              ("ssao_sample_count", C.c_int32), ("ssao_radius", C.c_float), ("ssao_amount", C.c_float),
                                                             ("enable_clipping", C.c_int32)]

    def copy(self) -> "RtSettings":
        out = RtSettings()
        C.memmove(C.byref(out), C.byref(self), C.sizeof(RtSettings))
        return out


class RtRenderStats(C.Structure):
    _fields_ = [("primary_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("reflection_rays", C.c_uint64),
                ("reflection_shadow_rays", C.c_uint64), ("primary_hits", C.c_uint64), ("kernel_launches", C.c_uint32),
                ("device_ms", C.c_float), ("trace_primary_ms", C.c_float), ("shade_ms", C.c_float),
                ("reflect_ms", C.c_float), ("compact_ms", C.c_float), ("resolve_ms", C.c_float),
                ("primary_volume_tests", C.c_uint64), ("primary_triangle_tests", C.c_uint64),
                ("shadow_volume_tests", C.c_uint64), ("shadow_triangle_tests", C.c_uint64),
                ("reflection_volume_tests", C.c_uint64), ("reflection_triangle_tests", C.c_uint64),
                ("traced_primary_rays", C.c_uint64), ("primary_fetched_bytes", C.c_uint64), ("shadow_fetched_bytes", C.c_uint64),
                ("reflection_fetched_bytes", C.c_uint64)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}

    @property
    def total_rays(self) -> int:
        return self.primary_rays + self.shadow_rays + self.reflection_rays + self.reflection_shadow_rays

    @property
    def traced_rays(self) -> int:
        """Rays that were really traced: `total_rays` minus the samples written as misses without a ray (screen cull)."""
        return self.traced_primary_rays + self.shadow_rays + self.reflection_rays + self.reflection_shadow_rays

    @property
    def work_bytes(self) -> int:
        """56 B per 7-slab volume test + 36 B per triangle test (needs RT_OPT_COUNT_WORK)."""
        v = self.primary_volume_tests + self.shadow_volume_tests + self.reflection_volume_tests
        t = self.primary_triangle_tests + self.shadow_triangle_tests + self.reflection_triangle_tests
        return 56 * v + 36 * t


class RtBvhInfo(C.Structure):
    _fields_ = [("triangles", C.c_uint64), ("nodes", C.c_uint64), ("leaves", C.c_uint64), ("empty_leaves", C.c_uint64),
                ("interior", C.c_uint64), ("max_depth_reached", C.c_uint32), ("max_leaf_size", C.c_uint32),
                ("child_records", C.c_uint64), ("device_bytes", C.c_uint64), ("build_ms", C.c_double),
                ("upload_ms", C.c_double)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


FP, IP, UP, BP = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)

# name -> (restype, argtypes): every symbol include/rtb200.h declares
ABI = {
    "rt_default_settings": (None, [C.POINTER(RtSettings)]),
    "rt_pixel_seed": (C.c_uint32, [C.c_uint32, C.c_uint32]),
    "rt_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "rt_destroy": (None, [C.c_void_p]),
    "rt_last_error": (C.c_char_p, [C.c_void_p]),
    "rt_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_int64]),
    "rt_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rt_set_host_threads": (C.c_int, [C.c_int]),
    "rt_frame_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]),
    "rt_frame_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "rt_frame_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rt_frame_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rt_frame_to_host": (C.c_int, [C.c_void_p, C.c_void_p, UP, C.c_size_t]),
    "rt_set_triangles": (C.c_int, [C.c_void_p, FP, FP, IP, C.c_size_t]),
    "rt_build_bvh": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "rt_bvh_info": (C.c_int, [C.c_void_p, C.POINTER(RtBvhInfo)]),
    "rt_transform_triangles": (C.c_int, [C.c_void_p, FP, C.c_int, C.c_int]),
    "rt_set_materials": (C.c_int, [C.c_void_p, C.POINTER(RtMaterial), C.c_size_t]),
    "rt_set_texture_f32": (C.c_int, [C.c_void_p, C.c_int, FP, C.c_int, C.c_int]),
    "rt_set_texture_u8": (C.c_int, [C.c_void_p, C.c_int, BP, C.c_int, C.c_int]),
    "rt_clear_texture": (C.c_int, [C.c_void_p, C.c_int]),
    "rt_set_camera": (C.c_int, [C.c_void_p, FP, FP, FP]),
    "rt_set_projection": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float]),
    "rt_perspective_inverse": (None, [C.c_float, C.c_float, C.c_float, C.c_float, FP]),
    "rt_invert_transform": (None, [FP, FP]),
    "rt_transform_point": (None, [FP, FP, FP]),
    "rt_set_light": (C.c_int, [C.c_void_p, FP]),
    "rt_add_sphere": (C.c_int, [C.c_void_p, FP, C.c_float, C.c_int32]),
    "rt_add_plane": (C.c_int, [C.c_void_p, FP, FP, C.c_int32]),
    "rt_clear_analytic_shapes": (C.c_int, [C.c_void_p]),
    "rt_render": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), UP, C.POINTER(RtRenderStats)]),
    "rt_render_device": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(RtRenderStats)]),
    "rt_render_device_begin": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rt_render_device_end": (C.c_int, [C.c_void_p, C.POINTER(RtRenderStats)]),
    "rt_tile_count": (C.c_int, [C.POINTER(RtSettings), C.c_int, C.c_int, C.c_int]),
    "rt_pack_tiles": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rt_unpack_tiles": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rt_unpack_gathered": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rt_intersect": (C.c_int, [C.c_void_p, FP, FP, C.c_size_t, IP, FP, FP, FP]),
    "rt_occluded": (C.c_int, [C.c_void_p, FP, FP, C.c_size_t, BP]),
    "rt_generate_primary_rays": (C.c_int, [C.c_void_p, C.POINTER(RtSettings), FP, FP]),
    "rt_resolve_ssaa": (C.c_int, [C.c_void_p, UP, C.c_int, C.c_int, C.c_int, UP]),
    "rt_obj_load": (C.c_int, [C.c_char_p, FP, C.c_int32, C.POINTER(C.c_void_p), C.c_char_p, C.c_size_t]),
    "rt_obj_free": (None, [C.c_void_p]),
    "rt_obj_triangle_count": (C.c_size_t, [C.c_void_p]),
    "rt_obj_material_count": (C.c_size_t, [C.c_void_p]),
    "rt_obj_xyz9": (FP, [C.c_void_p]),
    "rt_obj_uv6": (FP, [C.c_void_p]),
    "rt_obj_material_indices": (IP, [C.c_void_p]),
    "rt_obj_materials": (C.POINTER(RtMaterial), [C.c_void_p]),
    "rt_obj_material_name": (C.c_char_p, [C.c_void_p, C.c_size_t]),
    "rt_precompute_materials": (None, [C.POINTER(RtMaterial), C.c_size_t]),
}


def bind(lib: C.CDLL) -> C.CDLL:
    for name, (res, args) in ABI.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    return lib


_LIB = None


def load_library(path=None) -> C.CDLL:
    """Opens raytracercpp_b200/librtb200.so (CUDA, sm_100a).  Raises if it has not been built.  `path` names another
    build of the same sources (kernel A/B experiments: python -m raytracercpp_b200.build --out ... -D...)."""
    global _LIB
    if path is not None:
        return bind(C.CDLL(str(path)))
    if _LIB is None:
        if not LIB_PATH.exists():
            raise FileNotFoundError(f"{LIB_PATH} is missing: run `python -m raytracercpp_b200.build` (needs nvcc). "
                                    "There is no CPU implementation to fall back to.")
        _LIB = bind(C.CDLL(str(LIB_PATH)))
    return _LIB


def default_settings(lib=None, **kw) -> RtSettings:
    lib = lib or load_library()
    s = RtSettings()
    lib.rt_default_settings(C.byref(s))
    for k, v in kw.items():
        if not hasattr(s, k):
            raise AttributeError(k)
        setattr(s, k, float(v) if k in ("displacement_mapping_strength", "ssao_radius", "ssao_amount") else int(v))
    return s


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def load_obj(path, transform=None, current_material_count=0, lib=None):
    """rt_obj_load: read_meshio_data + MeshIOUtils::create_triangles (mesh_io.cpp:426-591, utils/meshIOUtils.cpp:4-33).
    Returns (xyz9 [n, 9], uv6 [n, 6] or None, mat [n], materials as a list of dicts, material names)."""
    lib = lib or load_library()
    tr = _f32(transform).reshape(16) if transform is not None else None
    mesh, err = C.c_void_p(), C.create_string_buffer(512)
    rc = lib.rt_obj_load(str(path).encode(), tr.ctypes.data_as(FP) if tr is not None else None, int(current_material_count), C.byref(mesh), err, len(err))
    if rc != RT_OK:
        raise RtError(rc, err.value.decode(errors="replace"))
    try:
        n, nm = lib.rt_obj_triangle_count(mesh), lib.rt_obj_material_count(mesh)
        xyz9 = np.ctypeslib.as_array(lib.rt_obj_xyz9(mesh), shape=(n, 9)).copy()
        uvp = lib.rt_obj_uv6(mesh)
        uv6 = np.ctypeslib.as_array(uvp, shape=(n, 6)).copy() if uvp else None
        mat = np.ctypeslib.as_array(lib.rt_obj_material_indices(mesh), shape=(n,)).copy()
        mp = lib.rt_obj_materials(mesh)
        mats = [dict(ambient_coeff=tuple(mp[i].ambient_coeff), diffuse=tuple(mp[i].diffuse), specular=tuple(mp[i].specular),
                     emission=tuple(mp[i].emission), reflection=mp[i].reflection, roughness=mp[i].roughness, ns=mp[i].ns) for i in range(nm)]
        names = [lib.rt_obj_material_name(mesh, i).decode() for i in range(nm)]
    finally:
        lib.rt_obj_free(mesh)
    return xyz9, uv6, mat, mats, names


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def materials_array(mats):
    arr = (RtMaterial * max(len(mats), 1))()
    for i, m in enumerate(mats):
        for key in ("ambient_coeff", "diffuse", "specular", "emission"):
            v = m.get(key, (1.0, 1.0, 1.0) if key == "ambient_coeff" else (0.0, 0.0, 0.0))
            for j in range(3):
                getattr(arr[i], key)[j] = float(v[j])
        for key in ("reflection", "roughness", "ns", "specular_threshold"):
            setattr(arr[i], key, float(m.get(key, 0.0)))
    return arr


class Context:
    """One RtContext (one CUDA device).  Thin: every method is one C-ABI call."""

    def __init__(self, device: int = 0, lib=None):
        self.lib = lib or load_library()
        self.device = device
        h = C.c_void_p()
        rc = self.lib.rt_create(device, C.byref(h))
        if rc != RT_OK:
            raise RtError(rc, (self.lib.rt_last_error(None) or b"").decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.rt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != RT_OK:
            raise RtError(rc, (self.lib.rt_last_error(self.h) or b"").decode())

    def set_option(self, option: int, value: int):
        self._check(self.lib.rt_set_option(self.h, option, value))

    def set_stream(self, cuda_stream: int | None):
        self._check(self.lib.rt_set_stream(self.h, C.c_void_p(cuda_stream or 0)))

    # ---- scene ------------------------------------------------------------------------------------------
    def set_triangles(self, xyz9, uv6=None, mat=None):
        xyz9 = _f32(xyz9).reshape(-1, 9)
        uv6 = _f32(uv6).reshape(-1, 6) if uv6 is not None else None
        mat = np.ascontiguousarray(mat, dtype=np.int32) if mat is not None else None
        self._check(self.lib.rt_set_triangles(self.h, _p(xyz9, C.c_float), _p(uv6, C.c_float), _p(mat, C.c_int32), len(xyz9)))

    def build_bvh(self, max_depth=12, leaf_max=40) -> dict:
        self._check(self.lib.rt_build_bvh(self.h, max_depth, leaf_max))
        return self.bvh_info()

    def bvh_info(self) -> dict:
        info = RtBvhInfo()
        self._check(self.lib.rt_bvh_info(self.h, C.byref(info)))
        return info.as_dict()

    def transform_triangles(self, m16, max_depth=12, leaf_max=40):
        m = _f32(m16).reshape(16)
        self._check(self.lib.rt_transform_triangles(self.h, _p(m, C.c_float), max_depth, leaf_max))

    def set_materials(self, mats):
        self._check(self.lib.rt_set_materials(self.h, materials_array(mats), len(mats)))

    def set_texture(self, slot: int, rgba):
        rgba = np.ascontiguousarray(rgba)
        h, w = rgba.shape[:2]
        if rgba.dtype == np.uint8:
            self._check(self.lib.rt_set_texture_u8(self.h, slot, _p(rgba, C.c_uint8), w, h))
        else:
            rgba = _f32(rgba)
            self._check(self.lib.rt_set_texture_f32(self.h, slot, _p(rgba, C.c_float), w, h))

    def clear_texture(self, slot: int):
        self._check(self.lib.rt_clear_texture(self.h, slot))

    def set_camera(self, proj_inv, cam_to_world, position):
        a, b, c = _f32(proj_inv).reshape(16), _f32(cam_to_world).reshape(16), _f32(position).reshape(3)
        self._check(self.lib.rt_set_camera(self.h, _p(a, C.c_float), _p(b, C.c_float), _p(c, C.c_float)))

    def set_projection(self, fov, aspect, znear=0.1, zfar=1000.0):
        """Camera::_perspective_proj_mat / _fov / _aspect_ratio for the SSAO post-process (RtSettings.enable_ssao)."""
        self._check(self.lib.rt_set_projection(self.h, float(fov), float(aspect), float(znear), float(zfar)))

    def set_light(self, p):
        p = _f32(p).reshape(3)
        self._check(self.lib.rt_set_light(self.h, _p(p, C.c_float)))

    def add_sphere(self, center, radius, mat_index):
        c = _f32(center).reshape(3)
        self._check(self.lib.rt_add_sphere(self.h, _p(c, C.c_float), float(radius), int(mat_index)))

    def add_plane(self, point, normal, mat_index):
        p, n = _f32(point).reshape(3), _f32(normal).reshape(3)
        self._check(self.lib.rt_add_plane(self.h, _p(p, C.c_float), _p(n, C.c_float), int(mat_index)))

    def clear_analytic_shapes(self):
        self._check(self.lib.rt_clear_analytic_shapes(self.h))

    # ---- host helpers -----------------------------------------------------------------------------------
    def perspective_inverse(self, fov, aspect, znear=0.1, zfar=1000.0):
        out = np.zeros(16, np.float32)
        self.lib.rt_perspective_inverse(fov, aspect, znear, zfar, _p(out, C.c_float))
        return out.reshape(4, 4)

    def invert_transform(self, m):
        m = _f32(m).reshape(16)
        out = np.zeros(16, np.float32)
        self.lib.rt_invert_transform(_p(m, C.c_float), _p(out, C.c_float))
        return out.reshape(4, 4)

    def transform_point(self, m, p):
        m, p = _f32(m).reshape(16), _f32(p).reshape(3)
        out = np.zeros(3, np.float32)
        self.lib.rt_transform_point(_p(m, C.c_float), _p(p, C.c_float), _p(out, C.c_float))
        return out

    # ---- rendering --------------------------------------------------------------------------------------
    def render(self, settings: RtSettings, out=None):
        """rt_render: host ARGB32 [H, W] (row 0 = bottom row) + RtRenderStats."""
        if out is None:
            out = np.empty((settings.image_height, settings.image_width), np.uint32)
        stats = RtRenderStats()
        self._check(self.lib.rt_render(self.h, C.byref(settings), _p(out, C.c_uint32), C.byref(stats)))
        return out, stats

    def render_device(self, settings: RtSettings, d_ptr: int, tile_size=64, tile_mod=1, tile_rem=0):
        stats = RtRenderStats()
        self._check(self.lib.rt_render_device(self.h, C.byref(settings), C.c_void_p(d_ptr), tile_size, tile_mod, tile_rem, C.byref(stats)))
        return stats

    def render_device_begin(self, settings: RtSettings, d_ptr: int, tile_size=64, tile_mod=1, tile_rem=0):
        """Enqueues the frame and returns; render_device_end() waits for it and returns the stats."""
        self._check(self.lib.rt_render_device_begin(self.h, C.byref(settings), C.c_void_p(d_ptr), tile_size, tile_mod, tile_rem))

    def render_device_end(self) -> RtRenderStats:
        stats = RtRenderStats()
        self._check(self.lib.rt_render_device_end(self.h, C.byref(stats)))
        return stats

    def tile_count(self, settings, tile_size, tile_mod, tile_rem) -> int:
        n = self.lib.rt_tile_count(C.byref(settings), tile_size, tile_mod, tile_rem)
        if n < 0:
            raise RtError(n, "rt_tile_count")
        return n

    def pack_tiles(self, settings, d_frame: int, d_staging: int, tile_size, tile_mod, tile_rem):
        self._check(self.lib.rt_pack_tiles(self.h, C.byref(settings), C.c_void_p(d_frame), C.c_void_p(d_staging), tile_size, tile_mod, tile_rem))

    def unpack_gathered(self, settings, d_frame: int, d_gathered: int, tile_size, tile_mod, self_rem):
        self._check(self.lib.rt_unpack_gathered(self.h, C.byref(settings), C.c_void_p(d_frame), C.c_void_p(d_gathered), tile_size, tile_mod, self_rem))

    def unpack_tiles(self, settings, d_frame: int, d_staging: int, tile_size, tile_mod, tile_rem):
        self._check(self.lib.rt_unpack_tiles(self.h, C.byref(settings), C.c_void_p(d_frame), C.c_void_p(d_staging), tile_size, tile_mod, tile_rem))

    # ---- frames shared between the ranks of a box (rt_frame_*: CUDA IPC) ---------------------------------
    def frame_alloc(self, nbytes: int):
        """-> (device pointer, 64-byte handle) of a frame other ranks can map with frame_open."""
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        self._check(self.lib.rt_frame_alloc(self.h, nbytes, C.byref(ptr), handle))
        return ptr.value, bytes(handle)

    def frame_open(self, handle: bytes) -> int:
        ptr, buf = C.c_void_p(), (C.c_ubyte * 64).from_buffer_copy(handle)
        self._check(self.lib.rt_frame_open(self.h, buf, C.byref(ptr)))
        return ptr.value

    def frame_close(self, d_ptr: int):
        self._check(self.lib.rt_frame_close(self.h, C.c_void_p(d_ptr)))

    def frame_free(self, d_ptr: int):
        self._check(self.lib.rt_frame_free(self.h, C.c_void_p(d_ptr)))

    def frame_to_host(self, d_ptr: int, out: np.ndarray):
        """Device frame -> the (pageable) host array `out`, behind everything enqueued on the context's stream."""
        assert out.dtype == np.uint32 and out.flags.c_contiguous
        self._check(self.lib.rt_frame_to_host(self.h, C.c_void_p(d_ptr), _p(out, C.c_uint32), out.size))
        return out

    # ---- batch queries ----------------------------------------------------------------------------------
    def intersect(self, o3, d3):
        o3, d3 = _f32(o3).reshape(-1, 3), _f32(d3).reshape(-1, 3)
        n = len(o3)
        tri, t, u, v = np.empty(n, np.int32), np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.float32)
        self._check(self.lib.rt_intersect(self.h, _p(o3, C.c_float), _p(d3, C.c_float), n, _p(tri, C.c_int32), _p(t, C.c_float),
                                          _p(u, C.c_float), _p(v, C.c_float)))
        return tri, t, u, v

    def occluded(self, p3, n3):
        p3, n3 = _f32(p3).reshape(-1, 3), _f32(n3).reshape(-1, 3)
        out = np.empty(len(p3), np.uint8)
        self._check(self.lib.rt_occluded(self.h, _p(p3, C.c_float), _p(n3, C.c_float), len(p3), _p(out, C.c_uint8)))
        return out.astype(bool)

    def generate_primary_rays(self, settings):
        f = settings.ssaa_factor if settings.enable_ssaa else 1
        n = settings.image_width * f * settings.image_height * f
        o3, d3 = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
        self._check(self.lib.rt_generate_primary_rays(self.h, C.byref(settings), _p(o3, C.c_float), _p(d3, C.c_float)))
        return o3, d3

    def resolve_ssaa(self, argb, factor):
        argb = np.ascontiguousarray(argb, dtype=np.uint32)
        h, w = argb.shape
        out = np.empty((h // max(factor, 1), w // max(factor, 1)), np.uint32)
        self._check(self.lib.rt_resolve_ssaa(self.h, _p(argb, C.c_uint32), w, h, factor, _p(out, C.c_uint32)))
        return out
