"""Cuts the golden fixtures of tests/golden/ from the UNMODIFIED reference compiled in this container
(oracle/_ref/libref_strict.so = reference sources with -ffp-contract=off, oracle/_ref/libref.so = reference flags).

Run where the original sources are (export RTB200_REFERENCE=<RayTracerCPP>/tp2; make -C oracle ref):
    python tests/golden/make_golden.py
The .npz files are committed; the tests only read them.

Contents
  robot_scene.npz    robot.obj through the reference's own loader (read_meshio_data + MeshIOUtils::create_triangles,
                     Translation(0,-2,-4) = the GUI placement) : xyz9, uv6, mat, materials (RtMaterial rows)
  golden_rays.npz    20 000 seeded rays x BVH (12,40) and (10,8): tri id, t, u, v of BVH::intersect (strict build),
                     tri id of the reference-flag build
  golden_images.npz  cfg1/cfg2/cfg3 frames at reduced size from both builds, camera matrices, SSAA resolve vectors,
                     the 4 ray/triangle KATs of tp2/projets/tests.cpp:97-112 evaluated by the reference
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.bindings import CpuTracer, default_settings  # noqa: E402
from raytracercpp_b200 import scenes  # noqa: E402
from raytracercpp_b200.renderer import precompute_materials  # noqa: E402
from tests.conftest import require_reference  # noqa: E402

OUT = Path(__file__).resolve().parent
MAT_KEYS = ("ambient_coeff", "diffuse", "specular", "emission")


def mats_to_rows(mats):
    rows = np.zeros((len(mats), 16), np.float32)
    for i, m in enumerate(mats):
        rows[i, 0:3], rows[i, 3:6], rows[i, 6:9], rows[i, 9:12] = (m[k] for k in MAT_KEYS)
        rows[i, 12:16] = m["reflection"], m["roughness"], m["ns"], m.get("specular_threshold", 0.0)
    return rows


def golden_ray_set(n=20000, seed=123):
    rng = np.random.default_rng(seed)
    h = n // 2
    o1 = np.zeros((h, 3), np.float32)
    d1 = rng.normal(size=(h, 3)).astype(np.float32)
    d1[:, 2] = -np.abs(d1[:, 2]) * 3
    d1 /= np.linalg.norm(d1, axis=1, keepdims=True).astype(np.float32)
    o2 = (rng.uniform(-1.5, 1.5, size=(n - h, 3)) + np.array([0, -1, -4])).astype(np.float32)
    d2 = rng.normal(size=(n - h, 3)).astype(np.float32)        # un-normalised on purpose (reflection rays are, renderer.cpp:317)
    return np.concatenate([o1, o2]), np.concatenate([d1, d2])


def configs(mats):
    """name -> (settings kwargs, materials, textures)"""
    tex2 = {0: scenes.noise_texture((128, 128), 2), 1: scenes.noise_texture((128, 128), 1, "rgb"),
            2: scenes.normal_map_texture((128, 128), 4), 3: scenes.noise_texture((128, 128), 3)}
    mats3 = [dict(m) for m in mats]
    mats3[0].update(reflection=0.9, roughness=0.0, specular=(0.2, 0.2, 0.2), diffuse=(0.5, 0.5, 0.5))   # load_obj override, QT/mainwindow.cpp:259-262
    mats3[1].update(reflection=0.5, roughness=0.4)
    mats3 = precompute_materials(mats3)
    tex3 = {3: tex2[3], 4: scenes.sky_texture((128, 256))}
    mats_shapes = mats3 + precompute_materials([
        dict(ambient_coeff=(1, 1, 1), diffuse=(0.2, 0.6, 0.3), specular=(0.4, 0.4, 0.4), emission=(0, 0, 0), reflection=0.0, roughness=0.0, ns=30.0),
        dict(ambient_coeff=(1, 1, 1), diffuse=(0.7, 0.7, 0.8), specular=(0.6, 0.6, 0.6), emission=(0, 0, 0), reflection=0.6, roughness=0.3, ns=80.0)])
    return {
        "cfg1": (dict(image_width=320, image_height=180, compute_shadows=1), mats, {}),
        "cfg2": (dict(image_width=160, image_height=90, compute_shadows=1, enable_ssaa=1, ssaa_factor=2, enable_ao_mapping=1,
                      enable_diffuse_mapping=1, enable_normal_mapping=1), mats, tex2),
        "cfg3": (dict(image_width=240, image_height=135, compute_shadows=1, rough_reflections_sample_count=16, max_recursion_depth=1,
                      enable_roughness_mapping=1, enable_skysphere=1, rng_seed=7), mats3, tex3),
        "cfg3_mirror5": (dict(image_width=160, image_height=90, compute_shadows=1, max_recursion_depth=5, enable_skysphere=1), mats3, tex3),
        # parallax occlusion mapping on top of cfg2's maps (renderer.cpp:518-554)
        "cfg2_pom": (dict(image_width=160, image_height=90, compute_shadows=1, enable_ao_mapping=1, enable_diffuse_mapping=1, enable_normal_mapping=1,
                          enable_displacement_mapping=1, displacement_mapping_strength=0.05, parallax_mapping_steps=16), mats,
                     {**tex2, 11: scenes.noise_texture((96, 96), 9)}),
        # analytic shapes of the GUI (QT/mainwindow.cpp:828,883,914,930): a ground plane, a mirror sphere, a matte sphere, with the
        # robot's own mirror materials; materials len(mats3) and len(mats3)+1 are appended for them
        "cfg3_shapes": (dict(image_width=200, image_height=112, compute_shadows=1, max_recursion_depth=2, enable_skysphere=1), mats_shapes,
                        {4: tex3[4], "shapes": [("plane", (0, -2, 0), (0, 1, 0), len(mats3)), ("sphere", (1.4, -1.2, -3.5), 0.5, len(mats3) + 1),
                                                ("sphere", (-1.6, -1.5, -3.0), 0.4, len(mats3))]}),
        # the GUI's default miss shader (QT/mainwindow.cpp:45-46): cube-map skybox, seen directly and in mirror reflections
        "cfg3_skybox": (dict(image_width=200, image_height=112, compute_shadows=1, max_recursion_depth=2, enable_skybox=1), mats3,
                       {5 + i: scenes.noise_texture((48 + 8 * i, 40 + 4 * i), 20 + i, "rgb") for i in range(6)}),
    }


def render_with(tracer, scene, kw, mats, tex, fov=80.0, seeded=False):
    s = default_settings(**kw)
    r = tracer.renderer()
    r.configure(s, fov)
    r.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
    r.set_materials(mats)
    r.set_light([3, 3, 2])
    for slot, img in tex.items():
        if slot == "shapes":
            for sh in img:
                (r.add_sphere if sh[0] == "sphere" else r.add_plane)(sh[1], sh[2], sh[3])
        else:
            r.set_texture(slot, img)
    if seeded:
        sup, _ = r.trace_rows()
        f = s.ssaa_factor if s.enable_ssaa else 1
        return tracer.downscale(sup, f) if f > 1 else sup
    img, _ = r.render()
    return img


def main():
    ref = require_reference()
    strict, fma = CpuTracer("ref_strict"), CpuTracer("ref")
    T = np.eye(4, dtype=np.float32)
    T[1, 3], T[2, 3] = -2, -4
    xyz9, uv6, mat, mats = strict.load_obj(str(ref / "data" / "Robot" / "robot.obj"), T)
    mats = precompute_materials(mats)
    np.savez_compressed(OUT / "robot_scene.npz", xyz9=xyz9, uv6=uv6, mat=mat, materials=mats_to_rows(mats))
    scene = dict(xyz9=xyz9, uv6=uv6, mat=mat)

    o, d = golden_ray_set()
    rays = dict(o=o, d=d)
    for (depth, leaf) in ((12, 40), (10, 8)):
        bs, bf = strict.bvh(xyz9, depth, leaf), fma.bvh(xyz9, depth, leaf)
        tri, t, u, v = bs.intersect(o, d)
        tag = f"_{depth}_{leaf}"
        rays.update({"tri" + tag: tri, "t" + tag: t, "u" + tag: u, "v" + tag: v, "tri_fma" + tag: bf.intersect(o, d)[0]})
        st = bs.stats()
        rays["stats" + tag] = np.array([st[k] for k in ("nodes", "leaves", "empty_leaves", "interior", "max_depth_reached", "max_leaf_size")], np.int64)
    np.savez_compressed(OUT / "golden_rays.npz", **rays)

    imgs = {}
    for name, (kw, m, tex) in configs(mats).items():
        seeded = name.startswith("cfg3")
        imgs[name + "_strict"] = render_with(strict, scene, kw, m, tex, seeded=seeded)
        imgs[name + "_fma"] = render_with(fma, scene, kw, m, tex, seeded=seeded)
    p, pi = strict.camera_matrices(80.0, 16.0 / 9.0)
    imgs["proj_80_16x9"], imgs["proj_inv_80_16x9"] = p, pi
    p, pi = strict.camera_matrices(45.0, 1.0)
    imgs["proj_inv_45_1"] = pi
    m = np.array([[0.8, -0.1, 0.2, 1.0], [0.3, 0.9, -0.2, -2.0], [-0.1, 0.25, 1.1, 0.5], [0, 0, 0, 1]], np.float32)
    imgs["inv_in"], imgs["inv_out"] = m, strict.transform_inverse(m)
    rng = np.random.default_rng(5)
    sup = (rng.integers(0, 1 << 24, size=(24, 36), dtype=np.uint32) | np.uint32(0xff000000))
    imgs["resolve_in"] = sup
    for f in (2, 3, 4):
        imgs[f"resolve_out_{f}"] = strict.downscale(sup, f)
    # KATs of tests.cpp:97-112 (all four must be misses) + two hits for good measure
    tris = np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0], [0, 0, 0, 1, 0, 0, 0, 1, 0], [1, -1, -9, -1, -1, -9, -1, -1, -11],
                     [-1, 1, -11, -1, 1, -9, 1, 1, -9], [0, 0, 0, 1, 0, 0, 0, 1, 0], [-1, -1, -5, 1, -1, -5, 0, 1, -5]], np.float32)
    ro = np.array([[0, 0, -1], [-2, 0, -1], [0, 0, 0], [0, 0, 0], [0.25, 0.25, 1], [0, 0, 0]], np.float32)
    rd = np.array([[0, 0, 1], [0, 0, 1], [-0.577350259, 0.577350259, -0.577350259], [-0.577350259, 0.577350259, -0.577350259],
                   [0, 0, -1], [0.05, 0.1, -1]], np.float32)
    res = [strict.triangle_intersect(tris[i], ro[i], rd[i]) for i in range(len(tris))]
    imgs["kat_tris"], imgs["kat_o"], imgs["kat_d"] = tris, ro, rd
    imgs["kat_hit"] = np.array([r[0] for r in res])
    imgs["kat_tuv"] = np.array([[r[1], r[2], r[3]] for r in res], np.float32)
    np.savez_compressed(OUT / "golden_images.npz", **imgs)
    for f in ("robot_scene.npz", "golden_rays.npz", "golden_images.npz"):
        print(f, (OUT / f).stat().st_size, "bytes")
    print("kat hits:", imgs["kat_hit"])


if __name__ == "__main__":
    main()
