"""The load half of the GUI's load -> upload path: csrc/scene_io.cpp (rt_obj_load, rt_precompute_materials) against what the
reference's own loader makes of the same files -- read_meshio_data + MeshIOUtils::create_triangles, tp2/src/mesh_io.cpp:426-591,
tp2/projets/utils/meshIOUtils.cpp:4-33 -- bit for bit: from the committed goldens (tests/golden/make_golden_obj.py), from
robot_scene.npz (the reference's loader on its own robot.obj), and live where the reference is mounted."""
from pathlib import Path

import numpy as np
import pytest

from raytracercpp_b200 import api
from raytracercpp_b200.renderer import precompute_materials
from tests.conftest import REFERENCE

GOLDEN = Path(__file__).resolve().parent / "golden"
REF_DATA = REFERENCE / "data" if REFERENCE is not None else None


def reference_file(rel):
    path = REF_DATA / rel if REF_DATA is not None else None
    if path is None or not path.exists():
        pytest.skip("reference data not here (RTB200_REFERENCE)")
    return path


@pytest.fixture(scope="module")
def lib():
    return api.load_library()


def material_rows(mats):
    return np.float32([list(m["ambient_coeff"]) + list(m["diffuse"]) + list(m["specular"]) + list(m["emission"]) +
                       [m["reflection"], m["roughness"], m["ns"]] for m in mats]).reshape(len(mats), 15)


@pytest.mark.parametrize("name", ["fixture_uv", "fixture_plain"])
def test_obj_fixture_matches_reference_loader(lib, name):
    g = np.load(GOLDEN / "golden_obj.npz")
    tr = g["transform"] if name == "fixture_uv" else None
    xyz9, uv6, mat, mats, names = api.load_obj(GOLDEN / "obj" / (name + ".obj"), tr, lib=lib)
    assert np.array_equal(xyz9, g[name + "_xyz9"])
    assert np.array_equal(mat, g[name + "_mat"])
    if name == "fixture_uv":
        assert np.array_equal(uv6, g[name + "_uv6"])
        assert names == ["Red", "Shiny", "default"]            # "default" is appended by the first face without a usemtl
        assert set(mat.tolist()) == {0, 1, 2}                  # the unknown material name falls back to "default" too (mesh_io.cpp:519-520)
    else:
        assert uv6 is None and mats == [] and (mat == -1).all()
        assert (g[name + "_uv6"] == -1).all()                  # the reference's Triangle keeps its (-1, -1, -1) defaults
    assert np.array_equal(material_rows(mats), g[name + "_materials"])


def test_material_offset_and_errors(lib, tmp_path):
    a = api.load_obj(GOLDEN / "obj" / "fixture_uv.obj", lib=lib)
    b = api.load_obj(GOLDEN / "obj" / "fixture_uv.obj", current_material_count=7, lib=lib)   # a second mesh appended to 7 materials
    assert np.array_equal(b[2], a[2] + 7) and np.array_equal(a[0], b[0])
    with pytest.raises(api.RtError) as e:
        api.load_obj(tmp_path / "missing.obj", lib=lib)
    assert e.value.code == api.RT_ERR_INVALID and "missing.obj" in e.value.message
    bad = tmp_path / "bad.obj"
    bad.write_text("v 0 0 0\nv 1 0\n")                         # a position with two numbers: the reference stops there too
    with pytest.raises(api.RtError):
        api.load_obj(bad, lib=lib)
    nomtl = tmp_path / "nomtl.obj"
    nomtl.write_text("mtllib nowhere.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    with pytest.raises(api.RtError):
        api.load_obj(nomtl, lib=lib)


def test_robot_scene_fixture_is_what_the_loader_gives(lib, robot):
    """tests/golden/robot_scene.npz was cut with the reference's loader from its robot.obj at the GUI's placement,
    Translation(0, -2, -4) (QT/mainwindow.cpp:308-312); where that file is mounted the native loader must give the same."""
    path = reference_file("Robot/robot.obj")
    tr = np.float32([[1, 0, 0, 0], [0, 1, 0, -2], [0, 0, 1, -4], [0, 0, 0, 1]])
    xyz9, uv6, mat, mats, names = api.load_obj(path, tr, lib=lib)
    assert np.array_equal(xyz9, robot["xyz9"]) and np.array_equal(uv6, robot["uv6"]) and np.array_equal(mat, robot["mat"])
    want = robot["materials"]
    assert len(mats) == len(want)
    for m, w in zip(precompute_materials(mats), want):
        for k in ("ambient_coeff", "diffuse", "specular", "emission"):
            assert tuple(np.float32(m[k])) == tuple(np.float32(w[k]))
        assert np.float32(m["ns"]) == np.float32(w["ns"])


@pytest.mark.parametrize("rel", ["Robot/robot.obj", "Geometry/geometry.obj", "cube.obj"])
def test_reference_data_live(lib, ref_strict, rel):
    path = reference_file(rel)
    tr = np.float32([[0.02, 0, 0, -1], [0, 0.02, 0, -3], [0, 0, 0.02, -13], [0, 0, 0, 1]])
    xyz9, uv6, mat, mats, _ = api.load_obj(path, tr, lib=lib)
    rx, ruv, rmat, rmats = ref_strict.load_obj(str(path), tr)
    assert np.array_equal(xyz9, rx) and np.array_equal(mat, rmat)
    if uv6 is not None:
        assert np.array_equal(uv6, ruv)
    assert np.array_equal(material_rows(mats), material_rows(rmats))


def test_precompute_materials(lib):
    import ctypes as C
    rng = np.random.default_rng(4)
    mats = [dict(ambient_coeff=(1, 1, 1), diffuse=(0.3, 0.3, 0.3), specular=tuple(rng.uniform(0.01, 1.0, 3)), emission=(0, 0, 0),
                 reflection=0.0, roughness=0.0, ns=float(rng.uniform(1, 300))) for _ in range(64)]
    arr = api.materials_array(mats)
    lib.rt_precompute_materials(arr, len(mats))
    want = precompute_materials(mats)                          # the numpy restatement of QT/mainwindow.cpp:240-249
    got = np.float32([arr[i].specular_threshold for i in range(len(mats))])
    # std::pow(float, float) is libm's powf here as in the reference; numpy's float32 power is its own routine: one ulp apart at most
    assert np.abs(got.view(np.int32) - np.float32([w["specular_threshold"] for w in want]).view(np.int32)).max() <= 1
    assert ((got > 0) & (got < 1)).all()


def test_adapter_load_obj(hostsim_lib):
    """Renderer.load_obj = MainWindow::load_obj (QT/mainwindow.cpp:251-282) on the native loader: the GUI's overrides of
    material 0, materials appended after the ones already there, precomputed thresholds -- then a frame."""
    import raytracercpp_b200 as rt
    r = rt.Renderer(0, hostsim_lib)
    s = r.render_settings()
    s.image_width, s.image_height, s.compute_shadows = 48, 32, 1
    r.change_render_size(48, 32)
    r.change_camera_fov(80.0)
    r.load_obj(GOLDEN / "obj" / "fixture_uv.obj")
    mats = r.get_materials()
    assert len(mats) == 3 and mats[0]["reflection"] == np.float32(0.9) and mats[0]["diffuse"] == (0.5, 0.5, 0.5) and mats[1]["reflection"] == 0.0
    assert all("specular_threshold" in m for m in mats)
    r.ray_trace()
    first = r.get_image().copy()
    background = 0xff000000 | (135 << 16) | (206 << 8) | 235
    assert (first != background).mean() > 0.05
    r.load_obj(GOLDEN / "obj" / "fixture_uv.obj", np.float32([[1, 0, 0, 0.5], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]]))
    assert len(r.get_materials()) == 6                      # appended, indices offset by the 3 already there
    r.ray_trace()
    assert (r.get_image() != first).any()
    r.close()


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_random_obj_files_live(lib, ref_strict, tmp_path, seed):
    """Randomly written OBJ + MTL files (polygons of 3-7 vertices, the four vertex forms, negative indices, CRLF lines,
    comments, materials switched back and forth, faces before any usemtl, unknown material names, several mtllib lines)
    through the native loader and through the compiled reference's loader: the same triangles, texture coordinates,
    material indices and material table.  Files either carry texture coordinates on every face vertex or on none -- the
    reference reads past its texcoord array when a file mixes the two."""
    rng = np.random.default_rng(seed)
    with_uv = bool(seed % 2)
    n_pos, n_tex, n_nrm = int(rng.integers(8, 40)), int(rng.integers(4, 20)), int(rng.integers(1, 6))
    eol = "\r\n" if seed % 3 == 0 else "\n"
    names = ["alpha", "beta gamma", "delta"]
    mtl = ["# materials" + eol]
    for k, nm in enumerate(names):
        mtl.append(f"newmtl {nm}{eol}")
        for key in ("Ka", "Kd", "Ks", "Ke")[: int(rng.integers(1, 5))]:
            mtl.append(f"  {key} " + " ".join(f"{x:.6f}" for x in rng.uniform(0, 1, 3)) + eol)
        if k != 1:
            mtl.append(f"Ns {rng.uniform(1, 400):.3f}{eol}")
        mtl.append(f"Ni 1.45{eol}d 1.0{eol}illum 2{eol}map_Kd tex_{k}.png{eol}")
    (tmp_path / "m.mtl").write_text("".join(mtl))
    lines = ["# random mesh" + eol]
    if seed != 4:
        lines.append("mtllib m.mtl" + eol)                     # seed 4: no material library at all
    pos_written = tex_written = nrm_written = 0

    def emit_vertices(count):
        nonlocal pos_written, tex_written, nrm_written
        for _ in range(count):
            lines.append("v " + " ".join(f"{x:.5f}" for x in rng.uniform(-2, 2, 3)) + eol)
            pos_written += 1
        for _ in range(max(1, count // 2)):
            lines.append("vt " + " ".join(f"{x:.5f}" for x in rng.uniform(0, 1, 2)) + eol)
            tex_written += 1
        lines.append("vn " + " ".join(f"{x:.5f}" for x in rng.normal(size=3)) + eol)
        nrm_written += 1

    emit_vertices(n_pos)
    for f in range(int(rng.integers(10, 40))):
        if rng.random() < 0.25:
            lines.append(f"usemtl {names[int(rng.integers(0, 3))] if rng.random() < 0.85 else 'nobody'}{eol}")
        if rng.random() < 0.2:
            emit_vertices(int(rng.integers(1, 5)))
        if rng.random() < 0.1:
            lines.append("# a comment" + eol + eol)
        verts = []
        for _ in range(int(rng.integers(3, 8))):
            p = int(rng.integers(1, pos_written + 1))
            t = int(rng.integers(1, tex_written + 1))
            n = int(rng.integers(1, nrm_written + 1))
            if rng.random() < 0.3:
                p, t, n = p - pos_written - 1, t - tex_written - 1, n - nrm_written - 1     # the same vertices, counted from the end
            form = int(rng.integers(0, 2))
            if with_uv:
                verts.append(f"{p}/{t}/{n}" if form else f"{p}/{t}")
            else:
                verts.append(f"{p}//{n}" if form else f"{p}")
        lines.append(("f " if rng.random() < 0.8 else "f   ") + " ".join(verts) + ("  " if rng.random() < 0.3 else "") + eol)
    path = tmp_path / "mesh.obj"
    path.write_text("".join(lines))
    tr = np.float32([[0.7, 0.1, 0, 0.3], [0, 1.1, 0.2, -1], [0.1, 0, 0.9, -5], [0, 0, 0, 1]])
    xyz9, uv6, mat, mats, _ = api.load_obj(path, tr, current_material_count=2, lib=lib)
    rx, ruv, rmat, rmats = ref_strict.load_obj(str(path), tr)
    assert len(xyz9) == len(rx) > 10
    assert np.array_equal(xyz9, rx) and np.array_equal(mat, rmat + 2)
    assert (uv6 is not None) == with_uv
    if with_uv:
        assert np.array_equal(uv6, ruv)
    assert np.array_equal(material_rows(mats), material_rows(rmats))
