"""Asset ingestion and display — the rows next to the hot path (SURVEY.md §8f #2, #4): the OBJ loader that feeds the BVH
builder, and the Display.shader / screenshot path behind the accumulated image."""
import os

import numpy as np
import pytest

from conftest import CUDA_LIB, ORACLE_LIB, render
import ray_tracing_b200 as rt
from ray_tracing_b200 import scenes

OBJ = """# two faces: a quad with v/vt/vn corners and a triangle with v//vn corners
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
v 2 0 1
vn 0 0 1
vn 0 1 0
vt 0 0
f 1/1/1 2/1/1 3/1/1 4/1/1
f 2//2 5//2 3//2
"""


def test_obj_loader_quads_handedness_and_vertex_split(tmp_path):
    p = tmp_path / "m.obj"
    p.write_text(OBJ)
    v, idx, n = rt.load_obj(str(p), unity_handedness=False)
    assert idx.size == 9                                          # quad -> 2 triangles, + 1
    assert v.shape == (7, 3)                                      # vertices 2 and 3 are used with two different normals
    assert idx[:6].tolist() == [0, 1, 2, 0, 2, 3]                 # fan triangulation
    vu, iu, nu = rt.load_obj(str(p), unity_handedness=True)
    assert np.array_equal(vu[:, 0], -v[:, 0]) and np.array_equal(vu[:, 1:], v[:, 1:])     # X negated
    assert iu[:3].tolist() == [0, 2, 1]                           # winding reversed
    # orientation is preserved by the pair of flips: cross(B-A, C-A) keeps pointing along the (mirrored) authored normal
    a, b, c = vu[iu[0]], vu[iu[1]], vu[iu[2]]
    assert np.dot(np.cross(b - a, c - a), nu[iu[0]]) > 0           # geometric face vector still agrees with the (mirrored) normal
    a0, b0, c0 = v[idx[0]], v[idx[1]], v[idx[2]]
    assert np.dot(np.cross(b0 - a0, c0 - a0), n[idx[0]]) > 0
    tris, nodes, st = rt.build_bvh(vu, iu, nu)
    assert st["TriangleCount"] == 3


def test_obj_loader_without_normals_and_errors(tmp_path):
    p = tmp_path / "n.obj"
    p.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    v, idx, n = rt.load_obj(str(p), unity_handedness=False)
    assert np.allclose(n, [[0, 0, 1]] * 3)                        # area-weighted face normal
    bad = tmp_path / "bad.obj"
    bad.write_text("v 0 0 0\nf 1 2 3\n")
    with pytest.raises(ValueError):
        rt.load_obj(str(bad))
    with pytest.raises(ValueError):
        rt.load_obj(str(tmp_path / "missing.obj"))


@pytest.fixture(scope="module")
def reference_assets(tmp_path_factory):
    """The original project's Assets: its five scenes and their meshes, cut down (tests/golden/make_reference_excerpt.py)."""
    from test_round2_abi import extract_reference_excerpt
    return extract_reference_excerpt(tmp_path_factory.mktemp("reference"))


DRAGON_TRIANGLES = 2588             # Dragon_80K.obj (87,130 triangles) decimated; same silhouette


def test_reference_dragon_loads_and_traces(oracle_path, reference_assets):
    v, idx, n = rt.load_obj(os.path.join(reference_assets, "Graphics", "Dragon_80K.obj"))
    assert idx.size // 3 == DRAGON_TRIANGLES
    tris, nodes, st = rt.build_bvh(v, idx, n)
    assert st["TriangleCount"] == DRAGON_TRIANGLES and st["LeafDepthMax"] <= 32
    mesh = scenes.MeshDesc(v, idx, n)
    l2w, w2l = scenes.trs(position=(-0.58, 1.37, 0.09), euler_deg=(0, 59.33, 0), scale=(4.98, 4.98, 4.98))   # Glass Dragon.unity:2075-2088
    sc = scenes.Scene(name="dragon", width=48, height=27, meshes=[mesh],
                      models=[scenes.ModelDesc(0, l2w, w2l, scenes.material(emission=(1, 1, 1), emissionStrength=1.0, specularProbability=0.0))],
                      cam_local_to_world=scenes.trs(position=(0, 1.9, -5.67))[0], fov=54.5, settings=dict(maxBounceCount=1))
    frame, _ = render(oracle_path, sc)
    lit = frame[..., :3].sum(-1) > 0
    assert 0.05 < lit.mean() < 0.6                                # the dragon covers part of the view


def test_display_divides_by_frame_and_encodes_srgb(oracle_path):
    sc = scenes.cornell_spheres(32, 24, 3, 2)
    mgr = rt.RayComputeManager(oracle_path)
    scenes.apply(sc, mgr)
    mgr.OnEnable()
    for _ in range(3):
        mgr.RenderFrame()
    acc = mgr.accumulatedResult
    disp = rt.RayTraceDisplay(mgr)
    img = disp.OnRenderImage()
    assert img.shape == (24, 32, 4) and img.dtype == np.uint8
    # reference semantics incl. its off-by-one: sum of 3 frames / numAccumulatedFrames (= 4)   (SURVEY.md §3.4)
    lin = np.clip(acc[::-1, :, :3] / 4.0, 0, 1).astype(np.float64)
    srgb = np.where(lin <= 0.0031308, 12.92 * lin, 1.055 * np.power(lin, 1 / 2.4) - 0.055)
    assert np.abs(img[..., :3].astype(np.int32) - np.floor(srgb * 255 + 0.5).astype(np.int32)).max() <= 1
    assert np.all(img[..., 3] == np.floor(np.clip(3 / 4.0, 0, 1) ** (1 / 2.4) * 1.055 * 255 - 0.055 * 255 + 0.5))   # alpha = 3/4
    p = os.path.join(os.path.dirname(oracle_path), "_screenshot_test.png")
    try:
        disp.save_screenshot(p)
        assert open(p, "rb").read(8) == b"\x89PNG\r\n\x1a\n"
    finally:
        if os.path.exists(p):
            os.remove(p)


@pytest.mark.gpu
def test_display_matches_oracle_on_gpu():
    sc = scenes.knot_room(96, 54, max_bounces=4, rays_per_pixel=2, nu=80, nv=8)
    outs = []
    for lib in (ORACLE_LIB, CUDA_LIB):
        mgr = rt.RayComputeManager(lib)
        scenes.apply(sc, mgr)
        mgr.OnEnable()
        mgr.RenderFrame(); mgr.RenderFrame()
        outs.append(rt.RayTraceDisplay(mgr).OnRenderImage())
        mgr.accumulate = False
        outs.append(rt.RayTraceDisplay(mgr).OnRenderImage())       # not accumulating: the frame image with Frame = 1
        mgr.OnDestroy()
    assert np.array_equal(outs[0], outs[2]) and np.array_equal(outs[1], outs[3])


# ---- the reference's serialized scenes (Unity YAML) ---------------------------------------------------------------------------

def test_exr_export_is_lossless(tmp_path, oracle_path):
    """The float4 accumulation buffer through write_exr / read_exr: bit-identical, NaN and inf included; header fields as the format wants."""
    _, accum = render(oracle_path, scenes.cornell_spheres(37, 21, 3, 2), frames=2)
    img = accum[::-1].copy()                                       # display orientation: row 0 = top
    img[0, 0] = (np.nan, np.inf, -np.inf, -0.0)
    p = str(tmp_path / "a.exr")
    rt.write_exr(p, img)
    back = rt.read_exr(p)
    assert back.shape == img.shape and np.array_equal(back.view(np.uint32), img.view(np.uint32))
    raw = open(p, "rb").read()
    assert raw[:4] == bytes([0x76, 0x2F, 0x31, 0x01]) and b"channels\x00chlist\x00" in raw and b"compression\x00compression\x00\x01\x00\x00\x00\x00" in raw
    assert len(raw) > 21 * (8 + 37 * 16)                        # 21 scan-line blocks of 8 + 4 channels x 37 floats, plus header and offset table
    with pytest.raises(ValueError):
        rt.write_exr(p, np.zeros((4, 4, 3), np.float32))


def test_builtin_unity_meshes():
    from ray_tracing_b200 import unity_scene
    cube, quad = unity_scene.builtin_cube(), unity_scene.builtin_quad()
    assert cube.triangle_count == 12 and cube.vertices.shape == (24, 3) and np.abs(cube.vertices).max() == 0.5
    for t in range(12):                                            # outward-facing: cross(B-A, C-A) along the vertex normal and away from the centre
        a, b, c = (cube.vertices[cube.indices[3 * t + k]] for k in range(3))
        n = np.cross(b - a, c - a)
        assert np.dot(n, cube.normals[cube.indices[3 * t]]) > 0 and np.dot(n, a + b + c) > 0
    assert quad.triangle_count == 2 and np.allclose(quad.normals, [[0, 0, -1]] * 4)


def test_reference_scenes_load_with_the_serialized_settings(oracle_path, reference_assets):
    from ray_tracing_b200 import unity_scene
    SCENES_DIR = os.path.join(reference_assets, "Scenes")
    expect = {   # SURVEY.md Appendix B
        "Glass Dragon": dict(models=11, bounces=10, fov=54.5, cam=(0.0, 1.9, -5.67), diverge=1.5, defocus=0.0),
        "Glass Balls": dict(models=17, bounces=10, fov=60.0, cam=(0.0, 1.99, -5.895), diverge=1.5, defocus=0.0),
        "Sphere Refract": dict(models=10, bounces=32, fov=38.0, cam=(0.0, 1.28, -11.65), diverge=1.5, defocus=100.0),
    }
    for name, e in expect.items():
        sc = unity_scene.load_unity_scene(os.path.join(SCENES_DIR, name + ".unity"), width=64, height=36)
        assert len(sc.models) == e["models"] and sc.settings["maxBounceCount"] == e["bounces"] and sc.fov == e["fov"]
        assert np.allclose(sc.cam_local_to_world[:3, 3], e["cam"], atol=1e-3)
        assert sc.settings["divergeStrength"] == e["diverge"] and sc.settings["defocusStrength"] == e["defocus"]
    assert sc.settings["focusDistance"] == pytest.approx(5.3)      # Sphere Refract: depth of field
    # Glass Dragon: the dragon mesh is the shipped OBJ, glass, as serialized (Glass Dragon.unity:1988-2073)
    sc = unity_scene.load_unity_scene(os.path.join(SCENES_DIR, "Glass Dragon.unity"), width=64, height=36)
    dragon = [m for m in sc.models if sc.meshes[m.mesh].triangle_count == DRAGON_TRIANGLES]
    assert len(dragon) == 1 and int(dragon[0].material["flag"]) == scenes.MAT_GLASS and float(dragon[0].material["ior"]) == 1.5
    assert np.allclose(np.linalg.norm(dragon[0].local_to_world[:3, 0]), 4.98, atol=1e-2)
    sc.settings["numRaysPerPixel"] = 16
    frame, _ = render(oracle_path, sc)
    assert np.isfinite(frame).all() and (frame[..., :3].sum(-1) > 0).mean() > 0.1


# ---- binary FBX (Text.fbx / Water.fbx of the reference) -----------------------------------------------------------------------

def _fbx_node(name, props=b"", nprops=0, children=b"", version=7400):
    """One FBX node record (32-bit offsets); the caller fixes up the absolute end offset."""
    return (name.encode(), nprops, props, children)


def _write_fbx(path, tree, version=7400):
    import struct
    wide = version >= 7500
    out = bytearray(b"Kaydara FBX Binary  \x00\x1a\x00" + struct.pack("<I", version))
    null = b"\x00" * (25 if wide else 13)

    def emit(node):
        name, nprops, props, children = node
        start = len(out)
        out.extend(b"\x00" * (24 if wide else 12)); out.append(len(name)); out.extend(name); out.extend(props)
        for c in children:
            emit(c)
        if children:
            out.extend(null)
        struct.pack_into("<QQQ" if wide else "<III", out, start, len(out), nprops, len(props))
    for n in tree:
        emit(n)
    out.extend(null)
    out.extend(b"\x00" * 200)                                      # footer padding
    open(path, "wb").write(bytes(out))


def _p_str(s):
    import struct
    b = s.encode()
    return b"S" + struct.pack("<I", len(b)) + b


def _p_arr(code, arr, deflate):
    import struct, zlib
    raw = arr.tobytes()
    body = zlib.compress(raw) if deflate else raw
    return code.encode() + struct.pack("<III", arr.size, 1 if deflate else 0, len(body)) + body


def _p_i64(v):
    import struct
    return b"L" + struct.pack("<q", v)


@pytest.mark.parametrize("version", [7400, 7500])
def test_fbx_reader_on_a_synthetic_file(tmp_path, version):
    """Container (both offset widths, raw and deflated arrays), polygon end markers, fan triangulation, ByPolygonVertex /
    IndexToDirect normals, node-name ownership through Connections, Unity handedness."""
    from ray_tracing_b200 import fbx_mesh
    verts = np.array([0, 0, 0, 1, 0, 0, 1, 1, 0, 0, 1, 0, 2, 0, 1], dtype="<f8")
    pvi = np.array([0, 1, 2, ~3, 1, 4, ~2], dtype="<i4")            # a quad and a triangle
    normals = np.array([0, 0, 1, 0, 1, 0], dtype="<f8")
    nidx = np.array([0, 0, 0, 0, 1, 1, 1], dtype="<i4")
    layer = _fbx_node("LayerElementNormal", children=[
        _fbx_node("MappingInformationType", _p_str("ByPolygonVertex"), 1), _fbx_node("ReferenceInformationType", _p_str("IndexToDirect"), 1),
        _fbx_node("Normals", _p_arr("d", normals, False), 1), _fbx_node("NormalsIndex", _p_arr("i", nidx, True), 1)])
    geom = _fbx_node("Geometry", _p_i64(77) + _p_str("geo\x00\x01Geometry") + _p_str("Mesh"), 3, children=[
        _fbx_node("Vertices", _p_arr("d", verts, True), 1), _fbx_node("PolygonVertexIndex", _p_arr("i", pvi, False), 1), layer])
    model = _fbx_node("Model", _p_i64(88) + _p_str("Sign.001\x00\x01Model") + _p_str("Mesh"), 3)
    conns = _fbx_node("Connections", children=[_fbx_node("C", _p_str("OO") + _p_i64(88) + _p_i64(0), 3), _fbx_node("C", _p_str("OO") + _p_i64(77) + _p_i64(88), 3)])
    path = tmp_path / "t.fbx"
    _write_fbx(str(path), [_fbx_node("Objects", children=[geom, model]), conns], version)
    meshes = fbx_mesh.load_fbx_meshes(str(path))
    (fid, (name, m)), = meshes.items()
    assert name == "Sign.001" and fid == fbx_mesh.unity_mesh_file_id("Sign.001")
    assert m.triangle_count == 3
    tri = m.vertices.reshape(3, 3, 3)
    assert np.array_equal(tri[0], [[-1, 1, 0], [-1, 0, 0], [0, 0, 0]])          # (0,1,2) reversed, X negated
    assert np.array_equal(tri[1], [[0, 1, 0], [-1, 1, 0], [0, 0, 0]])           # (0,2,3) reversed
    assert np.array_equal(m.normals[:6], [[0, 0, 1]] * 6) and np.array_equal(m.normals[6:], [[0, 1, 0]] * 3)
    a, b, c = tri[0]
    assert np.dot(np.cross(b - a, c - a), m.normals[0]) > 0                     # orientation survives the two flips
    # recomputed normals (normalImportMode 1): flat faces more than the smoothing angle apart keep their own face normal
    calc = fbx_mesh.load_fbx_meshes(str(path), normal_import_mode=1, smooth_angle_deg=30.0)[fid][1]
    assert np.allclose(calc.normals[:6], [[0, 0, 1]] * 6, atol=1e-6)
    assert np.allclose(np.linalg.norm(calc.normals, axis=1), 1.0, atol=1e-6)
    with pytest.raises(ValueError):
        (tmp_path / "ascii.fbx").write_text("; FBX 7.4.0 project file\n")
        fbx_mesh.load_fbx_meshes(str(tmp_path / "ascii.fbx"))


def test_unity_mesh_file_ids_known_answers():
    """XXH64 against its published test vectors, and the sub-asset ids the reference's scenes store for its two .fbx files
    (Text.unity:317-5749, Splash.unity) — fileID = XXH64("Type:Mesh->" + name + "0")."""
    from ray_tracing_b200 import fbx_mesh
    assert fbx_mesh.xxh64(b"") == 0xEF46DB3751D8E999 and fbx_mesh.xxh64(b"abc") == 0x44BC2CF5AD770999
    assert fbx_mesh.xxh64(b"Nobody inspects the spammish repetition") == 0xFBCEA83C8A378BF1
    pinned = {"Text": 6686097678407549244, "Text.001": 4882115322962003972, "Text.002": 2210965410299338194, "Text.003": -7432939776326845586,
              "Text.004": 3038654674045518180, "Text.005": -3932407843921001191, "Text.006": 552887423116881197, "Text.007": -5082522871635176651,
              "Text.008": -8413837161920484157, "Text.009": -1661537731292281231, "waterTest2": 1552480332205418273}
    for name, fid in pinned.items():
        assert fbx_mesh.unity_mesh_file_id(name) == fid, name


def test_reference_fbx_scenes_load_and_trace(oracle_path, reference_assets):
    """Text.unity (ten glyph meshes of Text.fbx, normals recomputed as its .meta asks) and Splash.unity (Water.fbx, bvhQuality Low),
    with every geometry of both files cut to its first polygons plus the ones that hold its extreme vertices: every mesh id resolves,
    the geometry sits inside the room, the scene traces."""
    from ray_tracing_b200 import unity_scene
    SCENES_DIR = os.path.join(reference_assets, "Scenes")
    sc = unity_scene.load_unity_scene(os.path.join(SCENES_DIR, "Text.unity"), width=64, height=36)
    glyphs = sorted(m.triangle_count for m in sc.meshes if m.triangle_count not in (2, 12, DRAGON_TRIANGLES))
    assert glyphs == [100, 101, 107, 114, 116, 120, 121, 123, 124, 126] and len(sc.models) == 18      # the ten glyph meshes of Text.fbx
    for md in sc.models:
        m = sc.meshes[md.mesh]
        w = (md.local_to_world[:3, :3] @ m.vertices.T.astype(np.float64)).T + md.local_to_world[:3, 3]
        assert w[:, 0].min() > -3.1 and w[:, 0].max() < 3.1 and w[:, 1].min() > -0.2 and w[:, 1].max() < 4.2      # inside the 5.6 x 4 room
    sc.settings.update(numRaysPerPixel=16, maxBounceCount=8)
    frame, _ = render(oracle_path, sc)
    assert np.isfinite(frame).all() and (frame[..., :3].sum(-1) > 0).mean() > 0.05     # one small ceiling light: a dark, noisy room
    sp = unity_scene.load_unity_scene(os.path.join(SCENES_DIR, "Splash.unity"), width=48, height=27)
    water = [m for m in sp.models if sp.meshes[m.mesh].triangle_count == 1505]
    assert len(water) == 1 and sp.settings["bvhQuality"] == 0
    m = sp.meshes[water[0].mesh]
    w = (water[0].local_to_world[:3, :3] @ m.vertices.T.astype(np.float64)).T + water[0].local_to_world[:3, 3]
    assert np.allclose(w.min(0), [-3.95, -0.04, -1.93], atol=0.02) and np.allclose(w.max(0), [3.95, 5.85, 2.02], atol=0.02)   # fills the room wall to wall
