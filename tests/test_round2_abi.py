"""Round 2 additions to the C-ABI, checked without a GPU on the SIMT interpreter build of the product's own sources (tests/simt)
and on the oracle: the multi-GPU group context (rtCreateMulti: tiles + the per-frame exchange inside rtDispatch), and the
hardening items of the round-1 review (modelCount set on its own, root bounds the reference never reads, trees deeper than the
traversal stacks, unchanged per-frame uploads).  The same bodies run against librt_b200.so under `-m gpu`
(tests/test_gpu_round2_abi.py)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ORACLE_LIB, REPO, assert_bit_equal, render
import ray_tracing_b200 as rt
from ray_tracing_b200 import capi, scenes
from ray_tracing_b200.capi import NODE_DTYPE, TRIANGLE_DTYPE

sys.path.insert(0, os.path.join(REPO, "tests", "simt"))
import build as simt_build   # noqa: E402


@pytest.fixture(scope="session")
def simt_lib():
    return simt_build.build()


# ---- bodies shared with the GPU file (lib = any library with the ABI) -----------------------------------------------------------

def group_equals_single(lib, devices, sc, frames=2, options=None):
    """ONE manager on several devices (rtCreateMulti) renders the image one device renders, bit for bit; its statistics are the sums."""
    fref, aref, sref = render(lib, sc, frames=frames, want_stats=True, options=options)
    mgr = rt.RayComputeManager(lib, devices=devices)
    scenes.apply(sc, mgr)
    ctx = mgr.context
    for k, v in (options or {}).items():
        ctx.set_option(k, v)
    mgr.OnEnable()
    ctx.reset_stats()
    for _ in range(frames):
        mgr.RenderFrame()
    st = ctx.stats()
    assert_bit_equal(mgr.raytraceFrameTex, fref, f"group of {len(devices)}: FrameRender")
    assert_bit_equal(mgr.accumulatedResult, aref, f"group of {len(devices)}: AccumulatedRender")
    assert st["rays"] == sref["rays"]
    # a different band height is a layout choice only
    ctx.set_tile(0, len(devices), 3)
    mgr.ResetAccumulatedRender()
    for _ in range(frames):
        mgr.RenderFrame()
    assert_bit_equal(mgr.accumulatedResult, aref, "bands of 3 rows")
    with pytest.raises(capi.RtError):
        ctx.set_tile(1, len(devices), 8)                     # a group is rank 0 of its own GPU count
    mgr.OnDestroy()


def one_model_scene(width=48, height=32, nu=40, nv=8):
    sc = scenes.knot_room(width, height, 3, 2, nu=nu, nv=nv)
    sc.models = sc.models[:1]
    sc.meshes = sc.meshes[:1]
    sc.settings = dict(sc.settings, useSky=True)
    return sc


def model_count_alone(lib):
    """ADVICE (high): rtSetInt("modelCount") without re-sending ModelInfo must re-plan the scene (pair plan, roots, DevModel array)."""
    sc = scenes.knot_room(48, 32, 3, 1, nu=30, nv=6)
    out = {}
    for name, path in (("oracle", ORACLE_LIB), ("lib", lib)):
        for kernel in ((None,) if name == "oracle" else (0, 1, 2)):
            mgr = rt.RayComputeManager(path)
            scenes.apply(sc, mgr)
            ctx = mgr.context
            if kernel is not None:
                ctx.set_option("kernel", kernel)
            mgr.OnEnable()
            imgs = []
            for count in (1, 3, 2, 3):
                ctx.set_int("modelCount", count)
                ctx.dispatch_full(0)
                imgs.append(mgr.raytraceFrameTex.copy())
            out[(name, kernel)] = imgs
            mgr.OnDestroy()
    for kernel in (0, 1, 2):
        for i, (a, b) in enumerate(zip(out[("lib", kernel)], out[("oracle", None)])):
            assert_bit_equal(a, b, f"kernel {kernel}, modelCount step {i}")
    assert not np.array_equal(out[("oracle", None)][0], out[("oracle", None)][1])      # the count does change the picture


def root_bounds_are_never_read(lib):
    """ADVICE (medium): the reference pushes the root unconditionally and tests child boxes only (RayCommon.hlsl:241-270); a Nodes
    buffer whose root carries a far-away placeholder box renders the same with model skipping and with the TLAS."""
    sc = one_model_scene()
    m = sc.meshes[0]
    _, nodes, _ = rt.build_bvh(m.vertices, m.indices, m.normals, "High")
    bad = nodes.copy()
    bad["boundsMin"][0] = (1e6, 1e6, 1e6)
    bad["boundsMax"][0] = (1e6 + 1, 1e6 + 1, 1e6 + 1)

    def run(path, options):
        mgr = rt.RayComputeManager(path)
        scenes.apply(sc, mgr)
        ctx = mgr.context
        for k, v in options.items():
            ctx.set_option(k, v)
        mgr.OnEnable()
        ctx.set_buffer("Nodes", bad)
        mgr.ResetAccumulatedRender()
        mgr.RenderFrame(); mgr.RenderFrame()
        a = mgr.accumulatedResult.copy()
        mgr.OnDestroy()
        return a
    ref = run(ORACLE_LIB, {})
    good = render(ORACLE_LIB, sc, frames=2)[1]
    assert_bit_equal(ref, good, "the oracle itself does not read the root's bounds")
    assert (ref[..., :3] != good[..., :3]).sum() == 0 and np.count_nonzero(ref[..., :3]) > 0
    for opts in ({"kernel": 0}, {"kernel": 1}, {"kernel": 2}, {"kernel": 1, "tlas": 1}, {"kernel": 2, "tlas": 1}, {"kernel": 2, "modelSkip": 0}):
        assert_bit_equal(run(lib, opts), ref, f"placeholder root box, {opts}")


def chain_bvh(depth):
    """A degenerate tree: every inner node has a one-triangle leaf and the next inner node; `depth` levels of inner nodes."""
    tris = np.zeros(depth + 1, dtype=TRIANGLE_DTYPE)
    for i in range(depth + 1):
        x = -2.0 + 4.0 * i / depth
        tris["posA"][i] = (x, 0.2, 0.0); tris["posB"][i] = (x + 0.03, 1.8, 0.0); tris["posC"][i] = (x + 0.06, 0.2, 0.0)
        tris["normA"][i] = tris["normB"][i] = tris["normC"][i] = (0, 0, -1)
    nodes = np.zeros(2 * depth + 1, dtype=NODE_DTYPE)
    lo = np.minimum(np.minimum(tris["posA"], tris["posB"]), tris["posC"]); hi = np.maximum(np.maximum(tris["posA"], tris["posB"]), tris["posC"])
    for level in range(depth):                                   # inner node `level` at index 0 (root) or 2 * level
        idx = 0 if level == 0 else 2 * level
        nodes["startIndex"][idx] = 2 * level + 1                 # children at 2*level+1 (leaf), 2*level+2 (next inner / last leaf)
        nodes["triangleCount"][idx] = 0
        nodes["boundsMin"][idx] = lo[level:].min(axis=0); nodes["boundsMax"][idx] = hi[level:].max(axis=0)
        leaf = 2 * level + 1
        nodes["startIndex"][leaf] = level; nodes["triangleCount"][leaf] = 1
        nodes["boundsMin"][leaf] = lo[level]; nodes["boundsMax"][leaf] = hi[level]
    last = 2 * depth
    nodes["startIndex"][last] = depth; nodes["triangleCount"][last] = 1
    nodes["boundsMin"][last] = lo[depth]; nodes["boundsMax"][last] = hi[depth]
    return tris, nodes


def deep_trees(lib):
    """Trees deeper than the traversal stacks are refused with RT_E_STATE (by the oracle too: its stack has the same 64 entries);
    the deepest legal chain, 63 levels of inner nodes, renders like the oracle."""
    sc = one_model_scene(40, 24)
    sc.settings = dict(sc.settings, useSky=True)

    def run(path, depth, options):
        tris, nodes = chain_bvh(depth)
        mgr = rt.RayComputeManager(path)
        scenes.apply(sc, mgr)
        ctx = mgr.context
        for k, v in options.items():
            ctx.set_option(k, v)
        mgr.OnEnable()
        ctx.set_buffer("Triangles", tris)
        ctx.set_buffer("Nodes", nodes)
        try:
            mgr.ResetAccumulatedRender()
            mgr.RenderFrame()
            return mgr.accumulatedResult.copy()
        finally:
            mgr.OnDestroy()
    ref = run(ORACLE_LIB, 63, {})
    assert np.count_nonzero(ref[..., :3]) > 0
    for opts in ({"kernel": 0}, {"kernel": 1}, {"kernel": 2}, {"kernel": 2, "countStats": 1}):
        assert_bit_equal(run(lib, 63, opts), ref, f"chain of 63 inner levels, {opts}")
    for path in (ORACLE_LIB, lib):
        with pytest.raises(capi.RtError) as e:
            run(path, 64, {})
        assert e.value.code == capi.RT_E_STATE and "too deep" in str(e.value)


def unchanged_uploads_are_skipped_but_changes_are_not(lib):
    """Re-sending the same ModelInfo / Spheres bytes (what the reference does every frame, RCM:192-204) is a no-op; a changed byte is not."""
    sc = scenes.knot_room(48, 32, 3, 1, nu=30, nv=6)
    sc.spheres = scenes.cornell_spheres(8, 8, 1, 1).spheres[6:8]
    fo, ao = render(ORACLE_LIB, sc, frames=3)
    fg, ag = render(lib, sc, frames=3)                        # RenderFrame re-sends ModelInfo and Spheres before every dispatch
    assert_bit_equal(ag, ao, "three frames with identical re-sent buffers")
    # and a material that changes between frames is seen
    def moving(path):
        mgr = rt.RayComputeManager(path)
        scenes.apply(sc, mgr)
        mgr.OnEnable()
        mgr.RenderFrame()
        mat = sc.models[0].material.copy(); mat["diffuseCol"] = (0.1, 0.9, 0.1, 1.0)
        mgr.set_model_material(0, mat)
        sp = sc.spheres.copy(); sp["radius"][0] *= 0.5
        mgr.set_spheres(sp)
        mgr.RenderFrame()
        a = mgr.accumulatedResult.copy()
        mgr.OnDestroy()
        return a
    assert_bit_equal(moving(lib), moving(ORACLE_LIB), "material and sphere changed between frames")


# ---- on the SIMT build -----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [2, 3])
def test_simt_group_context_renders_the_single_context_image(simt_lib, n):
    sc = scenes.knot_room(64, 45, 3, 2, nu=30, nv=6, glass=True)
    sc.spheres = scenes.cornell_spheres(8, 8, 1, 1).spheres[6:9]
    group_equals_single(simt_lib, list(range(n)), sc)
    group_equals_single(simt_lib, list(range(n)), scenes.cornell_spheres(50, 37, 3, 2), options={"kernel": 2})


def test_simt_group_context_with_tlas_and_per_frame_updates(simt_lib):
    sc = scenes.instanced_knots(56, 40, 3, 1, instances=70)
    group_equals_single(simt_lib, [0, 1], sc, frames=1)


def test_simt_model_count_alone_replans_the_scene(simt_lib):
    model_count_alone(simt_lib)


def test_simt_root_bounds_are_never_read(simt_lib):
    root_bounds_are_never_read(simt_lib)


def test_simt_deep_trees_are_refused_not_truncated(simt_lib):
    deep_trees(simt_lib)


def test_simt_unchanged_uploads(simt_lib):
    unchanged_uploads_are_skipped_but_changes_are_not(simt_lib)


def test_group_and_comm_error_paths(simt_lib, oracle_path):
    L = capi.RtLib(simt_lib)
    with pytest.raises(capi.RtError):
        L.create_multi([0, 0])                                # one rank per GPU
    with pytest.raises(capi.RtError):
        L.create_multi([])
    with pytest.raises(capi.RtError) as e:
        L.unique_id()                                         # the interpreter build carries no NCCL and says so
    assert "NCCL" in str(e.value)
    ctx = L.create_multi([0])                                 # a group of one is a plain context
    ctx.set_tile(0, 1, 8)
    ctx.destroy()
    O = capi.RtLib(oracle_path)
    with pytest.raises(capi.RtError):
        O.create_multi([0, 1])


def _build_example(tmp_path, name):
    exe = str(tmp_path / name)
    src = [os.path.join(REPO, "examples", name + ".cpp"), os.path.join(REPO, "ray_tracing_b200", "host", "RayComputeManager.cpp"),
           os.path.join(REPO, "ray_tracing_b200", "host", "BVH.cpp")]
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O1", "-ffp-contract=off", "-I", os.path.join(REPO, "include"),
           "-I", os.path.join(REPO, "ray_tracing_b200", "host")] + src + ["-ldl", "-pthread", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_cpp_tiled_example_on_the_interpreter_build(tmp_path, simt_lib, oracle_path):
    """examples/render_tiled.cpp, the C++ host of the multi-GPU form: --gpus 3 (one process, rtCreateMulti) writes the bytes
    --gpus 1 writes, and both equal the oracle's image."""
    exe = _build_example(tmp_path, "render_tiled")
    outs = {}
    for tag, lib, extra in (("oracle", oracle_path, []), ("one", simt_lib, []), ("three", simt_lib, ["--gpus", "3"])):
        out = str(tmp_path / f"{tag}.bin")
        r = subprocess.run([exe, lib, out, "--frames", "2", "--size", "96x54"] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr + r.stdout
        assert re.search(r"alpha=2 fnv1a=[0-9a-f]{16}", r.stdout), r.stdout
        outs[tag] = open(out, "rb").read()
    assert len(outs["one"]) == 96 * 54 * 16
    assert outs["one"] == outs["oracle"] and outs["three"] == outs["one"]


# ---- an ingested scene (SURVEY 8f #2): the committed Unity-YAML + OBJ fixture -----------------------------------------------------

FIXTURE_SCENE = os.path.join(REPO, "tests", "fixtures", "unity_project", "Assets", "Scenes", "Fixture.unity")
REFERENCE_EXCERPT = os.path.join(REPO, "tests", "golden", "reference_excerpt.tar.xz")


def extract_reference_excerpt(dest) -> str:
    """Unpacks the original project's five scenes with their meshes cut down (tests/golden/make_reference_excerpt.py) into `dest`;
    returns the Assets directory."""
    import tarfile
    with tarfile.open(REFERENCE_EXCERPT) as tar:
        tar.extractall(str(dest), filter="data")
    return os.path.join(str(dest), "Assets")


def load_fixture(width=None, height=None):
    from ray_tracing_b200 import unity_scene
    return unity_scene.load_unity_scene(FIXTURE_SCENE, width=width, height=height)


def ingested_scene_equals_oracle(lib, sc, frames=2, kernels=(0, 1, 2)):
    fo, ao, so = render(ORACLE_LIB, sc, frames=frames, want_stats=True)
    assert np.count_nonzero(ao[..., :3]) > 0
    for k in kernels:
        for opts in ({"kernel": k}, {"kernel": k, "countStats": 1}):
            fg, ag, sg = render(lib, sc, frames=frames, options=opts, want_stats=True)
            assert_bit_equal(ag, ao, f"{sc.name} {opts}")
            assert sg["rays"] == so["rays"]
            if opts.get("countStats"):
                assert all(sg[key] == so[key] for key in ("boxTests", "triTests")), (sc.name, opts)


def test_fixture_scene_is_read_like_a_reference_scene():
    sc = load_fixture()
    assert (sc.width, sc.height) == (480, 270) and abs(sc.fov - 52.0) < 1e-6
    assert sc.settings["maxBounceCount"] == 10 and sc.settings["numRaysPerPixel"] == 1 and sc.settings["renderSeed"] == 20260923
    assert abs(sc.settings["divergeStrength"] - 1.5) < 1e-6 and sc.settings["useSky"] is False
    assert [m.triangle_count for m in sc.meshes] == [12, 2, 528]            # built-in Cube, built-in Quad, Blob.obj (quads fanned)
    assert len(sc.models) == 9                                               # the inactive object and the disabled component are skipped
    assert [m.mesh for m in sc.models] == [0, 0, 0, 0, 0, 1, 2, 2, 2]        # three instances share the OBJ mesh
    flags = [int(m.material["flag"]) for m in sc.models]
    assert flags.count(2) == 1 and flags.count(1) == 1
    glass = next(m for m in sc.models if int(m.material["flag"]) == 2)
    # parent (rotated 12 degrees about Y, scaled (1, 1.1, 1)) x child (rotated 25 degrees, scaled 0.9): non-uniform world scale
    s = np.linalg.norm(np.asarray(glass.local_to_world)[:3, :3], axis=0)
    assert np.allclose(s, (0.9, 0.99, 0.9), atol=1e-6)
    assert np.allclose(np.asarray(glass.local_to_world) @ np.asarray(glass.world_to_local), np.eye(4), atol=1e-5)
    assert np.allclose(sc.sun_forward, (0.0, -np.sin(np.radians(50)), np.cos(np.radians(50))), atol=1e-6)


def test_simt_fixture_scene_equals_oracle(simt_lib):
    ingested_scene_equals_oracle(simt_lib, load_fixture(64, 36), frames=2)


def test_fixture_generator_reproduces_the_committed_files(tmp_path):
    """tests/fixtures/make_unity_fixture.py is the script that made the fixture; its output is what is committed."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_unity_fixture", os.path.join(REPO, "tests", "fixtures", "make_unity_fixture.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    mod.ROOT = str(tmp_path / "Assets")
    mod.main()
    for rel in ("Scenes/Fixture.unity", "Graphics/Blob.obj", "Graphics/Blob.obj.meta"):
        assert open(os.path.join(mod.ROOT, rel)).read() == open(os.path.join(REPO, "tests", "fixtures", "unity_project", "Assets", rel)).read(), rel


# ---- sample chunks: a pixel's chain changes lanes between samples (kernel 1 on small tiles) -----------------------------------------

def sample_chunks_are_schedule_only(lib, sizes=((40, 24), (9, 5), (64, 36))):
    """Option sampleChunks: the same samples in the same order whatever the number of chunks — including more chunks than samples,
    one sample per chunk, images smaller than a warp (predecessor and successor chunk in the same warp), accumulation over frames,
    the sphere accelerator, the TLAS instantiation, row-band tiles and the instrumented build."""
    for (w, h) in sizes:
        for sc, extra in ((scenes.cornell_spheres(w, h, 4, 7), {}), (scenes.knot_room(w, h, 4, 5, nu=30, nv=6, glass=True), {}),
                          (scenes.random_soup(w, h, max_bounces=3, rays_per_pixel=6, triangles=500, spheres=90), {}),
                          (scenes.instanced_knots(w, h, 3, 4, instances=8), {"tlas": 1})):
            fo, ao, so = render(ORACLE_LIB, sc, frames=2, want_stats=True)
            for kernel in (1, 2):
                for chunks in (2, 3, 16, 64):
                    opts = dict(extra, kernel=kernel, sampleChunks=chunks)
                    fg, ag, sg = render(lib, sc, frames=2, options=opts, want_stats=True)
                    assert_bit_equal(ag, ao, f"{sc.name} {w}x{h} {opts}")
                    assert_bit_equal(fg, fo, f"{sc.name} {w}x{h} frame {opts}")
                    assert sg["rays"] == so["rays"]
    sc = scenes.knot_room(48, 40, 4, 6, nu=30, nv=6)
    fo, ao, so = render(ORACLE_LIB, sc, frames=1, want_stats=True)
    rows = [y for y in range(sc.height) if (y // 8) % 3 == 1]
    for kernel in (1, 2):
        fg, ag, sg = render(lib, sc, frames=1, options={"kernel": kernel, "sampleChunks": 3, "countStats": 1}, want_stats=True)
        assert_bit_equal(ag, ao, f"instrumented, chunks of a third, kernel {kernel}")
        assert all(sg[k] == so[k] for k in ("rays", "boxTests", "triTests"))
        ft, at = render(lib, sc, frames=1, options={"kernel": kernel, "sampleChunks": 4}, tile=(1, 3, 8))
        assert_bit_equal(at[rows], ao[rows], f"row bands of rank 1 of 3, four chunks, kernel {kernel}")
    # (kernel 2 ignores the option: its own hand-off was measured slower than whole pixels and removed)
    # one sample per pixel: nothing to split
    sc1 = scenes.cornell_spheres(24, 16, 3, 1)
    assert_bit_equal(render(lib, sc1, frames=2, options={"kernel": 1, "sampleChunks": 8})[1], render(ORACLE_LIB, sc1, frames=2)[1], "1 spp")


def test_simt_sample_chunks_are_schedule_only(simt_lib):
    sample_chunks_are_schedule_only(simt_lib)


@pytest.mark.parametrize("order", ["1", "2"])
def test_simt_sample_chunks_under_other_lane_schedules(simt_lib, monkeypatch, order):
    monkeypatch.setenv("RT_SIMT_ORDER", order)
    sample_chunks_are_schedule_only(simt_lib, sizes=((33, 7),))


def test_simt_sample_chunks_on_a_rank_without_rows(simt_lib):
    """Found by tools/simt_fuzz.py (seed 515245772): a 7x1 image in bands of one row over three ranks leaves ranks 1 and 2 no pixel;
    forced sample chunks then divided by a job count of zero."""
    sc = scenes.knot_room(7, 1, 3, 2, nu=20, nv=6)
    fo, ao = render(ORACLE_LIB, sc, frames=1)
    for kernel in (1, 2):
        for rank in (0, 1, 2):
            ft, at = render(simt_lib, sc, frames=1, options={"kernel": kernel, "sampleChunks": 7}, tile=(rank, 3, 1))
            if rank == 0:
                assert_bit_equal(at, ao, f"kernel {kernel}")


# ---- the parameter space of the reference's own scenes (SURVEY Appendix B), applied to the fixture scene -----------------------------

SHIPPED_SETTINGS = {   # manager block of each shipped scene: resolution, MaxBounce, BVH quality, defocus / focus distance, camera field of view
    "Glass Dragon": dict(size=(1920, 1080), maxBounceCount=10, bvhQuality=1, defocusStrength=0.0, focusDistance=1.0, fov=54.5),
    "Glass Balls": dict(size=(1388, 781), maxBounceCount=10, bvhQuality=1, defocusStrength=0.0, focusDistance=1.0, fov=60.0),
    "Sphere Refract": dict(size=(1573, 885), maxBounceCount=32, bvhQuality=1, defocusStrength=100.0, focusDistance=5.3, fov=38.0),
    "Splash": dict(size=(1388, 781), maxBounceCount=32, bvhQuality=0, defocusStrength=0.0, focusDistance=1.0, fov=60.0),
    "Text": dict(size=(1280, 720), maxBounceCount=32, bvhQuality=1, defocusStrength=0.0, focusDistance=1.0, fov=60.0),
}


def fixture_with_shipped_settings(name, scale):
    st = SHIPPED_SETTINGS[name]
    w, h = max(8, int(st["size"][0] * scale)), max(6, int(st["size"][1] * scale))     # odd sizes on purpose (781, 885 rows: partial 8x8 groups)
    sc = load_fixture(w, h)
    sc.fov = st["fov"]
    sc.settings = dict(sc.settings, maxBounceCount=st["maxBounceCount"], bvhQuality=st["bvhQuality"], defocusStrength=st["defocusStrength"],
                       focusDistance=st["focusDistance"], numRaysPerPixel=1, divergeStrength=1.5, useSky=False, accumulate=True)
    sc.name = f"fixture with the settings of {name}"
    return sc


@pytest.mark.parametrize("name", sorted(SHIPPED_SETTINGS))
def test_simt_fixture_under_the_settings_of_every_shipped_scene(simt_lib, name):
    """1 ray per pixel per frame over several accumulated frames (numRaysPerPixel: 1 in all five scenes), 10 or 32 bounces, the depth of
    field of Sphere Refract, the Low-quality BVH of Splash: the kernels against the oracle, traversal counters included."""
    ingested_scene_equals_oracle(simt_lib, fixture_with_shipped_settings(name, 1.0 / 24.0), frames=3)


def test_simt_group_context_api_surface(simt_lib):
    """What else a host may do with the context rtCreateMulti returns: resize, reset, options, statistics, pipelined readback, display,
    BVH build, a second group beside the first; and what it may not (a communicator of its own)."""
    import ctypes as C
    sc = scenes.knot_room(40, 30, 3, 2, nu=30, nv=6)
    fo, ao = render(simt_lib, sc, frames=2)
    L = capi.RtLib(simt_lib)
    mgr = rt.RayComputeManager(simt_lib, devices=[0, 1, 2])
    other = rt.RayComputeManager(simt_lib, devices=[3, 4])
    for m in (mgr, other):
        scenes.apply(sc, m); m.OnEnable()
    ctx = mgr.context
    with pytest.raises(capi.RtError):
        ctx.comm_init(b"\0" * 128, 0, 3)                     # a group has its communicator
    with pytest.raises(capi.RtError):
        ctx.comm_destroy()
    mgr.RenderFrame(); other.RenderFrame(); mgr.RenderFrame(); other.RenderFrame()
    assert_bit_equal(mgr.accumulatedResult, ao, "group of three"); assert_bit_equal(other.accumulatedResult, ao, "group of two beside it")
    # pipelined readback and display read the leader's complete textures
    buf = np.empty((30, 40, 4), dtype=np.float32)
    ctx.readback_async("AccumulatedRender", buf.ctypes.data, buf.nbytes); ctx.readback_wait()
    assert_bit_equal(buf, ao, "rtReadbackAsync on a group")
    rgba = np.empty((30, 40, 4), dtype=np.uint8)
    ctx.display_async(True, 2, rgba.ctypes.data, rgba.nbytes); ctx.synchronize()
    assert np.array_equal(rgba, ctx.display(True, 2))
    # statistics are sums over the group; reset reaches every member
    st = ctx.stats()
    assert st["rays"] == render(simt_lib, sc, frames=2, want_stats=True)[2]["rays"]
    ctx.reset_stats()
    assert ctx.stats()["rays"] == 0
    # reset + resize + a kernel option, then the same image again at the new size
    mgr.set_screen(24, 16)
    mgr.ResetAccumulatedRender()
    ctx.set_option("kernel", 1)
    mgr.RenderFrame()
    assert_bit_equal(mgr.accumulatedResult, render(simt_lib, sc, frames=1, width=24, height=16)[1], "after resize")
    # rtBuildBVH through the group's context
    m = scenes.knot_mesh(nu=30, nv=6)
    th, nh, _ = rt.build_bvh(m.vertices, m.indices, m.normals, 1)
    tg, ng = ctx.build_bvh(m.vertices, m.indices, m.normals, 1)
    assert np.array_equal(ng.view(np.uint8), nh.view(np.uint8)) and np.array_equal(tg.view(np.uint8), th.view(np.uint8))
    mgr.OnDestroy(); other.OnDestroy()
