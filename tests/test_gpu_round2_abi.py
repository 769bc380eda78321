"""Round 2 additions to the C-ABI on the B200 (`-m gpu`): the bodies of tests/test_round2_abi.py against librt_b200.so, the
pipelined readback, and — on a box with at least two GPUs — the multi-GPU forms with the real NCCL all-gather inside rtDispatch
(one process: rtCreateMulti; one process per GPU: examples/render_tiled.cpp with rtCommInit, no Python in the data plane)."""
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import CUDA_LIB, ORACLE_LIB, REPO, assert_bit_equal, render
import ray_tracing_b200 as rt
from ray_tracing_b200 import scenes
import test_round2_abi as R

pytestmark = pytest.mark.gpu


def _gpu_count():
    import torch
    return torch.cuda.device_count()


def test_model_count_alone_replans_the_scene_on_gpu():
    R.model_count_alone(CUDA_LIB)


def test_root_bounds_are_never_read_on_gpu():
    R.root_bounds_are_never_read(CUDA_LIB)


def test_deep_trees_are_refused_not_truncated_on_gpu():
    R.deep_trees(CUDA_LIB)


def test_unchanged_uploads_on_gpu():
    R.unchanged_uploads_are_skipped_but_changes_are_not(CUDA_LIB)


def test_group_of_one_and_error_paths_on_gpu():
    from ray_tracing_b200 import capi
    L = capi.RtLib(CUDA_LIB)
    with pytest.raises(capi.RtError):
        L.create_multi([0, 0])
    sc = scenes.knot_room(96, 54, 3, 2, nu=40, nv=8)
    fref, aref = render(CUDA_LIB, sc, frames=2)
    mgr = rt.RayComputeManager(CUDA_LIB, devices=[0])
    scenes.apply(sc, mgr)
    mgr.OnEnable(); mgr.RenderFrame(); mgr.RenderFrame()
    assert_bit_equal(mgr.accumulatedResult, aref, "group of one GPU")
    mgr.OnDestroy()


def test_pipelined_readback_returns_every_frame_on_gpu():
    """rtReadbackAsync / rtDisplayAsync: the copy of frame k, taken while frame k+1 renders, is frame k's image."""
    import torch
    sc = scenes.knot_room(160, 90, 3, 1, nu=40, nv=8)
    refs = []
    mgr = rt.RayComputeManager(CUDA_LIB)
    scenes.apply(sc, mgr); mgr.OnEnable()
    for _ in range(4):
        mgr.RenderFrame(); refs.append(mgr.accumulatedResult.copy())
    mgr.OnDestroy()
    mgr = rt.RayComputeManager(CUDA_LIB)
    scenes.apply(sc, mgr); mgr.OnEnable()
    ctx = mgr.context
    bufs = [torch.empty((90, 160, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    got = []
    for k in range(4):
        mgr.RenderFrame()
        ctx.readback_async("AccumulatedRender", bufs[k & 1].data_ptr(), bufs[k & 1].numel() * 4)
        ctx.readback_wait()
        got.append(bufs[k & 1].numpy().copy())
    for k in range(4):
        assert_bit_equal(got[k], refs[k], f"pipelined readback, frame {k}")
    # two copies queued back to back without a host wait in between: the second waits for the first on the device
    mgr.ResetAccumulatedRender()
    mgr.RenderFrame()
    ctx.readback_async("AccumulatedRender", bufs[0].data_ptr(), bufs[0].numel() * 4)
    mgr.RenderFrame()
    ctx.readback_async("AccumulatedRender", bufs[1].data_ptr(), bufs[1].numel() * 4)
    ctx.readback_wait()
    assert_bit_equal(bufs[1].numpy(), refs[1], "second of two queued copies")
    rgba = torch.empty((90, 160, 4), dtype=torch.uint8).pin_memory()
    ctx.display_async(True, 2, rgba.data_ptr(), rgba.numel())
    ctx.synchronize()
    assert np.array_equal(rgba.numpy(), ctx.display(True, 2))
    mgr.OnDestroy()


def test_group_context_over_real_gpus_equals_one_gpu():
    n = _gpu_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    sc = scenes.knot_room(320, 180, 4, 2, nu=80, nv=8, glass=True)
    sc.spheres = scenes.cornell_spheres(8, 8, 1, 1).spheres[6:9]
    R.group_equals_single(CUDA_LIB, list(range(min(n, 4))), sc)
    R.group_equals_single(CUDA_LIB, list(range(n)), scenes.cornell_spheres(200, 150, 4, 2))


def test_cpp_tiled_example_ranks_equal_one_gpu(tmp_path):
    """N copies of examples/render_tiled.cpp (one per GPU, rtCommInit with the id passed through a file — no Python, no torch) and
    the one-process form (--gpus N, rtCreateMulti) write the bytes one GPU writes."""
    n = min(_gpu_count(), 4)
    if n < 2:
        pytest.skip("needs at least two GPUs")
    exe = R._build_example(tmp_path, "render_tiled")
    def run_one(tag, extra):
        out = str(tmp_path / f"{tag}.bin")
        r = subprocess.run([exe, CUDA_LIB, out, "--frames", "3"] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr + r.stdout
        return open(out, "rb").read(), r.stdout
    one, _ = run_one("one", [])
    multi, log = run_one("multi", ["--gpus", str(n)])
    assert multi == one, log
    idf = str(tmp_path / "nccl.id")
    procs = []
    for r in range(n):
        out = str(tmp_path / f"rank{r}.bin")
        procs.append(subprocess.Popen([exe, CUDA_LIB, out, "--frames", "3", "--rank", str(r), "--world", str(n), "--device", str(r), "--id-file", idf],
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(logs)
    assert open(str(tmp_path / "rank0.bin"), "rb").read() == one, logs[0]
    assert re.search(rf"world={n} ", logs[0])


def test_ingested_fixture_scene_all_kernels_on_gpu():
    """SURVEY 8f #2 on the GPU: a scene read from Unity YAML + OBJ (instanced mesh, built-in Cube / Quad, glass, checker, emitter,
    transform hierarchy) traced by all three kernels equals the oracle, traversal counters included."""
    R.ingested_scene_equals_oracle(CUDA_LIB, R.load_fixture(320, 180), frames=2)
    R.ingested_scene_equals_oracle(CUDA_LIB, R.load_fixture(), frames=1, kernels=(2,))


@pytest.fixture(scope="module")
def reference_assets(tmp_path_factory):
    return R.extract_reference_excerpt(tmp_path_factory.mktemp("reference"))


@pytest.mark.parametrize("name", ["Glass Dragon", "Glass Balls", "Sphere Refract", "Splash", "Text"])
def test_reference_scene_on_gpu(name, reference_assets):
    from ray_tracing_b200 import unity_scene
    sc = unity_scene.load_unity_scene(os.path.join(reference_assets, "Scenes", name + ".unity"), width=160, height=90)
    R.ingested_scene_equals_oracle(CUDA_LIB, sc, frames=1, kernels=(1, 2))


def test_sample_chunks_are_schedule_only_on_gpu():
    R.sample_chunks_are_schedule_only(CUDA_LIB, sizes=((160, 90), (9, 5)))
    # and the automatic choice: a mesh scene with about two pixels per resident lane (640 x 360 on one GPU) picks kernel 1 and chunks by itself
    sc = scenes.knot_room(640, 360, max_bounces=5, rays_per_pixel=8, nu=120, nv=10)
    fo, ao = render(ORACLE_LIB, sc, frames=1)
    fa, aa = render(CUDA_LIB, sc, frames=1)
    fw, aw = render(CUDA_LIB, sc, frames=1, options={"sampleChunks": 0})
    assert_bit_equal(aa, aw, "automatic chunks vs whole pixels")
    assert_bit_equal(aa, ao, "automatic chunks vs the oracle")


@pytest.mark.parametrize("name", sorted(R.SHIPPED_SETTINGS))
def test_fixture_under_the_settings_of_every_shipped_scene_on_gpu(name):
    R.ingested_scene_equals_oracle(CUDA_LIB, R.fixture_with_shipped_settings(name, 0.2), frames=3)
