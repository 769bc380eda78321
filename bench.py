#!/usr/bin/env python
"""bench.py — the headline measurement: Mrays/s and ms/frame of the path-tracing hot path at 1920x1080, 8 bounces.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                     the reference's CPU statement of the path (oracle) on the host cores
    python bench.py ... --dump-outputs DIR                   also writes the images of the last timed step to DIR/*.npy, to compare builds

Default workload = BVH traversal at the metric's own resolution and bounce count (BASELINE.json configs[2] shape): an
87,132-triangle mesh in a Cornell room (3 models, BVHs by the reference's builder), 1920x1080, 8 bounces, 256 samples per pixel
in one frame.  A "step" is one frame: one RayTrace dispatch over the whole image (the (R = spp, F = 1) split of SURVEY.md 8d).
A "ray" is one CalculateRayCollision call (RayCommon.hlsl:487), counted by the kernel itself.  The same JSON line carries, under
"extra", the other workloads measured the same way in the same process: configs[1] (9-sphere Cornell box, 64 spp), the
configs[4] shape (1,000,000 triangles + 10,000 spheres, 4096x4096, 16 bounces) and the reference's own operating mode, one
sample per pixel per frame (all five shipped scenes: numRaysPerPixel 1), for both scenes.

  value     whole-job Mrays/s with everything resident in HBM: per step only the Frame uniform changes, the dispatch, and
            for N > 1 the per-frame all-gather of finished tiles, which rtDispatch itself issues (NCCL inside the C-ABI).
  e2e       the same metric through the public host API (RayComputeManager.RenderFrame -> C-ABI) with HOST buffers: every
            step re-uploads ModelInfo / Spheres / uniforms from host memory with one value changed (so the bytes really
            travel; the reference re-sends them each frame, RayComputeManager.cs:192-204) and the host that shows the image
            (rank 0) reads the accumulated float4 image into pinned memory (rtReadbackAsync: frame k's copy overlaps frame
            k+1's kernel; the last copy is inside the timed region).
  roofline  HBM roofline of the trace kernel on ALGORITHMIC bytes (SURVEY.md 8d):
            32*boxTests + 72*triTests + 224*rays*modelCount + 104*sphereTests + 48*W*H per frame, counts from an instrumented
            replay of the very frames that were timed, divided by the kernel's own CUDA-event time; peak = measured copy
            bandwidth (MEASURED_PEAKS.json).  "physical" = what the memory system really moved for ONE launch of the same
            workload: DRAM and L2 bytes and issue-slot use from an ncu pass over a child process of this run (rank 0's
            tile), against the HBM peak and an L2 bandwidth measured in this run.  A workload whose algorithmic index
            exceeds 1.2 (its data never leaves shared memory / L1) is reported against the limiter the counters name.
  cpu_baseline  the oracle (CPU port of the reference shader) on this box's host cores, bounded pixel sample.
"""
from __future__ import annotations

import argparse
import csv
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # name: scene factory kwargs + description
    "knot256": dict(kind="knot", width=1920, height=1080, bounces=8, spp=256,
                    desc="87,132-triangle knot in a Cornell room (3 models, BVH), 1920x1080, 8 bounces, 256 spp per frame (BASELINE.json configs[2] shape)"),
    "cornell64": dict(kind="cornell", width=1920, height=1080, bounces=8, spp=64,
                      desc="9-sphere Cornell box, 1920x1080, 8 bounces, 64 spp per frame (BASELINE.json configs[1])"),
    "knot64": dict(kind="knot", width=1920, height=1080, bounces=8, spp=16,
                   desc="87,132-triangle knot in a Cornell room (3 models, BVH), 1920x1080, 8 bounces, 16 spp per frame (configs[2] shape at 16 spp)"),
    # the reference's own usage: one sample per pixel per frame, many accumulated frames (all five shipped scenes, SURVEY.md 8d)
    "cornell1": dict(kind="cornell", width=1920, height=1080, bounces=8, spp=1,
                     desc="9-sphere Cornell box, 1920x1080, 8 bounces, 1 spp per frame (the (R = 1, F = spp) split of configs[1])"),
    "knot1": dict(kind="knot", width=1920, height=1080, bounces=8, spp=1,
                  desc="87,132-triangle knot in a Cornell room (3 models, BVH), 1920x1080, 8 bounces, 1 spp per frame"),
    "instances16": dict(kind="instances", width=1920, height=1080, bounces=8, spp=16,
                        desc="24 models sharing two meshes (a 7,680-triangle knot instanced 23 times, glass / opaque / emissive, + room), "
                             "1920x1080, 8 bounces, 16 spp per frame (the many-Model shape of the reference's shipped scenes)"),
    "instances500": dict(kind="instances", width=1920, height=1080, bounces=8, spp=8, instances=498,
                         desc="500 models sharing two meshes (a 7,680-triangle knot instanced 498 times + room + light), 1920x1080, 8 bounces, "
                              "8 spp per frame (many-Model shape: the TLAS over the models' world boxes, option tlas, is on automatically above 64 models)"),
    "instances62": dict(kind="instances", width=1920, height=1080, bounces=8, spp=8, instances=60, desc="62 models sharing two meshes, 1920x1080, 8 bounces, 8 spp per frame (TLAS threshold sweep)"),
    "instances126": dict(kind="instances", width=1920, height=1080, bounces=8, spp=8, instances=124, desc="126 models sharing two meshes, 1920x1080, 8 bounces, 8 spp per frame (TLAS threshold sweep)"),
    "instances250": dict(kind="instances", width=1920, height=1080, bounces=8, spp=8, instances=248, desc="250 models sharing two meshes, 1920x1080, 8 bounces, 8 spp per frame (TLAS threshold sweep)"),
    "cluster4k": dict(kind="cluster", width=3840, height=2160, bounces=12, spp=4,
                      desc="871,212-triangle glass knot cluster (one mesh, one deep BVH) in a room, 3840x2160, 12 bounces, 4 spp per frame (configs[3] shape at 4 spp)"),
    "soup4k": dict(kind="soup", width=4096, height=4096, bounces=16, spp=2,
                   desc="1,000,000 random triangles in 3 models + 10,000 spheres, sky on, 4096x4096, 16 bounces, 2 spp per frame (configs[4] shape at 2 spp)"),
    "soup4k16": dict(kind="soup", width=4096, height=4096, bounces=16, spp=16,
                     desc="1,000,000 random triangles in 3 models + 10,000 spheres, sky on, 4096x4096, 16 bounces, 16 spp per frame (configs[4] shape, the R = 16 split of SURVEY 8d)"),
}
DEFAULT_WORKLOAD = "knot256"
DEFAULT_EXTRA = ["cornell64", "soup4k", "cluster4k", "cornell1", "knot1"]
# steps / warm-up of the extra workloads (the main workload uses --steps / --warmup): bounded so that the default run stays within minutes
EXTRA_STEPS = {"soup4k": (3, 3), "soup4k16": (2, 3), "cluster4k": (4, 3), "cornell1": (64, 8), "knot1": (64, 8)}
METRIC = "Mrays/s at 1920x1080, 8 bounces (ray = one CalculateRayCollision call)"
FALLBACK_HBM_GBS = 6650.0
DUMP_PIXELS = 1 << 20               # --dump-outputs: images above this many pixels are written as this seeded pixel sample (40 MiB in all)
L2_NOTE = "GPU arm: L2 flushed between steps (256 MiB write inside the timed region); n/a to the CPU arm"


def make_scene(w):
    from ray_tracing_b200 import scenes
    if w["kind"] == "cornell":
        return scenes.cornell_spheres(w["width"], w["height"], w["bounces"], w["spp"])
    if w["kind"] == "instances":
        return scenes.instanced_knots(w["width"], w["height"], w["bounces"], w["spp"], instances=w.get("instances", 23))
    if w["kind"] == "cluster":
        return scenes.knot_cluster(w["width"], w["height"], w["bounces"], w["spp"])
    if w["kind"] == "soup":
        return scenes.random_soup(w["width"], w["height"], w["bounces"], w["spp"], triangles=1_000_000, spheres=10_000)
    return scenes.knot_room(w["width"], w["height"], w["bounces"], w["spp"])


def workload_config(name, w):
    """The part of `config` that names the workload — identical in the b200 and the reference arm."""
    return {"workload": w["desc"], "name": name, "width": w["width"], "height": w["height"], "max_bounces": w["bounces"],
            "spp_per_frame": w["spp"], "l2": L2_NOTE}


def algorithmic_parts(st, model_count, width, height, frames):
    return {"box": 32 * (st["boxTests"] + st.get("sphereBoxTests", 0)), "tri": 72 * st["triTests"], "model": 224 * st["rays"] * model_count,
            "sphere": 104 * st["sphereTests"], "frame": 48 * width * height * frames}


def algorithmic_bytes(st, model_count, width, height, frames):
    return sum(algorithmic_parts(st, model_count, width, height, frames).values())


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle on the host cores (cpu_baseline leg and --impl reference)
# ---------------------------------------------------------------------------------------------------------------------

def effective_cores():
    """Host threads this process can really use: the affinity mask, capped by a cgroup CPU quota if one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def cpu_sample(w, steps, warmup, pixels=None):
    """Times the oracle on a seeded sparse pixel sample of the workload (exact: pixels are independent and seeded from
    their global index).  Returns (Mrays/s, ms per step, cores, sample description)."""
    import ctypes as C
    import ray_tracing_b200 as rt
    from ray_tracing_b200 import build as b, scenes
    if pixels is None:
        pixels = max(4096, int(131072 * 64 / max(w["spp"], 1)))       # about the same number of paths per step for every spp
    sc = make_scene(w)
    mgr = rt.RayComputeManager(b.LIB_ORACLE)
    scenes.apply(sc, mgr)
    mgr.OnEnable()
    L = C.CDLL(b.LIB_ORACLE)
    rng = np.random.RandomState(11)
    xy = np.stack([rng.randint(0, w["width"], pixels), rng.randint(0, w["height"], pixels)], axis=1).astype(np.int32)
    out = np.empty((pixels, 4), dtype=np.float32)
    ctx = mgr.context
    ctx.set_option("threads", effective_cores())
    handle = C.c_void_p(ctx.handle.value)
    times, rays = [], 0
    for i in range(warmup + steps):
        ctx.set_int("Frame", 1 + i)
        ctx.reset_stats()
        t0 = time.perf_counter()
        rc = L.orRenderPixels(handle, xy.ctypes.data_as(C.c_void_p), pixels, out.ctypes.data_as(C.c_void_p))
        dt = time.perf_counter() - t0
        assert rc == 0
        if i >= warmup:
            times.append(dt)
            rays += ctx.stats()["rays"]
    cores = effective_cores()
    total = sum(times)
    sample = f"{pixels} seeded random pixels x {w['spp']} spp of the {w['width']}x{w['height']} frame per step, {cores} threads"
    return rays / total / 1e6, 1e3 * total / max(len(times), 1), cores, sample


def run_reference(args, name, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, ms, cores, sample = cpu_sample(w, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, w),
        "note": "CPU restatement of RayCommon.hlsl (oracle/): the reference's HLSL / C# cannot run here (no Unity, no C# toolchain)",
        "cpu_baseline": {"value": round(value, 3), "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 3), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def mark(self):
        return len(self.samples)

    def summary(self, start=0, end=None):
        rows = [r for r in self.samples[start:end] if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons, "samples": len(rows)}

    def stop(self):
        if self.proc:
            self.proc.terminate()


def measured_hbm_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def measure_l2_peak(torch, dev):
    """L2 copy bandwidth, measured like MEASURED_PEAKS measures HBM: b.copy_(a) over buffers that stay in the 126 MB L2
    (2 x 24 MiB), read + write bytes, best of 20 timings of 8 back-to-back copies, CUDA events."""
    n = 24 << 20
    a = torch.empty(n, dtype=torch.uint8, device=dev); b = torch.empty(n, dtype=torch.uint8, device=dev)
    a.zero_(); b.zero_()
    for _ in range(5):
        b.copy_(a)
    best = 1e9
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(8):                       # eight back-to-back copies per timing: the launch ramp of a 10 us kernel is not bandwidth
            b.copy_(a)
        e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / 8)
    return 2 * n / (best * 1e-3) / 1e9


NCU_METRICS = ["dram__bytes_read.sum", "dram__bytes_write.sum", "lts__t_bytes.sum", "lts__t_sector_hit_rate.pct", "l1tex__t_sector_hit_rate.pct",
               "smsp__issue_active.avg.pct_of_peak_sustained_elapsed", "smsp__thread_inst_executed_per_inst_executed.ratio", "gpu__time_duration.sum"]
_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "nsecond": 1e-9, "usecond": 1e-6, "msecond": 1e-3, "second": 1.0, "ns": 1e-9, "us": 1e-6, "ms": 1e-3, "s": 1.0}


def ncu_probe(name, local, rank, world, band_rows, lib, timeout=240):
    """Counters of ONE launch of the trace kernel on this workload (this rank's tile), from an ncu pass over a child process:
    the second RayTrace dispatch of `bench.py --probe`.  Returns a dict or {"unavailable": why}."""
    log = f"/tmp/rt_b200_probe_{os.getpid()}_{name}.csv"
    cmd = ["ncu", "--metrics", ",".join(NCU_METRICS), "--clock-control", "none", "-k", "regex:k_raytrace", "--launch-skip", "1", "--launch-count", "1",
           "--csv", "--page", "raw", "--log-file", log,
           sys.executable, os.path.abspath(__file__), "--probe", "--workload", name, "--probe-tile", f"{rank},{world},{band_rows}", "--probe-device", str(local)]
    if lib:
        cmd += ["--lib", lib]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID")}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        rows = [row for row in csv.reader(io.StringIO(open(log).read())) if row]
        os.remove(log)
        hdr = next(i for i, row in enumerate(rows) if "Kernel Name" in row)
        names, units, vals = rows[hdr], rows[hdr + 1], rows[hdr + 2]

        def get(k):
            i = names.index(k)
            return float(vals[i].replace(",", "")) * _UNIT.get(units[i], 1.0)
        out = {"kernel": vals[names.index("Kernel Name")].split("(")[0][:80]}
        out["dram_bytes"] = int(get("dram__bytes_read.sum") + get("dram__bytes_write.sum"))
        out["l2_bytes"] = int(get("lts__t_bytes.sum"))
        out["l2_hit_pct"] = round(get("lts__t_sector_hit_rate.pct"), 1)
        out["l1_hit_pct"] = round(get("l1tex__t_sector_hit_rate.pct"), 1)
        out["issue_active_pct"] = round(get("smsp__issue_active.avg.pct_of_peak_sustained_elapsed"), 1)
        out["lanes_per_instruction"] = round(get("smsp__thread_inst_executed_per_inst_executed.ratio"), 2)
        out["profiled_launch_ms"] = round(get("gpu__time_duration.sum") * 1e3, 3)
        return out
    except Exception as e:                      # no ncu, no permission for the counters, parse error: the physical block says so
        return {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}


def run_probe(args, w):
    """Child of ncu_probe: two RayTrace dispatches of the workload on one GPU (the given tile), nothing else."""
    import ray_tracing_b200 as rt
    from ray_tracing_b200 import build as b, scenes
    rank, world, band = [int(x) for x in args.probe_tile.split(",")]
    sc = make_scene(w)
    mgr = rt.RayComputeManager(args.lib or b.LIB_CUDA, device=args.probe_device)
    scenes.apply(sc, mgr)
    ctx = mgr.context
    apply_options(ctx, args)
    ctx.set_tile(rank, world, band)
    mgr.OnEnable()
    for f in (1, 2):
        ctx.set_int("Frame", f)
        ctx.dispatch_full(0)
    ctx.synchronize()
    mgr.OnDestroy()


OPTION_FLAGS = [("kernel", "kernel"), ("pool_slots", "poolSlots"), ("smem_nodes", "smemNodes"), ("model_skip", "modelSkip"), ("sort_rays", "sortRays"),
                ("tail_lanes", "tailLanes"), ("pair_order", "pairOrder"), ("grid_fit", "gridFit"), ("l2_persist", "l2Persist"),
                ("treelet_prefetch", "treeletPrefetch"), ("tlas", "tlas")]


def apply_options(ctx, args):
    for attr, opt in OPTION_FLAGS:
        v = getattr(args, attr, None)
        if v is not None:
            ctx.set_option(opt, v)


def dump_outputs(ctx, out_dir):
    """Writes what the timed path computed in its last step, as a caller of it receives it: the frame image and the accumulated
    image, (H, W, 4) float32 each.  Larger than DUMP_PIXELS pixels, both are reduced to the same seeded sample of pixels,
    (DUMP_PIXELS, 4) each, and pixels.npy holds the sampled pixel indices (y * W + x) as float64."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"frame": ctx.readback("FrameRender"), "accumulated": ctx.readback("AccumulatedRender")}
    h, w = out["frame"].shape[:2]
    if h * w > DUMP_PIXELS:
        pix = np.sort(np.random.default_rng(0).choice(h * w, DUMP_PIXELS, replace=False))
        out = {k: v.reshape(h * w, 4)[pix] for k, v in out.items()}
        out["pixels"] = pix.astype(np.float64)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def measure(name, w, args, env, steps, warmup, full, dump_dir=None):
    """One workload, measured three ways (resident, instrumented replay, end to end).  `full`: also the ncu probe.
    `dump_dir`: write the images of the last timed step there (dump_outputs)."""
    torch, dist = env["torch"], env["dist"]
    import ray_tracing_b200 as rt
    from ray_tracing_b200 import build as b, multigpu, scenes
    rank, world, local, dev = env["rank"], env["world"], env["local"], env["dev"]
    sc = make_scene(w)
    W, H = w["width"], w["height"]
    mgr = rt.RayComputeManager(args.lib or b.LIB_CUDA, device=local)   # raises without the CUDA library / a GPU
    scenes.apply(sc, mgr)
    tiled = multigpu.TiledRenderer(mgr, rank, world, band_rows=args.band_rows, device=dev, fused=args.exchange == "fused",
                                   exchange="torch" if args.exchange == "torch" else "abi")   # also puts the context on a torch stream
    ctx, stream = tiled.ctx, tiled.stream
    apply_options(ctx, args)
    mgr.OnEnable()
    if tiled.fused:
        with torch.cuda.stream(stream):
            tiled._connect_peers()
            dist.barrier()
    model_count = len(sc.models)
    flush = env["flush"]
    pinned = [torch.empty((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(2)] if rank == 0 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_resident(frame_no):
        with torch.cuda.stream(stream):
            ctx.set_int("Frame", frame_no)
            if tiled.fused:
                tiled.frame_fence()
                ctx.dispatch_full(0)
                tiled.frame_fence()
            else:
                ctx.dispatch_full(0)                                   # N > 1: ends with pack -> ncclAllGather -> unpack (inside the ABI)
            if world > 1 and tiled.exchange == "torch":
                send, recv = tiled._views()
                ctx.pack_tile()
                dist.all_gather_into_tensor(recv, send)
                ctx.unpack_tiles()
            flush.zero_()                                             # evict L2 between steps

    touched = {"i": 0}

    def step_e2e(k):
        # one input really changes every step (a field the shader never reads for this material), so the upload is not skipped
        touched["i"] += 1
        if model_count:
            mat = sc.models[0].material.copy(); mat["absorptionStrength"] = float(touched["i"])
            mgr.set_model_material(0, mat)
        else:
            sp = sc.spheres.copy(); sp["material"]["ior"][0] = 1.0 + 1e-3 * touched["i"]
            mgr.set_spheres(sp)
        tiled.render_frame()                                          # RenderFrame(): host -> device uploads + dispatch (+ all-gather)
        if rank == 0:
            with torch.cuda.stream(stream):
                buf = pinned[k & 1]
                ctx.readback_async("AccumulatedRender", buf.data_ptr(), buf.numel() * 4)    # waits (on the device) for frame k-1's copy, then overlaps frame k+1

    # ---- device-resident timing ------------------------------------------------------------------------------------
    frame_no = 1
    sampler = env["sampler"]
    for _ in range(warmup):
        step_resident(frame_no); frame_no += 1
    barrier()
    ctx.reset_stats()
    first_timed = frame_no
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    c0 = sampler.mark()
    with torch.cuda.stream(stream):
        e0.record(stream)
    for _ in range(steps):
        step_resident(frame_no); frame_no += 1
    with torch.cuda.stream(stream):
        e1.record(stream)
    barrier()
    c1 = sampler.mark()
    ms_total = e0.elapsed_time(e1)
    if dump_dir and rank == 0:
        dump_outputs(ctx, dump_dir)
    st = ctx.stats()
    rays_local, kernel_ms, exchange_ms = st["rays"], st["kernelMs"], st.get("exchangeMs", 0.0)

    # ---- instrumented replay of the timed frames: exact traversal counts for the roofline -----------------------
    ctx.set_option("countStats", 1)
    ctx.set_option("exchange", 0)
    ctx.reset_stats()
    for f in range(first_timed, first_timed + steps):
        with torch.cuda.stream(stream):
            ctx.set_int("Frame", f)
            ctx.dispatch_full(0)
    cst = ctx.stats()
    ctx.set_option("countStats", 0)
    ctx.set_option("exchange", 0 if (world > 1 and tiled.exchange != "abi") else 1)
    assert cst["rays"] == rays_local, "instrumented replay traced different rays"

    # ---- end to end through the host API ---------------------------------------------------------------------------------
    mgr.ResetAccumulatedRender()
    for k in range(warmup):
        step_e2e(k)
    ctx.readback_wait()
    barrier()
    ctx.reset_stats()
    t0 = time.perf_counter()
    for k in range(steps):
        step_e2e(k)
    ctx.readback_wait()
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_rays_local = ctx.stats()["rays"]

    # ---- 1-spp workloads: end to end with what the reference's display pass consumes (Display.shader: tex / Frame, 8-bit sRGB) -----
    e2e_disp_s = None
    if w["spp"] == 1:
        rgba = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory() for _ in range(2)] if rank == 0 else None

        def step_display(k):
            touched["i"] += 1
            if model_count:
                mat = sc.models[0].material.copy(); mat["absorptionStrength"] = float(touched["i"])
                mgr.set_model_material(0, mat)
            else:
                sp = sc.spheres.copy(); sp["material"]["ior"][0] = 1.0 + 1e-3 * touched["i"]
                mgr.set_spheres(sp)
            tiled.render_frame()
            if rank == 0:
                with torch.cuda.stream(stream):
                    ctx.display_async(True, mgr.numAccumulatedFrames - 1, rgba[k & 1].data_ptr(), rgba[k & 1].numel())
        for k in range(warmup):
            step_display(k)
        ctx.readback_wait()
        barrier()
        ctx.reset_stats()
        t0 = time.perf_counter()
        for k in range(steps):
            step_display(k)
        ctx.readback_wait()
        barrier()
        e2e_disp_s = time.perf_counter() - t0
        disp_rays = ctx.stats()["rays"]

    # ---- reduce over ranks --------------------------------------------------------------------------------------------------
    if world > 1:
        if e2e_disp_s is not None:
            td = torch.tensor([e2e_disp_s], dtype=torch.float64, device=dev)
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
            e2e_disp_s = float(td.item())
            tr = torch.tensor([disp_rays], dtype=torch.int64, device=dev)
            dist.all_reduce(tr, op=dist.ReduceOp.SUM)
            disp_rays = int(tr.item())
        t = torch.tensor([ms_total, e2e_s, kernel_ms, exchange_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s, kernel_ms_max, exchange_ms = [float(x) for x in t.tolist()]
        r = torch.tensor([rays_local, e2e_rays_local], dtype=torch.int64, device=dev)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        rays, e2e_rays = [int(x) for x in r.tolist()]
    else:
        kernel_ms_max = kernel_ms
        rays, e2e_rays = rays_local, e2e_rays_local

    kernel_sel = args.kernel if args.kernel is not None else (2 if model_count > 0 else 1)
    kernel_label = {2: "k_raytrace_pool (persistent wavefront, per-warp path pools)",
                    1: "k_raytrace_wave (persistent threads, one path per lane)", 0: "k_raytrace_mega (reference-shaped)"}[kernel_sel]
    probe = None
    if full and rank == 0 and not args.no_probe and not env.get("probe_broken"):
        mgr.context.synchronize()
        probe = ncu_probe(name, local, rank, world, args.band_rows, args.lib)
        if "unavailable" in probe and ("Timeout" in probe["unavailable"] or "FileNotFound" in probe["unavailable"]):
            env["probe_broken"] = True          # no ncu on this box, or it hangs: do not pay the timeout once per workload
    if world > 1:
        dist.barrier()                                               # the other ranks wait while rank 0's child uses GPU 0

    rec = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        # roofline of the dominant kernel on THIS rank's launches (per launch = per frame)
        rows_here = len(multigpu.owned_rows(H, rank, world, args.band_rows)) if world > 1 else H
        counts = {"boxTests": cst["boxTests"], "triTests": cst["triTests"], "rays": cst["rays"], "sphereTests": cst["sphereTests"],
                  "sphereBoxTests": cst.get("sphereBoxTests", 0)}
        parts = algorithmic_parts(counts, model_count, W, rows_here, steps)
        alg = sum(parts.values())
        achieved = alg / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
        frac = achieved / peak
        k_ms = kernel_ms / steps
        roof = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(frac, 4),
                "traffic": probe.get("dram_bytes") if probe else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg // steps, "kernel_ms_per_launch": round(k_ms, 4),
                "algorithmic_parts_per_launch": {k: v // steps for k, v in parts.items()},
                "counts_per_launch": {"rays": cst["rays"] // steps, "boxTests": cst["boxTests"] // steps, "triTests": cst["triTests"] // steps,
                                      "sphereTests": cst["sphereTests"] // steps, "sphereBoxTests": cst.get("sphereBoxTests", 0) // steps},
                "formula": "32*(boxTests+sphereBoxTests) + 72*triTests + 224*rays*modelCount + 104*sphereTests + 48*W*H_of_this_rank, / kernel_ms_per_launch / peak"}
        if probe and "unavailable" not in probe:
            l2_peak = env["l2_peak"]
            phys = {"source": "ncu pass over one launch of this workload in a child process of this run (rank 0's tile); bytes / this run's un-profiled kernel time",
                    "dram": {"bytes_per_launch": probe["dram_bytes"], "GBs": round(probe["dram_bytes"] / (k_ms * 1e-3) / 1e9, 1),
                             "frac_of_hbm_peak": round(probe["dram_bytes"] / (k_ms * 1e-3) / 1e9 / peak, 4)},
                    "l2": {"bytes_per_launch": probe["l2_bytes"], "GBs": round(probe["l2_bytes"] / (k_ms * 1e-3) / 1e9, 1), "peak": round(l2_peak, 1),
                           "peak_source": "measured in this run: 24 MiB -> 24 MiB device copy resident in L2, read + write bytes, best of 20 x 8 copies",
                           "frac": round(probe["l2_bytes"] / (k_ms * 1e-3) / 1e9 / l2_peak, 4), "hit_pct": probe["l2_hit_pct"]},
                    "l1_hit_pct": probe["l1_hit_pct"],
                    "issue": {"active_pct_of_peak": probe["issue_active_pct"], "lanes_per_instruction": probe["lanes_per_instruction"]},
                    "profiled_launch_ms": probe["profiled_launch_ms"], "kernel": probe["kernel"]}
            fr = {"dram": phys["dram"]["frac_of_hbm_peak"], "l2": phys["l2"]["frac"], "alu": probe["issue_active_pct"] / 100.0}
            phys["limiter"] = max(fr, key=fr.get)
            roof["physical"] = phys
            if frac > 1.2:
                # the algorithmic bytes never reach HBM (spheres / models live in shared memory, L1): report against the limiter the counters name
                lim = phys["limiter"]
                roof["algorithmic_index"] = {"achieved": roof["achieved"], "peak": peak, "frac": roof["frac"],
                                             "note": "SURVEY 8(d) bytes / time / HBM peak; above 1 because most of these bytes are served on chip"}
                if lim == "alu":
                    issue_peak = 148 * 4 * 1.965            # warp instructions per ns at the maximum SM clock = G warp-inst/s
                    roof.update({"bound": "alu", "achieved": round(issue_peak * fr["alu"], 1), "peak": round(issue_peak, 1), "unit": "Gwarp-inst/s", "frac": round(fr["alu"], 4)})
                elif lim == "l2":
                    roof.update({"bound": "l2", "achieved": phys["l2"]["GBs"], "peak": phys["l2"]["peak"], "unit": "GB/s", "frac": phys["l2"]["frac"]})
                else:
                    roof.update({"bound": "hbm", "achieved": phys["dram"]["GBs"], "peak": peak, "unit": "GB/s", "frac": phys["dram"]["frac_of_hbm_peak"]})
        elif probe:
            roof["physical"] = probe
        if frac > 1.2 and roof["bound"] == "hbm" and "algorithmic_index" not in roof:
            roof["note"] = "algorithmic index above 1: most of these bytes are served from shared memory / L1, not HBM (no counters in this run to name the limiter)"
        h2d = (224 * model_count if model_count else 104 * len(sc.spheres)) + 4 * 40
        rec = {
            "value": round(rays / (ms_total * 1e-3) / 1e6, 2), "unit": "Mrays/s", "steps": steps, "warmup": warmup,
            "ms_per_step": round(ms_total / steps, 4),
            "config": workload_config(name, w),
            "run": dict(rays_per_frame=rays // steps,
                           tiling=(f"row bands of {args.band_rows} rows round-robin over {world} GPU(s), " +
                                   {"fused": "finished pixels stored into the peers' images by the trace kernel (CUDA-IPC over NVLink), 4-byte all-reduce as frame fence",
                                    "torch": "one NCCL all-gather of finished tiles per frame issued through torch.distributed",
                                    "abi": "one NCCL all-gather of finished tiles per frame issued by rtDispatch itself (rtCommInit: NCCL inside the C-ABI)"}[tiled.exchange])
                           if world > 1 else "single GPU",
                           kernel=kernel_label, options={opt: getattr(args, attr) for attr, opt in OPTION_FLAGS if getattr(args, attr, None) is not None}),
            "kernel_ms_per_launch_max_over_ranks": round(kernel_ms_max / steps, 4),
            "exchange_ms_per_step": round(exchange_ms / steps, 4) if world > 1 else 0.0,
            "clocks": sampler.summary(c0, c1),
            "e2e": {"value": round(e2e_rays / e2e_s / 1e6, 2), "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": W * H * 16,
                    "ms_per_step": round(1e3 * e2e_s / steps, 4),
                    "how": "RenderFrame through the host manager with one changed input per step (uploads really happen) + rtReadbackAsync of the accumulated float4 image "
                           "into pinned memory on rank 0 (frame k's copy overlaps frame k+1; last copy inside the timed region)"},
            "gpu_launches": steps * (1 + (2 if (world > 1 and not tiled.fused) else 0)),
            "roofline": roof,
        }
        if e2e_disp_s is not None:
            rec["e2e_display"] = {"value": round(disp_rays / e2e_disp_s / 1e6, 2), "unit": "Mrays/s", "ms_per_step": round(1e3 * e2e_disp_s / steps, 4),
                                  "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": W * H * 4,
                                  "how": "as e2e, but the host reads what the reference's display pass consumes: rtDisplayAsync = accumulated / Frame, sRGB, 8 bits per channel (Display.shader:42-47); "
                                         "the reference itself never reads the float4 target back (RayTraceDisplay.cs:9-23)"}
    mgr.OnDestroy()
    del tiled, mgr
    return rec


def run_gpu(args, name, w):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    sampler = ClockSampler(local); sampler.start()
    env = {"torch": torch, "dist": dist, "rank": rank, "world": world, "local": local, "dev": dev, "sampler": sampler,
           "flush": torch.empty(256 << 20, dtype=torch.uint8, device=dev),      # > 126 MB L2
           "l2_peak": measure_l2_peak(torch, dev) if rank == 0 else None}

    main = measure(name, w, args, env, args.steps, args.warmup, full=True, dump_dir=args.dump_outputs)
    extras = {}
    for xn in args.extra:
        if xn == name:
            continue
        xs, xw = EXTRA_STEPS.get(xn, (min(args.steps, 5), 3))
        try:
            extras[xn] = measure(xn, WORKLOADS[xn], args, env, xs, max(xw, 3), full=not args.no_extra_probe)
        except Exception as e:                                       # an extra workload must never take the main line down
            extras[xn] = {"error": f"{type(e).__name__}: {str(e)[:200]}"} if rank == 0 else None
    sampler.stop()

    if rank == 0:
        line = {"metric": METRIC, "value": main["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": main["ms_per_step"], "ms_per_frame": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "gpu_launches": main["gpu_launches"], "config": main["config"], "run": main["run"],
                "kernel_ms_per_launch_max_over_ranks": main["kernel_ms_per_launch_max_over_ranks"], "exchange_ms_per_step": main["exchange_ms_per_step"],
                "clocks": main["clocks"], "e2e": main["e2e"], "roofline": main["roofline"]}
        if world == 1 and not args.no_cpu:
            v, ms, cores, sample = cpu_sample(w, 1, 0)
            line["cpu_baseline"] = {"value": round(v, 3), "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample}
        line["extra"] = extras
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--extra", default=",".join(DEFAULT_EXTRA), help="comma-separated workloads measured after the main one and reported under \"extra\" (\"none\" = no extras)")
    ap.add_argument("--band-rows", type=int, default=8)
    ap.add_argument("--exchange", default="abi", choices=["abi", "torch", "fused", "allgather"],
                    help="N > 1: abi = one NCCL all-gather per frame issued by rtDispatch itself (default); torch = the same collective through torch.distributed; "
                         "fused = pixels stored into the peers' images by the trace kernel (CUDA-IPC over NVLink)")
    ap.add_argument("--kernel", type=int, default=None, help="0 = megakernel, 1 = persistent threads, 2 = pooled wavefront (default with meshes)")
    ap.add_argument("--pool-slots", type=int, default=None, help="paths per warp pool of kernel 2 (32, 64, 96)")
    ap.add_argument("--model-skip", type=int, default=None, help="kernels 1/2: skip models the ray cannot reach (1 default / 0)")
    ap.add_argument("--tlas", type=int, default=None, help="kernels 1/2: tree over the models' world boxes: -1 = automatic (default), 0 = linear test, 1 = on")
    ap.add_argument("--sort-rays", type=int, default=None, help="kernel 2: group the ray queue by direction octant (1/0)")
    ap.add_argument("--tail-lanes", type=int, default=None, help="kernel 2: leave the trace phase when this few lanes still trace")
    ap.add_argument("--treelet-prefetch", type=int, default=None, help="1 = flagged two-level treelets + L1 prefetch of both next records (needs --lib built with RT_TREELET_PREFETCH)")
    ap.add_argument("--l2-persist", type=int, default=None, help="1 = persisting L2 window over the node-pair records")
    ap.add_argument("--grid-fit", type=int, default=None, help="1 = size the persistent grid for a whole number of pixels per lane (multi-GPU tail), 0 = off")
    ap.add_argument("--pair-order", type=int, default=None, help="node-pair record order: 0 = breadth-first (default), d = treelets of d levels, depth-first")
    ap.add_argument("--smem-nodes", type=int, default=None, help="node pairs staged in shared memory (-1 = auto)")
    ap.add_argument("--lib", default=None, help="alternative build of librt_b200.so (A/B experiments)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-probe", action="store_true", help="skip the ncu pass (roofline.traffic / physical = null)")
    ap.add_argument("--no-extra-probe", action="store_true", help="ncu pass for the main workload only")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the frame and accumulated images of the main workload's last timed step to DIR/<name>.npy "
                         "(float32; above 2**20 pixels a seeded sample of 2**20 pixels, their indices in pixels.npy)")
    ap.add_argument("--probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--probe-tile", default="0,1,8", help=argparse.SUPPRESS)
    ap.add_argument("--probe-device", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        raise SystemExit("--dump-outputs: the GPU arm only")
    if args.exchange == "allgather":
        args.exchange = "abi"
    args.extra = [x for x in args.extra.split(",") if x and x != "none"]
    for x in args.extra:
        if x not in WORKLOADS:
            raise SystemExit(f"--extra: unknown workload {x}")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    w = WORKLOADS[args.workload]
    if args.probe:
        run_probe(args, w)
    elif args.impl == "reference":
        run_reference(args, args.workload, w)
    else:
        run_gpu(args, args.workload, w)


if __name__ == "__main__":
    main()
