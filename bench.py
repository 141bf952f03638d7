#!/usr/bin/env python
"""bench.py — headline benchmark of the path-tracing hot path (BASELINE.json).

Workload: configs[4], the RTOW book-2 final scene at 3840x2160, depth 50.  A "step" is one
progressive pass of --spp-per-step samples per pixel over the whole frame (default 64, so the
default 16 steps are exactly the 1024-spp BASELINE frame).  Metric: Msamples/s (whole job).

  python bench.py [--gpus N] [--steps K] [--warmup W]           this repo's CUDA path
  python bench.py --impl reference [...]                        the reference CPU renderer
  python bench.py [...] --dump-outputs DIR                      also write the frame of the timed steps as DIR/*.npy

N > 1 is launched by torchrun, one process per GPU; the frame is tile-sharded (tile t -> rank
t mod N), every rank renders ONLY its tiles into a compact buffer (1/N of the frame,
RT_FLAG_COMPACT_TILES), resolves them on its GPU and ONE NCCL gather of the resolved RGB8 tiles to
rank 0 (inside the timed region) finishes the frame: strong scaling, bit-identical image at any N.
(Frames with too few tiles shard the sample index and reduce full-frame int64 sums instead.)

The JSON line carries, besides the contract keys: `roofline` (FP32 intersection roof, the
binding one per SURVEY 8d; the FP32 peak is measured here with an FMA microbenchmark because
MEASURED_PEAKS.json only holds HBM and bf16 numbers; `traffic` = DRAM bytes of one launch from the
committed ncu capture beside the algorithmic frame bytes), `l1_bandwidth` (BVH-node + primitive
bytes per second against an L1 load-bandwidth microbenchmark: the scene is cache-resident, so this
is a cache figure, not an HBM one), `cpu_baseline` (the unmodified reference renderer timed on this
box's host cores on a bounded sample) and `e2e` (host scene description in, host RGB8 frame out
every step: rt_upload_scene + rt_render + the gathered, downloaded frame; the device-to-host copy
of step i overlaps the render of step i + 1).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCENE_DEFAULT = "final"
WORKLOADS = {"final": "C5 RTOW book-2 final scene (BASELINE configs[4])", "book1": "C1 RTOW book-1 final scene (configs[0])",
             "cornell": "C2 Cornell box (configs[1])", "cornell_smoke": "C3 Cornell box with smoke (configs[2])",
             "mesh": "C4 triangle-mesh scene (configs[3])"}
FLOPS = {"box": 24, "sphere": 30, "quad": 48, "tri": 44, "boundary": 40, "shade": 50}   # SURVEY 8d
BYTES = {"node": 64, "sphere": 16, "quad": 48, "tri": 48, "boundary": 32, "shade": 16}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default=SCENE_DEFAULT)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--spp-per-step", type=int, default=64)
    ap.add_argument("--depth", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--out-png", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the frame the timed steps rendered as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm renders a timing-dependent sample)")
    return args


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); smax.append(float(r[1])); power.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------
# the reference CPU renderer (oracle/_ref when it was built from /root/reference, else the port)
# ---------------------------------------------------------------------------------------
def cpu_reference_run(scene: str, width: int, height: int, spp: int, depth: int) -> dict:
    """One timed run of the reference CPU implementation on (width x height x spp).  Returns
    {value (Msamples/s), seconds, cores, kind, sample}."""
    assets = assets_dir()
    if not os.path.exists(os.path.join(assets, "VERSION")):   # build() generates them; a pure-Python generator otherwise (no .so is loaded)
        from raytracingoneweekendapplication_b200.assets import ensure_assets

        assets = ensure_assets()
    cores = os.cpu_count() or 1
    driver = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
    sample = f"{scene} {width}x{height} x {spp} spp, depth {depth}"
    if os.path.exists(driver):
        # the reference's own camera::render (its std::async row bands over hardware_concurrency()
        # threads, Camera.txt:59-100), wall-clocked externally (its own print is wrong, SURVEY F9);
        # rand() is the thread-local interposer (SURVEY F8), g++ -O3.
        out = subprocess.check_output([driver, "time", scene, "1", assets, str(width), str(height), str(spp), str(depth)],
                                      stderr=subprocess.DEVNULL).decode()
        info = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
        return {"value": info["msamples_per_s"], "unit": "Msamples/s", "seconds": info["seconds"], "cores": info["threads"],
                "kind": "reference", "sample": sample + f" ({info['width']}x{info['height']} rendered)"}
    from oracle import port
    from raytracingoneweekendapplication_b200 import capi

    sc = capi.Scene(scene)
    t0 = time.time()
    port.render(sc, width, height, spp, depth=depth, seed=1, threads=cores)
    dt = time.time() - t0
    return {"value": width * height * spp / dt * 1e-6, "unit": "Msamples/s", "seconds": dt, "cores": cores, "kind": "port", "sample": sample}


BASELINE_FRAMES = {"final": (3840, 2160, 50), "book1": (400, 225, 50), "cornell": (600, 600, 50), "cornell_smoke": (600, 600, 50),
                   "mesh": (1920, 1080, 50)}


def assets_dir() -> str:
    """The generated assets (textures, meshes) the scenes load; created by build() -- found without importing the package."""
    return os.environ.get("RT_B200_ASSETS") or os.path.join(ROOT, "scenes", "assets")


def reference_scene_info(scene: str) -> dict:
    driver = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
    if os.path.exists(driver):
        out = subprocess.check_output([driver, "scene", scene, "1", assets_dir()], stderr=subprocess.DEVNULL).decode()
        return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    w, h, d = BASELINE_FRAMES.get(scene, (1024, 576, 50))
    return {"width": w, "height": h, "depth": d}


def bounded_cpu_baseline(scene: str, width: int, height: int, depth: int, budget_s: float = 15.0) -> dict:
    """~10-30 s of CPU work on the same workload: one probe at a quarter-size frame, then the
    frame size that fits the budget at 1 spp (cost is linear in pixels x spp, Camera.txt:65-73)."""
    probe = cpu_reference_run(scene, max(64, width // 8), max(36, height // 8), 1, depth)
    rate = max(probe["value"], 1e-6) * 1e6
    want = rate * budget_s
    scale = min(1.0, (want / (width * height)) ** 0.5)
    w, h = max(64, int(width * scale) // 16 * 16), max(36, int(height * scale) // 8 * 8)
    spp = max(1, int(want / (w * h)))
    return cpu_reference_run(scene, w, h, min(spp, 64), depth)


def run_reference(args):
    """--impl reference: rank 0 times the reference CPU renderer; other ranks exit 0."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    # frame size and depth of the BASELINE config from the reference driver itself (`ref_driver scene`): nothing of this
    # repo's product (package, librt_b200.so) is imported or loaded on this arm
    width, height, depth = args.width, args.height, args.depth
    if not (width and height and depth):
        info = reference_scene_info(args.scene)
        width, height, depth = width or info["width"], height or info["height"], depth or info["depth"]
    # a bounded sample per step: the full frame would take minutes per step on a CPU
    probe = cpu_reference_run(args.scene, max(64, width // 8), max(36, height // 8), 1, depth)
    rate = max(probe["value"], 1e-6) * 1e6
    budget = 120.0 / max(1, args.steps + args.warmup)           # whole run within a few minutes
    scale = min(1.0, (rate * budget / (width * height)) ** 0.5)
    w, h = max(64, int(width * scale) // 16 * 16), max(36, int(height * scale) // 8 * 8)
    runs = [cpu_reference_run(args.scene, w, h, 1, depth) for _ in range(args.warmup + args.steps)][args.warmup:]
    secs = sum(r["seconds"] for r in runs)
    value = sum(r["value"] * r["seconds"] for r in runs) / secs if secs > 0 else 0.0
    line = {
        "impl": "reference", "metric": "path-tracing throughput", "value": value, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, len(runs)), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{WORKLOADS.get(args.scene, args.scene)} {width}x{height}, depth {depth}",
                   "scene": args.scene, "width": width, "height": height, "depth": depth,
                   "sample_width": w, "sample_height": h, "sample_spp": 1,
                   "step": (runs[0]["sample"] if runs else "") + ": a bounded sample of the same camera and scene; Msamples/s does not depend on the frame size"},
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": runs[0]["cores"] if runs else 0,
                         "kind": runs[0]["kind"] if runs else "reference", "sample": runs[0]["sample"] if runs else ""},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------
# this repo's CUDA path
# ---------------------------------------------------------------------------------------
def scene_bytes(d) -> int:
    import ctypes as C

    from raytracingoneweekendapplication_b200 import capi

    n = C.sizeof(capi.rt_scene_desc)
    n += (d.n_world + d.n_boundary_refs) * C.sizeof(capi.rt_prim_ref)
    n += d.n_spheres * C.sizeof(capi.rt_sphere) + d.n_quads * C.sizeof(capi.rt_quad) + d.n_triangles * C.sizeof(capi.rt_triangle)
    n += d.n_media * C.sizeof(capi.rt_medium) + d.n_xforms * C.sizeof(capi.rt_xform)
    n += d.n_materials * C.sizeof(capi.rt_material) + d.n_textures * C.sizeof(capi.rt_texture)
    n += d.n_perlins * C.sizeof(capi.rt_perlin) + d.n_lights * C.sizeof(capi.rt_point_light)
    for i in range(d.n_images):
        n += d.images[i].width * d.images[i].height * 3
    return n


DUMP_PIXELS = 1 << 20   # 32 bytes a pixel (two float32 RGB planes and the index): 32 MB at most


def dump_outputs(out_dir: str, planes: dict) -> None:
    """--dump-outputs: each (H, W, 3) plane of the frame as out_dir/<name>.npy, float32, flattened to (pixels, 3).  A
    frame of more than DUMP_PIXELS pixels is sampled: the same fixed, seeded set of pixels in every plane and in every
    run, their ascending flat indices in pixel_index.npy, so that two builds can be compared value for value."""
    import numpy as np

    planes = {k: v for k, v in planes.items() if v is not None}   # a tile-sharded multi-GPU frame comes back as RGB8 only
    h, w = next(iter(planes.values())).shape[:2]
    n = h * w
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    for name, plane in planes.items():
        np.save(os.path.join(out_dir, name + ".npy"), plane.reshape(n, -1)[idx].astype(np.float32))


def run_b200(args):
    import torch
    import torch.distributed as dist

    from raytracingoneweekendapplication_b200 import capi, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torchrun (python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sc = capi.Scene(args.scene)
    width, height = args.width or sc.width, args.height or sc.height
    depth = args.depth or sc.depth
    spp_step = args.spp_per_step
    ctx = capi.Context(local_rank)
    ctx.upload(sc)
    plan = sharding.plan(width, height, spp_step, rank, world, sharding.RT_SHARD_AUTO)
    shard = dict(shard_rank=rank, shard_count=world, shard_mode=plan.mode)
    # N > 1, tile-sharded: every rank owns 1/N of the tiles and renders them into a compact buffer inside the library;
    # what travels is the resolved RGB8 of those tiles (3 bytes per pixel), gathered on rank 0.
    # N > 1, sample-sharded (frames with too few tiles) and N = 1: a full-frame int64 buffer (a torch tensor bound with
    # rt_bind_accum), summed over ranks with one int64 reduce.
    compact = world > 1 and plan.mode == sharding.RT_SHARD_TILES
    if args.dump_outputs and world > 1 and not compact:   # every rank decides the same, before any rendering
        raise SystemExit("--dump-outputs: a sample-sharded multi-GPU run does not bring its frame to one host")
    tile = 16
    accum = g8 = g8_all = None
    cap = 0
    if compact:
        cap = max(ctx.lib.rt_shard_pixels(width, height, tile, r, world) for r in range(world))
        g8 = torch.zeros(cap * 3, dtype=torch.uint8, device="cuda")
        g8_all = [torch.zeros(cap * 3, dtype=torch.uint8, device="cuda") for _ in range(world)] if rank == 0 else None
        shard["compact"] = True
        shard["tile_size"] = tile
    else:
        accum = torch.zeros(width * height * 4, dtype=torch.int64, device="cuda")
        ctx.bind_accum(accum.data_ptr(), accum.numel() * 8, width, height)
    # a non-default torch stream: its handle is what rt_render launches on (handle 0, the legacy
    # default stream, would read as "NULL = the context's own stream" in the C ABI), and the
    # torch.cuda.Events below are recorded on the same stream
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i, first, stats=False):
        # passes after the first go out with RT_FLAG_OVERLAP: two lane streams with their own work counters inside the
        # library, so the drain of pass i (its last, longest paths) overlaps the start of pass i + 1 -- same sums
        ctx.render(width, height, spp_step, max_depth=depth, seed=1, spp_begin=i * spp_step, accumulate=not first, stats=stats,
                   stream=stream, blocking=False, overlap=not first, **shard)

    def exchange(total_spp):
        """The one exchange that finishes the frame on rank 0 (device-resident): resolved tiles gathered, or sums reduced."""
        if world == 1:
            return
        if compact:
            ctx.resolve_tiles(total_spp, g8.data_ptr(), cap)      # waits for this rank's passes, resolves its tiles on its GPU
            dist.gather(g8, g8_all, dst=0)                        # NCCL over NVLink, on the current (torch) stream
        else:
            sharding.reduce_frame(accum)

    # ---- warm-up (untimed) ---------------------------------------------------------------
    for i in range(args.warmup):
        step(i, first=(i == 0))
    exchange(spp_step * max(1, args.warmup))
    barrier()
    ctx.sync()

    # ---- timed region: exactly K steps + the one exchange ------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_k = torch.cuda.Event(enable_timing=True)
    ev0.record()
    launches = 0
    for i in range(args.steps):
        step(i, first=(i == 0))
        launches += 1
    ctx.join(stream)                         # stream order, no host wait: ev_k is recorded after the last pass has finished
    ev_k.record()
    exchange(spp_step * args.steps)
    launches += 1 if compact else 0          # resolve_kernel over this rank's tiles
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    ms_kernels = ev0.elapsed_time(ev_k)
    clocks = sampler.stop() if rank == 0 else None
    ctx.sync()
    t = torch.tensor([ms, ms_kernels], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_kernels = float(t[0]), float(t[1])
    total_samples = width * height * spp_step * args.steps
    value = total_samples / (ms * 1e-3) * 1e-6

    # the frame of the timed steps as a caller receives it (before the counted pass below overwrites the sums)
    frame_lin = frame_b8 = None
    if rank == 0 and (args.out_png or args.dump_outputs):
        if compact:
            frame_b8 = ctx.untile(torch.stack(g8_all).data_ptr(), cap * 3, 3, world, width, height, tile)
        elif world == 1:
            frame_lin, frame_b8 = ctx.download(spp_step * args.steps, linear=True, rgb8=True)

    if frame_b8 is not None and args.out_png:
        from raytracingoneweekendapplication_b200.host_png import write_png

        write_png(args.out_png, frame_b8)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"frame_linear": frame_lin, "frame_rgb8": frame_b8})

    # ---- per-launch algorithmic work (one counted pass of the same step, untimed) ---------------
    ctx.render(width, height, spp_step, max_depth=depth, seed=1, stats=True, **shard)   # blocking: fills counters
    st = ctx.stats()
    flops = (FLOPS["box"] * st["box_tests"] + FLOPS["sphere"] * st["sphere_tests"] + FLOPS["quad"] * st["quad_tests"] +
             FLOPS["tri"] * st["triangle_tests"] + FLOPS["boundary"] * st["boundary_tests"] + FLOPS["shade"] * st["rays"])
    nbytes = (BYTES["node"] * st["node_visits"] + BYTES["sphere"] * st["sphere_tests"] + BYTES["quad"] * st["quad_tests"] +
              BYTES["tri"] * st["triangle_tests"] + BYTES["boundary"] * st["boundary_tests"] + BYTES["shade"] * st["rays"] +
              32 * plan.pixels(width, height))
    launch_ms = ms_kernels / max(1, args.steps)      # one render_kernel launch per step
    counters = torch.tensor([flops, nbytes, st["rays"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    fp32_peak = ctx.measure_fp32_peak()
    l1_peak = ctx.measure_l1_peak()
    # DRAM traffic of one launch, from the committed ncu capture of this very command/config
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if tr.get("workload") == f"{args.scene} {width}x{height} {spp_step}spp" and world == 1:
            traffic = tr["traffic_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    ach_tflops = (flops / (launch_ms * 1e-3)) * 1e-12
    ach_gbs = (nbytes / (launch_ms * 1e-3)) * 1e-9

    # ---- e2e: host scene description in, host RGB8 frame out, every step ------------------------
    # What camera::render does per frame, in a loop: rt_upload_scene (the flattened description; an unchanged scene is
    # recognised by its fingerprint and only its staged arena is copied again), rt_render, and the frame handed out to
    # host memory -- N = 1: rt_download_begin; N > 1: every rank resolves its tiles, NCCL gather to rank 0, rt_untile_begin
    # there.  The device-to-host copy of step i runs on its own stream while step i + 1 renders; the loop ends when the
    # last frame is in host memory.
    e2e = None
    if not args.no_e2e:
        if accum is not None:
            ctx.bind_accum(None, 0, 0, 0)
        n_e2e = max(2, min(args.steps, 8))
        g8_mat = torch.zeros((world, cap * 3), dtype=torch.uint8, device="cuda") if (compact and rank == 0) else None
        g8_rows = list(g8_mat.unbind(0)) if g8_mat is not None else None
        eshard = dict(shard)

        parts = {"upload": 0.0, "render": 0.0, "exchange": 0.0, "hand_out": 0.0}

        def e2e_step(i):
            ta = time.perf_counter()
            ctx.upload(sc)                                                   # H2D: the scene
            tb = time.perf_counter()
            ctx.render(width, height, spp_step, max_depth=depth, seed=1, spp_begin=i * spp_step, blocking=False, **eshard)
            if world == 1:
                ctx.download_begin(spp_step, linear=False, rgb8=True)        # resolve + D2H queued behind the render
                parts["upload"] += tb - ta
                parts["hand_out"] += time.perf_counter() - tb
            elif compact:
                ctx.resolve_tiles(spp_step, g8.data_ptr(), cap)              # returns when this rank's pass is done and resolved
                tc = time.perf_counter()
                dist.gather(g8, g8_rows, dst=0)
                torch.cuda.current_stream().synchronize()                    # rank 0: the gathered tiles are on its GPU
                td = time.perf_counter()
                if rank == 0:
                    ctx.untile_begin(g8_mat.data_ptr(), cap * 3, 3, world, width, height, tile)
                parts["upload"] += tb - ta
                parts["render"] += tc - tb
                parts["exchange"] += td - tc
                parts["hand_out"] += time.perf_counter() - td
            else:
                ctx.sync()
                ptr, nb = ctx.accum_buffer()
                sharding.reduce_frame(_as_tensor(ptr, nb))                   # sample-sharded: int64 sums over NCCL
                torch.cuda.synchronize()
                if rank == 0:
                    ctx.download_begin(spp_step, linear=False, rgb8=True)

        # one untimed step first: the library allocates its frame, output and pinned buffers on first use
        e2e_step(0)
        if rank == 0:
            ctx.frame_end()
        barrier()
        t0 = time.perf_counter()
        checksum = 0
        for i in range(n_e2e):
            e2e_step(i)
            if rank == 0 and i > 0:
                checksum += int(ctx.frame_end()[1][0, 0, 0])                 # frame i - 1 is in host memory
        if rank == 0:
            checksum += int(ctx.frame_end()[1][0, 0, 0])
        ctx.sync()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        stu = ctx.stats()
        e2e = {"value": width * height * spp_step * n_e2e / float(tt[0]) * 1e-6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(stu["upload_bytes"]), "d2h_bytes_per_step": width * height * 3, "steps": n_e2e,
               "call": ("rt_upload_scene + rt_render + rt_download_begin / rt_frame_end per step" if world == 1 else
                        "rt_upload_scene + rt_render(compact tiles) + rt_resolve_tiles + NCCL gather + rt_untile_begin / rt_frame_end per step"),
               "ms_per_step": 1e3 * float(tt[0]) / n_e2e, "scene_description_bytes": scene_bytes(sc.desc),
               "scene_reused": bool(stu["scene_reused"]), "overlap": "device-to-host copy of step i overlaps the render of step i + 1",
               "host_ms_per_step_rank0": {k: 1e3 * v / (n_e2e + 1) for k, v in parts.items()}}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = bounded_cpu_baseline(args.scene, width, height, depth)
        except Exception as exc:  # the baseline is a reported number, never a reason to lose the bench line
            cpu = {"value": None, "unit": "Msamples/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(exc)}

    if rank == 0:
        line = {
            "metric": "path-tracing throughput", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": f"{WORKLOADS.get(args.scene, args.scene)} {width}x{height}, depth {depth}, {spp_step * args.steps} spp "
                            f"({spp_step} spp per step)",
                "scene": args.scene, "width": width, "height": height, "spp_per_step": spp_step, "depth": depth,
                "sharding": ({1: "tiles 16x16 interleaved, compact per-rank tile buffers, resolved RGB8 tiles gathered over NCCL",
                              2: "samples interleaved, int64 sums reduced over NCCL"}[plan.mode]) if world > 1 else "none",
                "passes": "steps after the first are enqueued with RT_FLAG_OVERLAP (two streams, two work counters: the drain of step i "
                          "overlaps the start of step i + 1; integer sums, same frame); launch_ms = timed region / steps",
                "l2": "frame accumulation buffer %d MB per rank%s is re-read every step; the scene (~1 MB) is "
                      "cache-resident by design" % (32 * plan.pixels(width, height) // 2 ** 20, " (> 126 MB L2)" if 32 * plan.pixels(width, height) > 126 * 2 ** 20 else ""),
            },
            "mrays_per_s": float(counters[2]) / (launch_ms * 1e-3) * 1e-6,
            "rays_per_sample": float(counters[2]) / (width * height * spp_step),
            "roofline": {"bound": "fp32", "achieved": ach_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": ach_tflops / fp32_peak if fp32_peak else None, "traffic": traffic,
                         "peak_source": "measured here: FP32 FMA microbenchmark (rt_measure_fp32_peak); MEASURED_PEAKS.json has no FP32 figure",
                         "algorithmic": "24/box + 30/sphere + 48/quad + 44/triangle + 40/boundary test + 50/ray shading (SURVEY 8d), "
                                        "counted on the device for this launch", "launch_ms": launch_ms, "per": "rank 0 launch"},
            "l1_bandwidth": {"bound": "l1", "achieved": ach_gbs, "peak": l1_peak, "unit": "GB/s", "frac": ach_gbs / l1_peak if l1_peak else None,
                             "algorithmic_bytes": nbytes, "peak_source": "measured here: L1 128-bit load microbenchmark (rt_measure_l1_peak)",
                             "algorithmic": "64 B/node visit + 16/48/48 B per sphere/quad/triangle test + 16 B/ray shading fetch + "
                                            "32 B/pixel accumulation",
                             "note": "the BVH and the primitives are L1/L2 resident (L1 hit rate 90 %), so their bytes are cache traffic; the only "
                                     "HBM traffic of a launch is the frame: see dram"},
            "dram": {"algorithmic_frame_bytes": 32 * plan.pixels(width, height), "measured_bytes_per_launch": traffic,
                     "source": "profiles/r2_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum of the same command)" if traffic else None},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "device_stats": {k: st[k] for k in ("regs_per_thread", "blocks", "threads_per_block", "bvh_nodes", "bvh_depth", "nonfinite_samples",
                                                "local_bytes_per_thread")},
            "ms_render_only": ms_kernels / args.steps,
            # active lanes per warp-level iteration of each phase of the megakernel (counted pass)
            "lane_occupancy": {
                "node_step_working": st["desc_lanes"] / max(1, st["desc_iters"]),
                "node_step_holding_a_ray": st["desc_trav_lanes"] / max(1, st["desc_iters"]),
                "leaf_visit": st["leaf_lanes"] / max(1, st["leaf_iters"]),
                "shade_phase": st["shade_lanes"] / max(1, st["shade_iters"]),
                "node_steps_per_ray": st["node_visits"] / max(1, st["rays"]),
                "leaf_visits_per_ray": st["leaf_lanes"] / max(1, st["rays"]),
                "shade_phases": st["shade_iters"], "node_iters": st["desc_iters"], "leaf_iters": st["leaf_iters"],
            },
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _as_tensor(ptr: int, nbytes: int):
    """A torch int64 view of a raw device pointer (the library-owned accumulation buffer)."""
    import torch

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (nbytes // 8,), "typestr": "<i8", "data": (ptr, False), "version": 3}
    return torch.as_tensor(h, device="cuda")


def main():
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL prints its version
    # there) are sent to stderr for the duration of the run, the line goes to the real stdout
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
