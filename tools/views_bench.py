#!/usr/bin/env python
"""What a multi-view batch (rt_render_views) saves per view, on two small-frame turntables of 64 views: C1 (book1,
400x225, 10 spp) and C2 (cornell, 600x600, 16 spp), depth 50, cameras from the host mirror's camera::turntable_camera.
Three arms alternate inside each of three rounds in one process:
  batch    one rt_render_views of the 64 views + one rt_download_views (RGB8)
  per_view 64 x (rt_upload_scene with camera k + rt_render + rt_download), the only way without batches
  one_view one view through rt_render_views against rt_render of the same frame and camera (device time, REPS each):
           what the general views instance costs against the instance rt_render picks for the scene
Wall times are host clocks around blocking calls (each ends in a device synchronise); device times are rt_stats.render_ms.
Every round also checks that each batch view is np.array_equal to the per-view frame.  Writes
profiles/r3_views_cost.jsonl (or argv[1]) with the card, power limit and SM clock read in the same run.
usage: views_bench.py [out.jsonl]"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200 import capi  # noqa: E402
from raytracingoneweekendapplication_b200.assets import ensure_assets  # noqa: E402

CONFIGS = [("C1", "book1", 400, 225, 10), ("C2", "cornell", 600, 600, 16)]
N_VIEWS, DEPTH, ROUNDS, REPS = 64, 50, 3, 10


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], text=True).strip()
        name, power, sm, sm_max = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit_w": float(power), "sm_mhz": int(sm), "sm_max_mhz": int(sm_max)}
    except (OSError, subprocess.CalledProcessError, ValueError) as e:
        return {"gpu": None, "error": str(e)}


def turntable(name):
    s = capi.load_scenes()
    assets = ensure_assets(None).encode()
    cams = []
    for k in range(N_VIEWS):
        c = capi.rt_camera()
        if s.rtsc_turntable_camera(name.encode(), 1, assets, N_VIEWS, k, C.byref(c)) != 0:
            raise RuntimeError(f"no turntable camera for {name}")
        cams.append(c)
    return cams


def with_camera(sc, cam):
    d = capi.rt_scene_desc.from_buffer_copy(sc.desc)
    d.camera = cam
    return d


def arm_batch(ctx, sc, cams, w, h, spp):
    ctx.upload(sc)
    t = time.perf_counter()
    ctx.render_views(cams, w, h, spp, max_depth=DEPTH)
    frames = ctx.download_views(spp, linear=False, rgb8=True)
    wall = (time.perf_counter() - t) * 1e3
    return {"wall_ms": wall, "device_ms": ctx.stats()["render_ms"]}, frames


def arm_per_view(ctx, sc, cams, w, h, spp):
    descs = [with_camera(sc, c) for c in cams]
    frames, device, upload = [], 0.0, 0.0
    t = time.perf_counter()
    for d in descs:
        ctx.upload(d)
        upload += ctx.stats()["upload_ms"]
        ctx.render(w, h, spp, max_depth=DEPTH)
        device += ctx.stats()["render_ms"]
        frames.append(ctx.download(spp, linear=False, rgb8=True))
    wall = (time.perf_counter() - t) * 1e3
    return {"wall_ms": wall, "device_ms": device, "upload_ms": upload}, np.stack(frames)


def arm_one_view(ctx, sc, cam, w, h, spp):
    ctx.upload(with_camera(sc, cam))
    single, views = [], []
    for _ in range(REPS):
        ctx.render(w, h, spp, max_depth=DEPTH)
        single.append(ctx.stats()["render_ms"])
        ctx.render_views([cam], w, h, spp, max_depth=DEPTH)
        views.append(ctx.stats()["render_ms"])
    return {"render_ms": sum(single) / REPS, "render_views_ms": sum(views) / REPS}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_views_cost.jsonl")
    ctx = capi.Context(0)
    rows = []
    for cfg, name, w, h, spp in CONFIGS:
        sc = capi.Scene(name)
        cams = turntable(name)
        arm_batch(ctx, sc, cams, w, h, spp)  # warm-up: module loads, buffers
        arm_per_view(ctx, sc, cams[:4], w, h, spp)
        arm_one_view(ctx, sc, cams[0], w, h, spp)
        for r in range(ROUNDS):
            a, fa = arm_batch(ctx, sc, cams, w, h, spp)
            b, fb = arm_per_view(ctx, sc, cams, w, h, spp)
            c = arm_one_view(ctx, sc, cams[r], w, h, spp)
            row = {"round": r, "config": cfg, "scene": name, "width": w, "height": h, "spp": spp, "views": N_VIEWS, "depth": DEPTH,
                   "batch": a, "per_view": b, "one_view": c,
                   "batch_ms_per_view": a["wall_ms"] / N_VIEWS, "per_view_ms_per_view": b["wall_ms"] / N_VIEWS,
                   "batch_device_ms_per_view": a["device_ms"] / N_VIEWS, "per_view_device_ms_per_view": b["device_ms"] / N_VIEWS,
                   "identical": bool(np.array_equal(fa, fb)), **gpu_info()}
            rows.append(row)
            print(json.dumps(row), flush=True)
        sc.close()
    ctx.close()
    with open(out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")
    if not all(r["identical"] for r in rows):
        sys.exit("a batch view differs from its single render")


if __name__ == "__main__":
    main()
