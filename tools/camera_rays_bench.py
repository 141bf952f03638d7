#!/usr/bin/env python
"""What caller-defined cameras (RT_FLAG_CAMERA_RAYS) cost, on C5 (final, 1920x1080) and C2 (cornell, 1024x1024), 64 spp,
depth 50.  Three passes alternate, 7 rounds each, and the best device time (rt_stats.render_ms) of each is kept:
  plain    the pass rt_render picks for the scene: its per-scene instance
  general  the same pass with RT_B200_GENERAL_INSTANCE=1: the general instance the rays instance is the twin of
  rays     a pass with RT_FLAG_CAMERA_RAYS from the uploaded camera's pinhole rays (a general instance: there are no
           per-scene rays instances), which loads 48 bytes per camera sample where camera_ray computes the direction
and, alternating the same way, the host time of rt_set_camera_rays (48 bytes per pixel from pageable host memory,
validated, copied and synchronised) at the frame size and at 3840x2160.  Writes profiles/r3_camera_rays_cost.jsonl (or
argv[1]) with the card, power limit and SM clock read in the same run.
usage: camera_rays_bench.py [out.jsonl]"""
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200 import capi  # noqa: E402

CONFIGS = [("C5", "final", 1920, 1080), ("C2", "cornell", 1024, 1024)]
SPP, DEPTH, ROUNDS = 64, 50, 7
UHD = (3840, 2160)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], text=True).strip()
        name, power, sm, sm_max = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit_w": float(power), "sm_mhz": int(sm), "sm_max_mhz": int(sm_max)}
    except (OSError, subprocess.CalledProcessError, ValueError) as e:
        return {"gpu": None, "error": str(e)}


def pinhole_rays(cam, w, h):
    """The camera's pixel-centre rays as (h, w, 12) rt_camera_ray records, in double rounded once to float."""
    lookfrom, lookat, vup = (np.array(list(v), dtype=np.float64) for v in (cam.lookfrom, cam.lookat, cam.vup))
    vh = 2 * math.tan(math.radians(cam.vfov) / 2) * cam.focus_dist
    vw = vh * (w / h)
    ww = (lookfrom - lookat) / np.linalg.norm(lookfrom - lookat)
    u = np.cross(vup, ww)
    u /= np.linalg.norm(u)
    v = np.cross(ww, u)
    du, dv = vw * u / w, -vh * v / h
    dir00 = -cam.focus_dist * ww - 0.5 * vw * u + 0.5 * vh * v + 0.5 * (du + dv)
    jj, ii = np.mgrid[0:h, 0:w]
    rec = np.empty((h, w, 12), dtype=np.float32)
    rec[..., 0:3] = lookfrom
    rec[..., 3:6] = dir00 + ii[..., None] * du + jj[..., None] * dv
    rec[..., 6:9] = du
    rec[..., 9:12] = dv
    return rec


def render_ms(ctx, w, h, general=False, rays=False):
    if general:
        os.environ["RT_B200_GENERAL_INSTANCE"] = "1"
    try:
        ctx.render(w, h, SPP, max_depth=DEPTH, seed=1, camera_rays=rays)
    finally:
        os.environ.pop("RT_B200_GENERAL_INSTANCE", None)
    return ctx.stats()["render_ms"]


def timed(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_camera_rays_cost.jsonl")
    ctx = capi.Context(0)
    rows = []
    for cfg, name, w, h in CONFIGS:
        sc = capi.Scene(name)
        ctx.upload(sc)
        rec, uhd = pinhole_rays(sc.desc.camera, w, h), pinhole_rays(sc.desc.camera, *UHD)
        ctx.set_camera_rays(uhd)  # the buffer at its largest: later calls reuse it
        ctx.set_camera_rays(rec)
        for general, rays in ((False, False), (True, False), (False, True)):  # warm-up: module loads, buffers
            render_ms(ctx, w, h, general, rays)
        times = {"plain": [], "general": [], "rays": [], "set_rays_ms": [], "set_rays_uhd_ms": []}
        for _ in range(ROUNDS):
            times["plain"].append(render_ms(ctx, w, h))
            times["general"].append(render_ms(ctx, w, h, general=True))
            times["rays"].append(render_ms(ctx, w, h, rays=True))
            times["set_rays_uhd_ms"].append(timed(lambda: ctx.set_camera_rays(uhd)))
            times["set_rays_ms"].append(timed(lambda: ctx.set_camera_rays(rec)))
        best = {k: min(v) for k, v in times.items()}
        row = {"config": cfg, "scene": name, "width": w, "height": h, "spp": SPP, "depth": DEPTH, "rounds": ROUNDS,
               "best_render_ms": {k: best[k] for k in ("plain", "general", "rays")},
               "rays_vs_general": best["rays"] / best["general"] - 1.0, "rays_vs_plain": best["rays"] / best["plain"] - 1.0,
               "best_set_rays_ms": best["set_rays_ms"], "set_rays_bytes": rec.nbytes,
               "best_set_rays_uhd_ms": best["set_rays_uhd_ms"], "set_rays_uhd_bytes": uhd.nbytes,
               "all": times, **gpu_info()}
        rows.append(row)
        print(json.dumps(row), flush=True)
        sc.close()
    ctx.close()
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
