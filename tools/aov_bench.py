#!/usr/bin/env python
"""What the auxiliary outputs (RT_FLAG_AOV) cost, on C5 (final, 1920x1080) and C2 (cornell, 1024x1024), 64 spp, depth 50.
Three passes alternate, 7 rounds each, and the best device time (rt_stats.render_ms) of each is kept:
  plain    the pass rt_render picks for the scene: its per-scene instance
  general  the same pass with RT_B200_GENERAL_INSTANCE=1: the general instance the AOV instance is the twin of
  aov      the pass with RT_FLAG_AOV (a general instance: there are no per-scene AOV instances)
and, with the same alternation, the host time of rt_download_aov (8 floats per pixel) against rt_download (linear radiance,
3 floats per pixel), each a blocking call that ends in a device synchronise, into host buffers allocated and touched
once (a fresh buffer of this size is new pages from the kernel each time, and the page faults would dominate).  Every
round also checks that the AOV pass leaves the sums np.array_equal to the plain pass's.  Writes
profiles/r3_aov_cost.jsonl (or argv[1]) with the card, power limit and SM clock read in the same run.
usage: aov_bench.py [out.jsonl]"""
import json
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


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], text=True).strip()
        name, power, sm, sm_max = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit_w": float(power), "sm_mhz": int(sm), "sm_max_mhz": int(sm_max)}
    except (OSError, subprocess.CalledProcessError, ValueError) as e:
        return {"gpu": None, "error": str(e)}


def render_ms(ctx, w, h, general=False, aov=False):
    if general:
        os.environ["RT_B200_GENERAL_INSTANCE"] = "1"
    try:
        ctx.render(w, h, SPP, max_depth=DEPTH, seed=1, aov=aov)
    finally:
        os.environ.pop("RT_B200_GENERAL_INSTANCE", None)
    return ctx.stats()["render_ms"]


def timed(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_aov_cost.jsonl")
    ctx = capi.Context(0)
    rows = []
    for cfg, name, w, h in CONFIGS:
        sc = capi.Scene(name)
        ctx.upload(sc)
        for general, aov in ((False, False), (True, False), (False, True)):  # warm-up: module loads, buffers
            render_ms(ctx, w, h, general, aov)
        lin, aovs = np.ones((h, w, 3), dtype=np.float32), np.ones((h, w, 8), dtype=np.float32)
        lib, hd = ctx.lib, ctx._h
        ctx.download_aov(SPP)
        ctx.download(SPP)
        times = {"plain": [], "general": [], "aov": [], "download_ms": [], "download_aov_ms": []}
        identical = True
        for _ in range(ROUNDS):
            times["plain"].append(render_ms(ctx, w, h))
            plain = ctx.accum_download()
            times["general"].append(render_ms(ctx, w, h, general=True))
            times["aov"].append(render_ms(ctx, w, h, aov=True))
            identical = identical and np.array_equal(ctx.accum_download(), plain)
            times["download_ms"].append(timed(lambda: ctx._check(lib.rt_download(hd, SPP, lin.ctypes.data, None))))
            times["download_aov_ms"].append(timed(lambda: ctx._check(lib.rt_download_aov(hd, SPP, aovs.ctypes.data))))
        best = {k: min(v) for k, v in times.items()}
        row = {"config": cfg, "scene": name, "width": w, "height": h, "spp": SPP, "depth": DEPTH, "rounds": ROUNDS,
               "best_render_ms": {k: best[k] for k in ("plain", "general", "aov")},
               "aov_vs_general": best["aov"] / best["general"] - 1.0, "aov_vs_plain": best["aov"] / best["plain"] - 1.0,
               "best_download_ms": best["download_ms"], "best_download_aov_ms": best["download_aov_ms"],
               "all": times, "identical": bool(identical), **gpu_info()}
        rows.append(row)
        print(json.dumps(row), flush=True)
        sc.close()
    ctx.close()
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")
    if not all(r["identical"] for r in rows):
        sys.exit("an AOV pass changed the sums")


if __name__ == "__main__":
    main()
