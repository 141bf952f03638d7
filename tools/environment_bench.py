#!/usr/bin/env python
"""What environment lighting (rt_set_environment) costs, on C1 (book1, whose paths mostly end in a miss) and C4 (mesh), at
1920x1080, and on C2 (cornell, a LITE scene) at 1024x1024, 64 spp, depth 50.  Five passes alternate, 7 rounds each, and
the best device time (rt_stats.render_ms) of each is kept:
  plain    the pass rt_render picks for the scene without an environment: its per-scene instance
  general  the same pass with RT_B200_GENERAL_INSTANCE=1: the general instance (LITE for a LITE scene)
  nolite   general with RT_B200_NO_LITE=1: the non-LITE general instance, the twin of the environment instances (which
           have no LITE versions; on C2, general against nolite is what LITE environment twins could gain)
  uniform  a 16x8 map whose texels are the camera's background (the environment instance, the background's arithmetic)
  sky      a 2048x1024 procedural sky with a sun disc
Every round checks that the uniform pass leaves the sums np.array_equal to the plain pass's.  Then the host time of
rt_set_environment (validation, packing, the copy to the device and its synchronise) for a 2048x1024 and an 8192x4096
map, best of 7.  Writes profiles/r3_environment_cost.jsonl (or argv[1]) with the card, power limit and SM clock read in
the same run.
usage: environment_bench.py [out.jsonl]"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from aov_bench import gpu_info  # noqa: E402
from raytracingoneweekendapplication_b200 import capi  # noqa: E402

CONFIGS = [("C1", "book1", 1920, 1080), ("C4", "mesh", 1920, 1080), ("C2", "cornell", 1024, 1024)]
SPP, DEPTH, ROUNDS = 64, 50, 7


def sky(w, h):
    """A blue-to-white gradient over the horizon, a dark ground, and a sun disc of radius 0.5 degrees at radiance 5e4."""
    theta = (np.pi * (0.5 - (np.arange(h, dtype=np.float32) + 0.5) / h))[:, None]
    phi = (2 * np.pi * ((np.arange(w, dtype=np.float32) + 0.5) / w - 0.5))[None, :]
    up = np.clip(np.sin(theta), 0.0, 1.0)
    m = np.empty((h, w, 3), np.float32)
    m[..., 0] = np.where(theta > 0, 0.9 - 0.6 * up, 0.15)
    m[..., 1] = np.where(theta > 0, 0.95 - 0.45 * up, 0.12)
    m[..., 2] = np.where(theta > 0, 1.0 - 0.1 * up, 0.1)
    sun = (np.abs(theta - 0.7) < np.radians(0.5)) & (np.abs(phi - 0.9) * np.cos(0.7) < np.radians(0.5))
    m[sun] = (5e4, 4.6e4, 4.0e4)
    return m


def render_ms(ctx, w, h, general=False, lite=True):
    if general:
        os.environ["RT_B200_GENERAL_INSTANCE"] = "1"
    if not lite:
        os.environ["RT_B200_NO_LITE"] = "1"
    try:
        ctx.render(w, h, SPP, max_depth=DEPTH, seed=1)
    finally:
        os.environ.pop("RT_B200_GENERAL_INSTANCE", None)
        os.environ.pop("RT_B200_NO_LITE", None)
    return ctx.stats()["render_ms"]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_environment_cost.jsonl")
    ctx = capi.Context(0)
    sky_map = sky(2048, 1024)
    rows = []
    for cfg, name, w, h in CONFIGS:
        sc = capi.Scene(name)
        ctx.upload(sc)
        uniform = np.broadcast_to(np.array(list(sc.desc.camera.background), dtype=np.float32), (8, 16, 3)).copy()
        arms = {"plain": lambda: (ctx.set_environment(None), render_ms(ctx, w, h))[1],
                "general": lambda: (ctx.set_environment(None), render_ms(ctx, w, h, general=True))[1],
                "nolite": lambda: (ctx.set_environment(None), render_ms(ctx, w, h, general=True, lite=False))[1],
                "uniform": lambda: (ctx.set_environment(uniform), render_ms(ctx, w, h))[1],
                "sky": lambda: (ctx.set_environment(sky_map), render_ms(ctx, w, h))[1]}
        for arm in arms.values():  # warm-up: module loads, buffers
            arm()
        times = {k: [] for k in arms}
        identical = True
        for _ in range(ROUNDS):
            for k, arm in arms.items():
                times[k].append(arm())
                if k == "plain":
                    plain = ctx.accum_download()
                elif k == "uniform":
                    identical = identical and np.array_equal(ctx.accum_download(), plain)
        ctx.set_environment(None)
        best = {k: min(v) for k, v in times.items()}
        row = {"config": cfg, "scene": name, "width": w, "height": h, "spp": SPP, "depth": DEPTH, "rounds": ROUNDS,
               "best_render_ms": best, "uniform_vs_nolite": best["uniform"] / best["nolite"] - 1.0,
               "sky_vs_nolite": best["sky"] / best["nolite"] - 1.0, "sky_vs_plain": best["sky"] / best["plain"] - 1.0,
               "nolite_vs_general": best["nolite"] / best["general"] - 1.0,
               "all": times, "identical": bool(identical), **gpu_info()}
        rows.append(row)
        print(json.dumps(row), flush=True)
        sc.close()
    for mw, mh in ((2048, 1024), (8192, 4096)):
        m = np.random.default_rng(1).uniform(0.0, 4.0, (mh, mw, 3)).astype(np.float32)
        ctx.set_environment(m)  # warm-up: the allocation
        ms = []
        for _ in range(ROUNDS):
            t = time.perf_counter()
            ctx.set_environment(m)
            ms.append((time.perf_counter() - t) * 1e3)
        row = {"call": "rt_set_environment", "map_width": mw, "map_height": mh, "bytes_on_device": (mw * mh + 3) * 16,
               "best_ms": min(ms), "all_ms": ms, **gpu_info()}
        rows.append(row)
        print(json.dumps(row), flush=True)
    ctx.close()
    os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
    with open(out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")
    if not all(r["identical"] for r in rows if "identical" in r):
        sys.exit("a uniform map changed the sums")


if __name__ == "__main__":
    main()
