#!/usr/bin/env python
"""What RT_FLAG_MOMENTS costs on C5 at 3840x2160, in 64-spp passes, split into its two parts: the per-scene instance
the default render runs against the general instance (RT_B200_GENERAL_INSTANCE=1), and the general instance against
its moments twin.  The three arms alternate inside each of three rounds in one process; each arm renders a progressive
frame of PASSES passes (the first non-accumulating) and reports the device time per pass (rt_stats.render_ms).
Writes profiles/r3_moments_cost.jsonl (or the path given as argv[1]) with the card, power limit and SM clock.
usage: moments_cost.py [out.jsonl]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200 import capi  # noqa: E402

W, H, SPP, PASSES, ROUNDS = 3840, 2160, 64, 4, 3
ARMS = [("per_scene", False, False), ("general", True, False), ("general_moments", True, True)]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], text=True).strip()
        name, power, sm, sm_max = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit_w": float(power), "sm_mhz": int(sm), "sm_max_mhz": int(sm_max)}
    except (OSError, subprocess.CalledProcessError, ValueError) as e:
        return {"gpu": None, "error": str(e)}


def frame_ms(ctx, sc, general, moments):
    if general:
        os.environ["RT_B200_GENERAL_INSTANCE"] = "1"
    else:
        os.environ.pop("RT_B200_GENERAL_INSTANCE", None)
    ms = []
    for k in range(PASSES):
        ctx.render(W, H, SPP, max_depth=sc.depth, seed=1, spp_begin=k * SPP, accumulate=k > 0, moments=moments)
        ms.append(ctx.stats()["render_ms"])
    return ms


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_moments_cost.jsonl")
    sc = capi.Scene("final")
    ctx = capi.Context(0)
    ctx.upload(sc)
    for _, general, moments in ARMS:  # warm-up: module loads and the moments buffer
        frame_ms(ctx, sc, general, moments)
    rows = []
    for r in range(ROUNDS):
        for arm, general, moments in ARMS:
            ms = frame_ms(ctx, sc, general, moments)
            row = {"round": r, "arm": arm, "scene": "final (C5)", "width": W, "height": H, "spp_per_pass": SPP, "passes": PASSES,
                   "ms_per_pass": ms, "mean_ms_per_pass": sum(ms) / len(ms),
                   "msamples_per_s": W * H * SPP / (sum(ms) / len(ms)) / 1e3, **gpu_info()}
            rows.append(row)
            print(json.dumps(row), flush=True)
    os.environ.pop("RT_B200_GENERAL_INSTANCE", None)
    ctx.close()
    with open(out, "w") as f:
        for row in rows:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
