#!/usr/bin/env python
"""What rt_refit_scene saves against rt_upload_scene for a moving scene, and what the refitted tree costs at render time.

update   host clock around blocking calls, best of 3: rt_refit_scene of the moved scene (after one refit that derives the
         tree's breadth-first order) against rt_upload_scene of the same moved scene in a context of its own.  Cases:
         C5 `final` (host-built tree), and the upload_scale.py terrain as ONE indexed rt_mesh under a moving xform at
         1e5, 1e6 and 4e6 triangles (device-built tree).
quality  C5 at 1280x720, 16 spp, depth 50: rt_stats.render_ms of a pass after k refits of a growing motion (the
         rotated box of spheres turned 7.5 degrees further each frame) against a fresh upload of the same frame,
         k = 1 .. 16: best of 7 passes per tree, the two trees' passes alternating.  Each pair of frames is compared: the pixels that differ (exact-t ties between the coincident faces
         of the ground boxes, which two trees may resolve differently) and whether primary t is equal everywhere.
One JSON line per case on stdout, with the card and its power limit read in the same run; also written to
profiles/r3_refit_cost.jsonl (or argv[1]).
usage: refit_bench.py [out.jsonl]"""
import ctypes as C
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from raytracingoneweekendapplication_b200 import capi  # noqa: E402
import upload_scale  # noqa: E402

REPS = 3
PASSES = 7


def turned(desc, keep, deg):
    """A copy of `desc` whose xforms are turned `deg` degrees further about their own y axis."""
    d = capi.rt_scene_desc.from_buffer_copy(desc)
    xf = (capi.rt_xform * max(1, d.n_xforms))()
    C.memmove(xf, desc.xforms, d.n_xforms * C.sizeof(capi.rt_xform))
    a = math.radians(deg)
    ry = np.array([[math.cos(a), 0, math.sin(a)], [0, 1, 0], [-math.sin(a), 0, math.cos(a)]])
    for x in xf[:d.n_xforms]:
        x.r[:] = list((ry @ np.array(x.r[:]).reshape(3, 3)).reshape(-1))
    d.xforms = C.cast(xf, C.POINTER(capi.rt_xform))
    keep.append(xf)
    return d


def terrain_desc(n):
    pos, idx, uvs = upload_scale.indexed_terrain(n)
    d, keep = upload_scale.scene_desc(mesh=(pos, idx, uvs))
    xf = (capi.rt_xform * 1)()
    xf[0].r[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
    keep["m"][0].xform = 0
    d.xforms, d.n_xforms = C.cast(xf, C.POINTER(capi.rt_xform)), 1
    keep["xf"] = xf
    return d, keep


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def update_case(label, desc, builder_expect):
    keep = []
    frames = [turned(desc, keep, 2.0 * k) for k in range(REPS + 2)]
    ctx = capi.Context(0)
    up = capi.Context(0)
    try:
        ctx.upload(desc)
        st = ctx.stats()
        assert st["bvh_on_device"] == builder_expect, (label, st["bvh_on_device"])
        first = timed(lambda: ctx.refit(frames[0]))
        refit = [timed(lambda f=f: ctx.refit(f)) for f in frames[1:REPS + 1]]
        rbytes = ctx.stats()["upload_bytes"]
        upload = [timed(lambda f=f: up.upload(f)) for f in frames[1:REPS + 1]]
        ubytes = up.stats()["upload_bytes"]
    finally:
        ctx.close()
        up.close()
    return {"case": label, "kind": "update", "tree": "device" if builder_expect else "host", "n_prims": None,
            "refit_ms_best": min(refit), "refit_ms_all": refit, "first_refit_ms": first, "upload_ms_best": min(upload),
            "upload_ms_all": upload, "speedup": min(upload) / min(refit), "refit_bytes": rbytes, "upload_bytes": ubytes,
            "bvh_nodes": st["bvh_nodes"], "bvh_depth": st["bvh_depth"]}


def quality(sc, w=1280, h=720, spp=16, depth=50, frames=16):
    keep = []
    out = []
    ctx = capi.Context(0)
    try:
        ctx.upload(sc.desc_ptr)
        ctx.render(w, h, spp, max_depth=depth, seed=1)   # warm-up
        for k in range(1, frames + 1):
            d = turned(sc.desc, keep, 7.5 * k)
            ctx.refit(d)
            f = capi.Context(0)
            try:
                f.upload(d)
                f.render(w, h, spp, max_depth=depth, seed=1)   # warm-up of the fresh context
                r_all, u_all = [], []
                for _ in range(PASSES):   # alternating, the same pass on either tree
                    ctx.render(w, h, spp, max_depth=depth, seed=1)
                    r_all.append(ctx.stats()["render_ms"])
                    f.render(w, h, spp, max_depth=depth, seed=1)
                    u_all.append(f.stats()["render_ms"])
                r_ms, u_ms = min(r_all), min(u_all)
                differ = int((ctx.accum_download() != f.accum_download()).any(axis=-1).sum())
                t_equal = bool(np.array_equal(ctx.aov(w, h)["t"], f.aov(w, h)["t"]))
            finally:
                f.close()
            out.append({"case": "C5", "kind": "quality", "k": k, "degrees": 7.5 * k, "refit_render_ms": r_ms,
                        "fresh_render_ms": u_ms, "ratio": r_ms / u_ms, "refit_render_ms_all": r_all, "fresh_render_ms_all": u_all, "pixels_differ": differ, "primary_t_equal": t_equal,
                        "w": w, "h": h, "spp": spp})
    finally:
        ctx.close()
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_refit_cost.jsonl")
    name, power = upload_scale.card()
    rows = []
    sc = capi.Scene("final")
    rows.append(update_case("C5 final", sc.desc, 0))
    rows[-1]["n_prims"] = sc.desc.n_world
    for n in (100_000, 1_000_000, 4_000_000):
        d, keep = terrain_desc(n)
        rows.append(update_case(f"terrain mesh {n}", d, 1))
        rows[-1]["n_prims"] = n + 1
        del keep
    rows += quality(sc)
    with open(out_path, "w") as f:
        for r in rows:
            r.update(gpu=name, power_limit=power)
            line = json.dumps(r)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
