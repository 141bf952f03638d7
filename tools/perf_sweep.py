"""A/B throughput of kernel variants on a GPU box.  Usage: perf_sweep.py [scene:w:h:spp ...]"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200 import capi

cases = [a.split(":") for a in sys.argv[1:] if ":" in a] or [["final", "1920", "1080", "16"], ["cornell", "600", "600", "32"],
                                                             ["book1", "800", "450", "16"], ["mesh", "1920", "1080", "8"],
                                                             ["cornell_smoke", "600", "600", "32"]]
variants = [a for a in sys.argv[1:] if ":" not in a] or ["v2"]
for name, w, h, spp in cases:
    w, h, spp = int(w), int(h), int(spp)
    sc = capi.Scene(name)
    row = {"scene": name, "w": w, "h": h, "spp": spp}
    ref = None
    for v in variants:
        os.environ["RT_B200_KERNEL"] = v
        ctx = capi.Context(0)
        ctx.upload(sc)
        ctx.render(w, h, spp, max_depth=sc.depth, seed=1)
        best = 1e30
        for _ in range(3):
            ctx.render(w, h, spp, max_depth=sc.depth, seed=1)
            best = min(best, ctx.stats()["render_ms"])
        img = ctx.download(spp)
        if ref is None:
            ref = img
        same = bool((img == ref).all())
        st = ctx.stats()
        row[v] = {"ms": round(best, 3), "msamples_s": round(w * h * spp / best / 1e3, 1), "regs": st["regs_per_thread"], "blocks": st["blocks"], "bit_identical_to_first": same}
        ctx.close()
    print(json.dumps(row), flush=True)
