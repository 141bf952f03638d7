"""Generates the golden fixtures in tests/golden/ from the REAL reference renderer.

Runs oracle/_ref/ref_driver (the untouched headers of /root/reference compiled by
oracle/Makefile) in this container and stores, per scene:

  primary_<scene>.npz   pixel-centre primary hits: leaf index, t (f64), normal, uv, and the
                        world-space geometry key of every leaf (to map the reference's leaf
                        numbering onto the flattened scene's primitive ids)
  kat_<scene>.npz       known-answer vectors for material::scatter/emitted + texture::value
                        with scripted uniforms
  image_<scene>.npz     a converged float radiance image (linear, before gamma) + its spp

Usage:  python tests/golden/make_golden.py [primary] [kat] [image] [image_quarter] [--scenes=a,b,c]
The fixtures are committed; /root/reference is not needed to run the tests.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200.assets import ensure_assets  # noqa: E402

DRIVER = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
OUT = os.path.dirname(os.path.abspath(__file__))
SEED = 1

# (width, height) of the primary-hit fixture and (width, height, spp) of the converged image
PRIMARY = {
    "book1": (200, 112), "cornell": (150, 150), "cornell_smoke": (150, 150), "mesh": (240, 135), "final": (240, 135),
    "quads": (100, 100), "emissive": (100, 56), "specular": (128, 72), "mixed": (128, 72), "kitchen_sink": (160, 90),
    # the reference's own inputs (monkey.obj, Images/earthmap.jpg): needs the reference tree (build.ensure_reference_assets)
    "monkey": (240, 135),
}
IMAGE = {
    "book1": (120, 68, 4096), "cornell": (64, 64, 32768), "cornell_smoke": (64, 64, 32768), "mesh": (128, 72, 2048),
    "final": (96, 54, 65536), "quads": (64, 64, 2048), "emissive": (64, 36, 2048), "specular": (96, 54, 4096),
    "mixed": (96, 54, 4096), "kitchen_sink": (96, 54, 4096), "monkey": (128, 72, 4096),
}
# C1-C3 once more at a QUARTER of the BASELINE frame (half the width, half the height), same gate
IMAGE_QUARTER = {"book1": (200, 112, 8192), "cornell": (300, 300, 32768), "cornell_smoke": (300, 300, 32768)}
# stored as float16 so that each file stays under 1 MB: the rounding moves the frame mean by < 0.03 sigma of the
# reference's Monte Carlo error and sits at 86-91 dB PSNR.  Not book1: its smooth sky rounds coherently (4 sigma).
HALF_PRECISION_QUARTER = {"cornell", "cornell_smoke"}
KAT = {"kitchen_sink": 600, "mixed": 400, "final": 400, "book1": 400, "specular": 200, "mesh": 300, "monkey": 600}


def run(*args) -> dict:
    out = subprocess.check_output([DRIVER, *map(str, args)], stderr=subprocess.DEVNULL)
    return json.loads(out.decode().strip().splitlines()[-1])


def main(argv):
    what = [a for a in argv if not a.startswith("--")] or ["primary", "kat", "image"]
    scenes = None
    for a in argv:
        if a.startswith("--scenes"):
            scenes = a.split("=", 1)[1].split(",")
    assets = ensure_assets()
    with tempfile.TemporaryDirectory() as tmp:
        if "primary" in what:
            for name, (w, h) in PRIMARY.items():
                if scenes and name not in scenes:
                    continue
                prefix = os.path.join(tmp, "p_" + name)
                info = run("primary", name, SEED, assets, w, h, prefix)
                h = info["height"]
                ids = np.fromfile(prefix + ".ids.i32", dtype=np.int32).reshape(h, w)
                rec = np.fromfile(prefix + ".hit.f64", dtype=np.float64).reshape(h, w, 9)
                leaves = np.fromfile(prefix + ".leaves.f64", dtype=np.float64).reshape(-1, 10)
                np.savez_compressed(os.path.join(OUT, f"primary_{name}.npz"), ids=ids, t=rec[..., 0],
                                    normal=rec[..., 1:4].astype(np.float32), point=rec[..., 4:7].astype(np.float32),
                                    uv=rec[..., 7:9].astype(np.float32), leaves=leaves, seed=SEED)
                print("primary", name, w, h, "hit fraction %.3f" % (ids >= 0).mean(), flush=True)
        if "kat" in what:
            for name, n in KAT.items():
                if scenes and name not in scenes:
                    continue
                prefix = os.path.join(tmp, "k_" + name)
                info = run("kat", name, SEED, assets, n, prefix)
                kat = np.fromfile(prefix + ".kat.f64", dtype=np.float64).reshape(-1, 40)
                leaves = np.fromfile(prefix + ".leaves.f64", dtype=np.float64).reshape(-1, 10)
                np.savez_compressed(os.path.join(OUT, f"kat_{name}.npz"), kat=kat, leaves=leaves, seed=SEED)
                print("kat", name, info["cases"], flush=True)
        jobs = [(name, v, f"image_{name}.npz") for name, v in IMAGE.items()] if "image" in what else []
        jobs += [(name, v, f"image_{name}_quarter.npz") for name, v in IMAGE_QUARTER.items()] if "image_quarter" in what else []
        if jobs:
            for name, (w, h, spp), out_name in jobs:
                if scenes and name not in scenes:
                    continue
                path = os.path.join(tmp, "i_" + name + ".f32")
                depth = run("scene", name, SEED, assets)["depth"]
                info = run("render", name, SEED, assets, w, h, spp, depth, path)
                img = np.fromfile(path, dtype=np.float32).reshape(info["height"], w, 3)
                var = np.fromfile(path + ".var", dtype=np.float32).reshape(info["height"], w, 3)
                if out_name == f"image_{name}_quarter.npz" and name in HALF_PRECISION_QUARTER:
                    img, var = img.astype(np.float16), var.astype(np.float16)
                np.savez_compressed(os.path.join(OUT, out_name), image=img, var=var, spp=spp, depth=depth, seed=SEED)
                print("image", name, w, info["height"], spp, "%.1fs" % info["seconds"], "mean", img.mean(axis=(0, 1)), flush=True)


if __name__ == "__main__":
    main(sys.argv[1:])
