"""In-tree build of the native pieces (no JIT cache: the .so files travel with the repo
snapshot to the GPU box).

  librt_b200.so      csrc/rt_b200.cu       nvcc, sm_100a only      the product
  libscenes_b200.so  scenes/scenes_capi.cpp g++                     host mirror + BASELINE scenes
  apps/rtow_b200     apps/rtow_main.cpp     g++                     the reference's main(), Linux
  oracle/...         oracle/Makefile        g++                     the CPU checkers (tests only)
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def _newer(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources if os.path.exists(s))


def _run(cmd, cwd=None):
    print("+", " ".join(cmd), flush=True)
    subprocess.check_call(cmd, cwd=cwd)


def build_cuda(force: bool = False, verbose_ptxas: bool = False) -> str:
    out = os.path.join(PKG, "librt_b200.so")
    csrc = os.path.join(PKG, "csrc")
    srcs = [os.path.join(csrc, f) for f in os.listdir(csrc)] + [os.path.join(ROOT, "include", "rt_b200.h")]
    if force or _newer(out, srcs):
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        cmd = [nvcc, *NVCC_FLAGS, "-I" + os.path.join(ROOT, "include"), "-o", out, os.path.join(csrc, "rt_b200.cu"), "-ldl"]
        if verbose_ptxas:
            cmd[1:1] = ["-Xptxas", "-v"]
        _run(cmd)
    return out


REFERENCE = "/root/reference"


def ensure_reference_assets() -> str | None:
    """Where the reference tree is mounted, its two shipped inputs (monkey.obj, Images/earthmap.jpg: BASELINE
    configs[3] / configs[4]) are copied into the git-ignored scenes/assets/reference/ so that the `monkey` scene can be
    built by both header sets and travels to the GPU box like the other built artefacts.  Never committed."""
    dst = os.path.join(ROOT, "scenes", "assets", "reference")
    pairs = [(os.path.join(REFERENCE, "monkey.obj"), "monkey.obj"), (os.path.join(REFERENCE, "Images", "earthmap.jpg"), "earthmap.jpg")]
    if all(os.path.exists(s) for s, _ in pairs):
        os.makedirs(dst, exist_ok=True)
        for src, name in pairs:
            if _newer(os.path.join(dst, name), [src]):
                shutil.copyfile(src, os.path.join(dst, name))
    return dst if all(os.path.exists(os.path.join(dst, n)) for _, n in pairs) else None


def build_host(force: bool = False) -> str:
    out = os.path.join(PKG, "libscenes_b200.so")
    host = os.path.join(PKG, "host")
    inc = ["-I" + os.path.join(ROOT, "include"), "-I" + host, "-I" + os.path.join(ROOT, "scenes")]
    # JPEG textures are decoded by the USER'S stb_image.h (host I/O outside the hot path): available where the
    # reference tree is mounted; elsewhere the prebuilt library travels, or the mirror reads PPM only
    if os.path.exists(os.path.join(REFERENCE, "stb_image.h")):
        inc += ["-DRTB200_USE_STB_IMAGE", "-idirafter", REFERENCE]
    srcs = [os.path.join(host, "rtow_host.h"), os.path.join(host, "png_write.h"), os.path.join(host, "frame_io.h"), os.path.join(host, "host_rng.h"),
            os.path.join(ROOT, "scenes", "scenes.h"), os.path.join(ROOT, "scenes", "scenes_capi.cpp"),
            os.path.join(ROOT, "include", "rt_b200.h")]
    if force or _newer(out, srcs):
        _run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", *inc, "-o", out, os.path.join(ROOT, "scenes", "scenes_capi.cpp"),
              "-L" + PKG, "-lrt_b200", "-Wl,-rpath,$ORIGIN"])
    app = os.path.join(ROOT, "apps", "rtow_b200")
    if force or _newer(app, srcs + [os.path.join(ROOT, "apps", "rtow_main.cpp")]):
        _run(["g++", "-O2", "-std=c++17", *inc, "-o", app, os.path.join(ROOT, "apps", "rtow_main.cpp"), "-L" + PKG, "-lrt_b200",
              "-Wl,-rpath,$ORIGIN/../raytracingoneweekendapplication_b200"])
    return out


def build_oracle() -> None:
    """The CPU checkers: the restatement always; the real reference when /root/reference exists."""
    _run(["make", "-C", os.path.join(ROOT, "oracle"), "all"])


def build_all(force: bool = False) -> None:
    build_cuda(force)
    build_host(force)
    build_oracle()
    from .assets import ensure_assets

    ensure_assets()
    ensure_reference_assets()


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
