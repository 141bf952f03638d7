"""ctypes binding of the C ABI in include/rt_b200.h (librt_b200.so) and of the scene
builder library (libscenes_b200.so).

There is no fallback of any kind here: if the CUDA library has not been built, or there
is no CUDA device, the calls raise.  `oracle/` is never imported from this module.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
RT_B200_ABI_VERSION = 4
RT_ACCUM_FRAC_BITS = 28

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_NOMEM, RT_ERR_STATE, RT_ERR_UNSUPPORTED, RT_ERR_KERNEL = range(7)
RT_PRIM_SPHERE, RT_PRIM_QUAD, RT_PRIM_TRIANGLE, RT_PRIM_MESH = range(4)
(RT_MAT_LAMBERTIAN, RT_MAT_METAL, RT_MAT_DIELECTRIC, RT_MAT_DIFFUSE_LIGHT, RT_MAT_EMISSIVE_LIGHT, RT_MAT_ISOTROPIC,
 RT_MAT_SPECULAR) = range(7)
RT_TEX_SOLID, RT_TEX_CHECKER, RT_TEX_CHECKER_TRIANGLE, RT_TEX_IMAGE, RT_TEX_NOISE = range(5)
RT_SHARD_AUTO, RT_SHARD_TILES, RT_SHARD_SAMPLES = range(3)
RT_FLAG_ACCUMULATE, RT_FLAG_ASYNC, RT_FLAG_STATS, RT_FLAG_NEE, RT_FLAG_SHADOWED_POINT_LIGHTS, RT_FLAG_COMPACT_TILES = 1, 2, 4, 8, 16, 32
RT_FLAG_OVERLAP = 64
RT_FLAG_MOMENTS = 128
RT_FLAG_AOV = 256
RT_FLAG_CAMERA_RAYS = 512

d3 = C.c_double * 3


class rt_xform(C.Structure):
    _fields_ = [("r", C.c_double * 9), ("t", d3)]


class rt_sphere(C.Structure):
    _fields_ = [("center0", d3), ("center_vec", d3), ("radius", C.c_double), ("material", C.c_int32), ("xform", C.c_int32)]


class rt_quad(C.Structure):
    _fields_ = [("Q", d3), ("u", d3), ("v", d3), ("material", C.c_int32), ("xform", C.c_int32)]


class rt_triangle(C.Structure):
    _fields_ = [("p0", d3), ("p1", d3), ("p2", d3), ("uv0", C.c_float * 2), ("uv1", C.c_float * 2), ("uv2", C.c_float * 2),
                ("material", C.c_int32), ("xform", C.c_int32)]


class rt_mesh(C.Structure):
    _fields_ = [("positions", C.POINTER(C.c_float)), ("indices", C.POINTER(C.c_uint32)), ("uvs", C.POINTER(C.c_float)),
                ("uv_indices", C.POINTER(C.c_uint32)), ("n_vertices", C.c_int32), ("n_triangles", C.c_int32), ("n_uvs", C.c_int32),
                ("material", C.c_int32), ("xform", C.c_int32), ("pad_", C.c_int32)]


class rt_prim_ref(C.Structure):
    _fields_ = [("type", C.c_int32), ("index", C.c_int32)]


class rt_medium(C.Structure):
    _fields_ = [("boundary_first", C.c_int32), ("boundary_count", C.c_int32), ("density", C.c_double),
                ("multiplicity", C.c_int32), ("material", C.c_int32), ("xform", C.c_int32), ("pad_", C.c_int32)]


class rt_material(C.Structure):
    _fields_ = [("type", C.c_int32), ("texture", C.c_int32), ("albedo", d3), ("param", C.c_double)]


class rt_texture(C.Structure):
    _fields_ = [("type", C.c_int32), ("even", C.c_int32), ("odd", C.c_int32), ("image", C.c_int32), ("perlin", C.c_int32),
                ("pad_", C.c_int32), ("color", d3), ("scale", C.c_double)]


class rt_image(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb", C.POINTER(C.c_uint8))]


class rt_perlin(C.Structure):
    _fields_ = [("randvec", (C.c_double * 3) * 256), ("perm_x", C.c_int32 * 256), ("perm_y", C.c_int32 * 256),
                ("perm_z", C.c_int32 * 256)]


class rt_point_light(C.Structure):
    _fields_ = [("position", d3), ("intensity", d3), ("size", C.c_double)]


class rt_camera(C.Structure):
    _fields_ = [("lookfrom", d3), ("lookat", d3), ("vup", d3), ("vfov", C.c_double), ("defocus_angle", C.c_double),
                ("focus_dist", C.c_double), ("background", d3)]


class rt_camera_ray(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("direction", C.c_float * 3), ("dx", C.c_float * 3), ("dy", C.c_float * 3)]


class rt_environment(C.Structure):
    _fields_ = [("rgb", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("rotation", C.c_double * 9)]


class rt_scene_desc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("abi_version", C.c_uint32),
        ("world", C.POINTER(rt_prim_ref)), ("n_world", C.c_int32),
        ("boundary_refs", C.POINTER(rt_prim_ref)), ("n_boundary_refs", C.c_int32),
        ("spheres", C.POINTER(rt_sphere)), ("n_spheres", C.c_int32),
        ("quads", C.POINTER(rt_quad)), ("n_quads", C.c_int32),
        ("triangles", C.POINTER(rt_triangle)), ("n_triangles", C.c_int32),
        ("media", C.POINTER(rt_medium)), ("n_media", C.c_int32),
        ("xforms", C.POINTER(rt_xform)), ("n_xforms", C.c_int32),
        ("materials", C.POINTER(rt_material)), ("n_materials", C.c_int32),
        ("textures", C.POINTER(rt_texture)), ("n_textures", C.c_int32),
        ("images", C.POINTER(rt_image)), ("n_images", C.c_int32),
        ("perlins", C.POINTER(rt_perlin)), ("n_perlins", C.c_int32),
        ("lights", C.POINTER(rt_point_light)), ("n_lights", C.c_int32),
        ("camera", rt_camera),
        ("meshes", C.POINTER(rt_mesh)), ("n_meshes", C.c_int32),
    ]


# size of an ABI-3 rt_scene_desc (everything before `meshes`), which rt_upload_scene still accepts with abi_version 3
RT_SCENE_DESC_V3_SIZE = rt_scene_desc.meshes.offset


class rt_render_params(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("width", C.c_int32), ("height", C.c_int32), ("samples_per_pixel", C.c_int32),
        ("max_depth", C.c_int32), ("spp_begin", C.c_int32), ("seed", C.c_uint64), ("tile_size", C.c_int32),
        ("shard_mode", C.c_int32), ("shard_rank", C.c_int32), ("shard_count", C.c_int32), ("flags", C.c_uint32),
        ("reserved_", C.c_int32), ("stream", C.c_void_p),
    ]


class rt_stats(C.Structure):
    _fields_ = [
        ("render_ms", C.c_double), ("upload_ms", C.c_double), ("samples", C.c_uint64), ("rays", C.c_uint64),
        ("node_visits", C.c_uint64), ("box_tests", C.c_uint64), ("sphere_tests", C.c_uint64), ("quad_tests", C.c_uint64),
        ("triangle_tests", C.c_uint64), ("medium_queries", C.c_uint64), ("boundary_tests", C.c_uint64),
        ("fp64_sphere_tests", C.c_uint64), ("nonfinite_samples", C.c_uint64), ("kernel_launches", C.c_uint32),
        ("bvh_nodes", C.c_uint32), ("bvh_depth", C.c_uint32), ("bvh_leaves", C.c_uint32), ("regs_per_thread", C.c_uint32),
        ("threads_per_block", C.c_uint32), ("blocks", C.c_uint32), ("local_bytes_per_thread", C.c_uint32),
        ("desc_iters", C.c_uint64), ("desc_lanes", C.c_uint64), ("desc_trav_lanes", C.c_uint64), ("leaf_iters", C.c_uint64),
        ("leaf_lanes", C.c_uint64), ("shade_iters", C.c_uint64), ("shade_lanes", C.c_uint64),
        ("trav_hist", C.c_uint64 * 208),
        ("bvh_on_device", C.c_uint32), ("reserved_", C.c_uint32), ("device_build_ms", C.c_double), ("device_copy_in_ms", C.c_double),
        ("device_top_ms", C.c_double),
        ("bvh_width", C.c_uint32), ("wide_nodes", C.c_uint32), ("wide_depth", C.c_uint32), ("reserved2_", C.c_uint32),
        ("empty_node_steps", C.c_uint64),
        ("devices", C.c_uint32), ("gather_mode", C.c_uint32),
        ("upload_bytes", C.c_uint64), ("scene_reused", C.c_uint32), ("reserved3_", C.c_uint32),
    ]

    def as_dict(self) -> dict:
        return {name: (list(getattr(self, name)) if name == "trav_hist" else getattr(self, name)) for name, _ in self._fields_}


EXPORTED_SYMBOLS = [
    "rt_create", "rt_destroy", "rt_last_error", "rt_upload_scene", "rt_render", "rt_sync", "rt_download", "rt_render_aov",
    "rt_accum_buffer", "rt_bind_accum", "rt_get_stats", "rt_measure_fp32_peak", "rt_probe_texture", "rt_probe_scatter",
    "rt_probe_hit", "rt_struct_size", "rt_accum_download", "rt_accum_upload", "rt_set_bvh_builder",
    "rt_set_bvh_width", "rt_device_count", "rt_shard_pixels", "rt_resolve_tiles", "rt_untile",
    "rt_download_begin", "rt_untile_begin", "rt_frame_end", "rt_measure_l1_peak", "rt_visible_devices", "rt_join",
    "rt_download_variance", "rt_moments_download", "rt_moments_upload", "rt_frame_noise",
    "rt_render_views", "rt_download_views", "rt_refit_scene", "rt_download_aov", "rt_set_camera_rays",
    "rt_set_environment",
]

ABI_STRUCTS = [rt_scene_desc, rt_render_params, rt_stats, rt_sphere, rt_quad, rt_triangle, rt_medium, rt_material, rt_texture,
               rt_image, rt_perlin, rt_point_light, rt_camera, rt_xform, rt_prim_ref, rt_mesh, rt_camera_ray,
               rt_environment]

_lib = None
_scenes = None


class RtError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"rt_b200 error {code}: {message}")
        self.code = code


def lib_path() -> str:
    # RT_B200_LIB: an alternative build of the same library (tuning experiments, tools/perf_sweep.py)
    return os.environ.get("RT_B200_LIB") or os.path.join(_PKG, "librt_b200.so")


def scenes_lib_path() -> str:
    return os.path.join(_PKG, "libscenes_b200.so")


def load() -> C.CDLL:
    """Load librt_b200.so.  Raises (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, i32, f32p, i32p = C.c_void_p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_int32)
    lib.rt_create.argtypes = [C.POINTER(vp), i32p, C.c_int]
    lib.rt_destroy.argtypes = [vp]
    lib.rt_destroy.restype = None
    lib.rt_last_error.argtypes = [vp]
    lib.rt_last_error.restype = C.c_char_p
    lib.rt_upload_scene.argtypes = [vp, C.POINTER(rt_scene_desc)]
    lib.rt_refit_scene.argtypes = [vp, C.POINTER(rt_scene_desc)]
    lib.rt_render.argtypes = [vp, C.POINTER(rt_render_params)]
    lib.rt_sync.argtypes = [vp]
    lib.rt_join.argtypes = [vp, vp]
    lib.rt_download.argtypes = [vp, i32, vp, vp]
    lib.rt_render_aov.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    lib.rt_accum_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.rt_bind_accum.argtypes = [vp, vp, C.c_size_t, i32, i32]
    lib.rt_get_stats.argtypes = [vp, C.POINTER(rt_stats)]
    lib.rt_set_bvh_builder.argtypes = [vp, i32]
    lib.rt_set_bvh_width.argtypes = [vp, i32]
    lib.rt_device_count.argtypes = [vp]
    lib.rt_shard_pixels.argtypes = [i32, i32, i32, i32, i32]
    lib.rt_shard_pixels.restype = C.c_size_t
    lib.rt_resolve_tiles.argtypes = [vp, i32, vp, vp, C.c_size_t]
    lib.rt_untile.argtypes = [vp, vp, C.c_size_t, i32, i32, i32, i32, i32, vp]
    lib.rt_download_begin.argtypes = [vp, i32, i32, i32]
    lib.rt_untile_begin.argtypes = [vp, vp, C.c_size_t, i32, i32, i32, i32, i32]
    lib.rt_frame_end.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.rt_accum_download.argtypes = [vp, vp, C.c_size_t]
    lib.rt_accum_upload.argtypes = [vp, vp, C.c_size_t, i32, i32]
    lib.rt_download_variance.argtypes = [vp, i32, vp]
    lib.rt_moments_download.argtypes = [vp, vp, C.c_size_t]
    lib.rt_moments_upload.argtypes = [vp, vp, C.c_size_t, i32, i32]
    lib.rt_frame_noise.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.rt_download_aov.argtypes = [vp, i32, vp]
    lib.rt_set_camera_rays.argtypes = [vp, vp, i32, i32]
    lib.rt_set_environment.argtypes = [vp, C.POINTER(rt_environment)]
    lib.rt_render_views.argtypes = [vp, C.POINTER(rt_render_params), C.POINTER(rt_camera), C.POINTER(C.c_uint64), i32]
    lib.rt_download_views.argtypes = [vp, i32, i32, i32, vp, vp]
    lib.rt_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double)]
    lib.rt_measure_l1_peak.argtypes = [vp, C.POINTER(C.c_double)]
    lib.rt_probe_texture.argtypes = [vp, i32, i32, vp, vp]
    lib.rt_probe_scatter.argtypes = [vp, i32, i32, vp, vp, vp]
    lib.rt_probe_hit.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.rt_struct_size.argtypes = [C.c_int]
    lib.rt_struct_size.restype = C.c_size_t
    for which, struct in enumerate(ABI_STRUCTS):
        if lib.rt_struct_size(which) != C.sizeof(struct):
            raise ImportError(f"ABI mismatch: {struct.__name__} is {C.sizeof(struct)} bytes here, "
                              f"{lib.rt_struct_size(which)} in {path}")
    _lib = lib
    return lib


def load_scenes() -> C.CDLL:
    global _scenes
    if _scenes is not None:
        return _scenes
    load()
    path = scenes_lib_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run __graft_entry__.build()")
    s = C.CDLL(path)
    s.rtsc_scene_count.restype = C.c_int
    s.rtsc_scene_name.argtypes = [C.c_int]
    s.rtsc_scene_name.restype = C.c_char_p
    s.rtsc_build.argtypes = [C.c_char_p, C.c_uint, C.c_char_p]
    s.rtsc_build.restype = C.c_void_p
    s.rtsc_set_indexed_meshes.argtypes = [C.c_int]
    s.rtsc_set_indexed_meshes.restype = C.c_int
    s.rtsc_desc.argtypes = [C.c_void_p]
    s.rtsc_desc.restype = C.POINTER(rt_scene_desc)
    s.rtsc_frame.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 4
    s.rtsc_frame.restype = None
    s.rtsc_free.argtypes = [C.c_void_p]
    s.rtsc_free.restype = None
    s.rtsc_render_png.argtypes = [C.c_char_p, C.c_uint, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p]
    s.rtsc_render_resumable.argtypes = [C.c_char_p, C.c_uint, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_char_p,
                                        C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    s.rtsc_render_turntable.argtypes = [C.c_char_p, C.c_uint, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int,
                                        C.c_int, C.c_int]
    s.rtsc_turntable_camera.argtypes = [C.c_char_p, C.c_uint, C.c_char_p, C.c_int, C.c_int, C.POINTER(rt_camera)]
    s.rtsc_panorama_rays.argtypes = [C.c_char_p, C.c_uint, C.c_char_p, C.c_int, C.c_int, C.POINTER(rt_camera_ray)]
    s.rtsc_write_exr.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p]
    s.rtsc_write_pfm.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p]
    s.rtsc_read_pfm.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p, C.c_size_t]
    s.rtsc_load_obj.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_double)]
    s.rtsc_load_obj.restype = C.c_void_p
    s.rtsc_scene_hash.argtypes = [C.c_void_p]
    s.rtsc_scene_hash.restype = C.c_uint64
    _scenes = s
    return s


class indexed_meshes:
    """`with indexed_meshes(True):` the scene builder loads OBJ files as indexed meshes (rt_mesh) instead of
    triangle soups -- for Scene and for the camera::render entry points (rtsc_render_png, rtsc_render_resumable)."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        self._was = load_scenes().rtsc_set_indexed_meshes(int(self.on))
        return self

    def __exit__(self, *exc):
        load_scenes().rtsc_set_indexed_meshes(self._was)


class Scene:
    """A BASELINE scene built by the C++ host mirror (scenes/scenes.h) and flattened.  indexed=True loads its OBJ
    files as indexed meshes (rt_mesh) instead of rt_triangle records: same triangles, same image."""

    def __init__(self, name: str, seed: int = 1, asset_dir: Optional[str] = None, indexed: bool = False):
        from .assets import ensure_assets

        self.name = name
        self._s = load_scenes()
        asset_dir = ensure_assets(asset_dir)
        with indexed_meshes(indexed):
            self._h = self._s.rtsc_build(name.encode(), seed, asset_dir.encode())
        if not self._h:
            raise ValueError(f"unknown scene {name!r}")
        self.desc_ptr = self._s.rtsc_desc(self._h)
        w, h, spp, depth = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._s.rtsc_frame(self._h, C.byref(w), C.byref(h), C.byref(spp), C.byref(depth))
        self.width, self.height, self.spp, self.depth = w.value, h.value, spp.value, depth.value

    @property
    def desc(self) -> rt_scene_desc:
        return self.desc_ptr.contents

    def close(self):
        if self._h:
            self._s.rtsc_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ObjScene(Scene):
    """An OBJ file loaded by the host mirror's mesh::loadObj: the fast path (one triangle_soup), with indexed=True
    the fast path into one indexed mesh (rt_mesh), or with per_triangle=True the reference's structure."""

    def __init__(self, path: str, per_triangle: bool = False, with_media: bool = False, scale: float = 1.0, indexed: bool = False):
        if per_triangle and indexed:
            raise ValueError("per_triangle and indexed are two different loaders")
        self.name = path
        self._s = load_scenes()
        ms = (C.c_double * 2)()
        self._h = self._s.rtsc_load_obj(path.encode(), 2 if indexed else int(per_triangle), int(with_media), scale, ms)
        if not self._h:
            raise ValueError(f"cannot load {path!r}")
        self.load_ms, self.flatten_ms = ms[0], ms[1]
        self.desc_ptr = self._s.rtsc_desc(self._h)
        w, h, spp, depth = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._s.rtsc_frame(self._h, C.byref(w), C.byref(h), C.byref(spp), C.byref(depth))
        self.width, self.height, self.spp, self.depth = w.value, h.value, spp.value, depth.value

    @property
    def hash(self) -> int:
        return self._s.rtsc_scene_hash(self._h)


def scene_names() -> list:
    s = load_scenes()
    return [s.rtsc_scene_name(i).decode() for i in range(s.rtsc_scene_count())]


class Context:
    """One rt_ctx: one GPU (device = an index) or several GPUs of this box (device = a list of indices)."""

    def __init__(self, device=0):
        self.lib = load()
        self._h = C.c_void_p()
        ids = [device] if isinstance(device, int) else list(device)
        dev = (C.c_int32 * max(1, len(ids)))(*ids)
        rc = self.lib.rt_create(C.byref(self._h), dev, len(ids))
        if rc != RT_OK:
            msg = self.lib.rt_last_error(self._h).decode() if self._h else "rt_create failed"
            if self._h:
                self.lib.rt_destroy(self._h)
                self._h = C.c_void_p()
            raise RtError(rc, msg)
        self.width = self.height = 0

    def _check(self, rc: int):
        if rc != RT_OK:
            raise RtError(rc, self.lib.rt_last_error(self._h).decode())

    def set_bvh_builder(self, mode: str) -> None:
        """'auto' | 'host' (binned SAH on the CPU) | 'device' (LBVH in CUDA kernels + SAH top levels) |
        'lbvh' (device, pure LBVH) for the next upload."""
        self._check(self.lib.rt_set_bvh_builder(self._h, {"auto": 0, "host": 1, "device": 2, "lbvh": 3}[mode]))

    def set_bvh_width(self, width: int) -> None:
        """2 (binary tree) | 4 | 8 (wide quantised tree) for the next upload."""
        self._check(self.lib.rt_set_bvh_width(self._h, width))

    @staticmethod
    def _desc_ptr(scene):
        if hasattr(scene, "desc_ptr"):          # capi.Scene or any object that keeps a description alive
            return scene.desc_ptr
        if isinstance(scene, rt_scene_desc):
            return C.pointer(scene)
        return scene

    def upload(self, scene) -> None:
        self._check(self.lib.rt_upload_scene(self._h, self._desc_ptr(scene)))

    def refit(self, scene) -> None:
        """rt_refit_scene: replace the uploaded scene by `scene`, which has its structure (same counts, primitive kinds,
        emitters and media classes) but may move, without a tree build: the tree keeps its topology, its boxes are
        recomputed.  Takes what upload() takes."""
        self._check(self.lib.rt_refit_scene(self._h, self._desc_ptr(scene)))

    def render(self, width: int, height: int, spp: int, max_depth: int = 50, seed: int = 1, spp_begin: int = 0,
               accumulate: bool = False, stats: bool = False, shard_rank: int = 0, shard_count: int = 1,
               shard_mode: int = RT_SHARD_AUTO, tile_size: int = 0, stream: Optional[int] = None, blocking: bool = True,
               nee: bool = False, shadowed_point_lights: bool = False, compact: bool = False, overlap: bool = False,
               moments: bool = False, aov: bool = False, camera_rays: bool = False) -> None:
        """camera_rays=True traces the primary rays set with set_camera_rays() instead of the uploaded camera's."""
        p = rt_render_params()
        p.struct_size = C.sizeof(rt_render_params)
        p.width, p.height, p.samples_per_pixel, p.max_depth = width, height, spp, max_depth
        p.spp_begin, p.seed, p.tile_size = spp_begin, seed, tile_size
        p.shard_mode, p.shard_rank, p.shard_count = shard_mode, shard_rank, shard_count
        p.flags = ((RT_FLAG_ACCUMULATE if accumulate else 0) | (RT_FLAG_STATS if stats else 0) | (0 if blocking else RT_FLAG_ASYNC) |
                   (RT_FLAG_NEE if nee else 0) | (RT_FLAG_SHADOWED_POINT_LIGHTS if shadowed_point_lights else 0) |
                   (RT_FLAG_COMPACT_TILES if compact else 0) | (RT_FLAG_OVERLAP if overlap else 0) | (RT_FLAG_MOMENTS if moments else 0) |
                   (RT_FLAG_AOV if aov else 0) | (RT_FLAG_CAMERA_RAYS if camera_rays else 0))
        p.stream = stream
        self._check(self.lib.rt_render(self._h, C.byref(p)))
        self.width, self.height = width, height

    def set_camera_rays(self, rays) -> None:
        """rt_set_camera_rays: one primary ray per pixel for render(..., camera_rays=True), an (H, W, 12) float32 array
        (numpy, or a contiguous CPU tensor) of rt_camera_ray records: origin, direction through the pixel centre, and the
        change of the direction per pixel in x and in y.  None frees them."""
        if rays is None:
            self._check(self.lib.rt_set_camera_rays(self._h, None, 0, 0))
            return
        if hasattr(rays, "numpy"):  # a torch tensor: its CPU memory as it is
            if rays.device.type != "cpu" or not rays.is_contiguous():
                raise ValueError("camera rays must be a contiguous CPU tensor")
            rays = rays.numpy()
        a = np.asarray(rays)
        if a.dtype != np.float32 or a.ndim != 3 or a.shape[2] != 12:
            raise ValueError(f"camera rays must be an (H, W, 12) float32 array, got {a.dtype} {a.shape}")
        a = np.ascontiguousarray(a)
        self._check(self.lib.rt_set_camera_rays(self._h, a.ctypes.data, a.shape[1], a.shape[0]))

    def set_environment(self, rgb, rotation=None) -> None:
        """rt_set_environment: an equirectangular map of linear radiance seen by every ray that leaves the scene, an
        (H, W, 3) float32 array (numpy, or a contiguous CPU tensor), row 0 at the +y pole; rotation: the 3x3 rotation from
        the map frame to the world (identity by default).  None goes back to the camera's background."""
        if rgb is None:
            self._check(self.lib.rt_set_environment(self._h, None))
            return
        if hasattr(rgb, "numpy"):  # a torch tensor: its CPU memory as it is
            if rgb.device.type != "cpu" or not rgb.is_contiguous():
                raise ValueError("an environment map must be a contiguous CPU tensor")
            rgb = rgb.numpy()
        a = np.asarray(rgb)
        if a.dtype != np.float32 or a.ndim != 3 or a.shape[2] != 3:
            raise ValueError(f"an environment map must be an (H, W, 3) float32 array, got {a.dtype} {a.shape}")
        a = np.ascontiguousarray(a)
        r = np.eye(3) if rotation is None else np.asarray(rotation, dtype=np.float64)
        if r.shape != (3, 3):
            raise ValueError(f"the rotation must be 3x3, got {r.shape}")
        e = rt_environment()
        e.rgb = a.ctypes.data
        e.width, e.height = a.shape[1], a.shape[0]
        e.rotation = (C.c_double * 9)(*r.reshape(9).tolist())
        self._check(self.lib.rt_set_environment(self._h, C.byref(e)))

    def render_views(self, cameras, width: int, height: int, spp: int, max_depth: int = 50, seed: int = 1, seeds=None,
                     spp_begin: int = 0, accumulate: bool = False, blocking: bool = True, nee: bool = False,
                     shadowed_point_lights: bool = False, tile_size: int = 0, stream: Optional[int] = None) -> None:
        """Render the uploaded scene from every rt_camera of `cameras` in one pass (rt_render_views), into the context's
        views frame.  View v equals render() of the scene uploaded with cameras[v], seeded with seeds[v] (or `seed`)."""
        cams = list(cameras)
        arr = (rt_camera * max(1, len(cams)))(*cams)
        seed_arr = None
        if seeds is not None:
            seeds = list(seeds)
            if len(seeds) != len(cams):
                raise ValueError(f"{len(seeds)} seeds for {len(cams)} cameras")
            seed_arr = (C.c_uint64 * max(1, len(seeds)))(*seeds)
        p = rt_render_params()
        p.struct_size = C.sizeof(rt_render_params)
        p.width, p.height, p.samples_per_pixel, p.max_depth = width, height, spp, max_depth
        p.spp_begin, p.seed, p.tile_size = spp_begin, seed, tile_size
        p.flags = ((RT_FLAG_ACCUMULATE if accumulate else 0) | (0 if blocking else RT_FLAG_ASYNC) | (RT_FLAG_NEE if nee else 0) |
                   (RT_FLAG_SHADOWED_POINT_LIGHTS if shadowed_point_lights else 0))
        p.stream = stream
        self._check(self.lib.rt_render_views(self._h, C.byref(p), arr if cams else None, seed_arr, len(cams)))
        self.views_shape = (len(cams), height, width)

    def download_views(self, total_spp: int, first: int = 0, count: Optional[int] = None, linear: bool = True, rgb8: bool = False):
        """Views [first, first + count) of the views frame as (count, H, W, 3) arrays: float32 radiance and / or RGB8,
        each view laid out like download()."""
        n, h, w = getattr(self, "views_shape", (0, 0, 0))
        if count is None:
            count = n - first
        shape = (max(count, 0), h, w, 3)
        lin = np.empty(shape, dtype=np.float32) if linear else None
        b8 = np.empty(shape, dtype=np.uint8) if rgb8 else None
        self._check(self.lib.rt_download_views(self._h, total_spp, first, count, lin.ctypes.data if linear else None,
                                               b8.ctypes.data if rgb8 else None))
        if linear and rgb8:
            return lin, b8
        return lin if linear else b8

    def sync(self) -> None:
        self._check(self.lib.rt_sync(self._h))

    def join(self, stream: Optional[int] = None) -> None:
        """Stream-ordered join (no host wait): `stream` runs on after every pass still in flight (RT_FLAG_OVERLAP)."""
        self._check(self.lib.rt_join(self._h, stream))

    def download(self, total_spp: int, linear: bool = True, rgb8: bool = False):
        n = self.width * self.height
        lin = np.empty((self.height, self.width, 3), dtype=np.float32) if linear else None
        b8 = np.empty((self.height, self.width, 3), dtype=np.uint8) if rgb8 else None
        self._check(self.lib.rt_download(self._h, total_spp, lin.ctypes.data if linear else None, b8.ctypes.data if rgb8 else None))
        assert n >= 0
        if linear and rgb8:
            return lin, b8
        return lin if linear else b8

    def aov(self, width: int, height: int) -> dict:
        n = width * height
        out = {
            "prim_id": np.empty(n, dtype=np.int32), "t": np.empty(n, dtype=np.float32),
            "normal": np.empty((n, 3), dtype=np.float32), "point": np.empty((n, 3), dtype=np.float32),
            "uv": np.empty((n, 2), dtype=np.float32),
        }
        self._check(self.lib.rt_render_aov(self._h, width, height, *[out[k].ctypes.data for k in ("prim_id", "t", "normal", "point", "uv")]))
        return out

    def device_count(self) -> int:
        return self.lib.rt_device_count(self._h)

    def resolve_tiles(self, total_spp: int, dev_rgb8: Optional[int], capacity_pixels: int, dev_linear: Optional[int] = None) -> None:
        """The compact tiles of the last compact render -> RGB8 / float radiance in caller-owned DEVICE buffers."""
        self._check(self.lib.rt_resolve_tiles(self._h, total_spp, dev_linear, dev_rgb8, capacity_pixels))

    def untile(self, dev_shards: int, shard_stride_bytes: int, bytes_per_pixel: int, shard_count: int, width: int, height: int,
               tile_size: int = 16) -> np.ndarray:
        """`shard_count` compact buffers side by side on this context's device -> the full frame (host array)."""
        if bytes_per_pixel == 3:
            out = np.empty((height, width, 3), dtype=np.uint8)
        elif bytes_per_pixel == 12:
            out = np.empty((height, width, 3), dtype=np.float32)
        else:
            out = np.empty((height, width, 4), dtype=np.uint64)
        self._check(self.lib.rt_untile(self._h, dev_shards, shard_stride_bytes, bytes_per_pixel, shard_count, width, height, tile_size,
                                       out.ctypes.data))
        return out

    def download_begin(self, total_spp: int, linear: bool = False, rgb8: bool = True) -> None:
        """Queue resolve + device-to-host copy (pinned memory, own stream) and return; pair with frame_end()."""
        self._check(self.lib.rt_download_begin(self._h, total_spp, int(linear), int(rgb8)))

    def untile_begin(self, dev_shards: int, shard_stride_bytes: int, bytes_per_pixel: int, shard_count: int, width: int, height: int,
                     tile_size: int = 16) -> None:
        self._check(self.lib.rt_untile_begin(self._h, dev_shards, shard_stride_bytes, bytes_per_pixel, shard_count, width, height, tile_size))
        self.width, self.height = width, height

    def frame_end(self):
        """(linear, rgb8) numpy VIEWS of the context's pinned buffer for the oldest outstanding begin (None for a plane
        that was not asked for); valid until two more begins."""
        lin, b8 = C.c_void_p(), C.c_void_p()
        self._check(self.lib.rt_frame_end(self._h, C.byref(lin), C.byref(b8)))
        n = self.width * self.height * 3
        a = np.ctypeslib.as_array((C.c_float * n).from_address(lin.value)).reshape(self.height, self.width, 3) if lin.value else None
        b = np.ctypeslib.as_array((C.c_uint8 * n).from_address(b8.value)).reshape(self.height, self.width, 3) if b8.value else None
        return a, b

    def accum_buffer(self):
        ptr, nbytes = C.c_void_p(), C.c_size_t()
        self._check(self.lib.rt_accum_buffer(self._h, C.byref(ptr), C.byref(nbytes)))
        return ptr.value, nbytes.value

    def bind_accum(self, device_ptr: Optional[int], nbytes: int, width: int, height: int) -> None:
        self._check(self.lib.rt_bind_accum(self._h, device_ptr, nbytes, width, height))
        self.width, self.height = width, height

    def accum_download(self) -> np.ndarray:
        """The raw frame sums (H, W, 4) uint64: R, G, B in 2^-28 units and the dropped-sample count."""
        out = np.empty((self.height, self.width, 4), dtype=np.uint64)
        self._check(self.lib.rt_accum_download(self._h, out.ctypes.data, out.nbytes))
        return out

    def accum_upload(self, sums: np.ndarray) -> None:
        sums = np.ascontiguousarray(sums, dtype=np.uint64)
        h, w = sums.shape[0], sums.shape[1]
        self._check(self.lib.rt_accum_upload(self._h, sums.ctypes.data, sums.nbytes, w, h))
        self.width, self.height = w, h

    def download_variance(self, total_spp: int) -> np.ndarray:
        """Unbiased per-sample variance (H, W, 3) float32 of a frame rendered with moments=True."""
        out = np.empty((self.height, self.width, 3), dtype=np.float32)
        self._check(self.lib.rt_download_variance(self._h, total_spp, out.ctypes.data))
        return out

    def moments_download(self) -> np.ndarray:
        """The raw second moments (H, W, 6) uint64: per channel the sums of the low and the high 48 bits of x^2."""
        out = np.empty((self.height, self.width, 6), dtype=np.uint64)
        self._check(self.lib.rt_moments_download(self._h, out.ctypes.data, out.nbytes))
        return out

    def moments_upload(self, m: np.ndarray) -> None:
        """Restore the moments of the frame accum_upload() restored just before."""
        m = np.ascontiguousarray(m, dtype=np.uint64)
        self._check(self.lib.rt_moments_upload(self._h, m.ctypes.data, m.nbytes, m.shape[1], m.shape[0]))

    def frame_noise(self, total_spp: int):
        """(mean linear radiance, RMS standard error of the pixel mean) of a frame rendered with moments=True."""
        mean, rms = C.c_double(), C.c_double()
        self._check(self.lib.rt_frame_noise(self._h, total_spp, C.byref(mean), C.byref(rms)))
        return mean.value, rms.value

    def download_aov(self, total_spp: int) -> dict:
        """The auxiliary outputs of a frame rendered with aov=True: `albedo` (H, W, 3), `normal` (H, W, 3), `depth` (H, W)
        and `coverage` (H, W) float32, views of one (H, W, 8) array (their `.base`)."""
        out = np.empty((self.height, self.width, 8), dtype=np.float32)
        self._check(self.lib.rt_download_aov(self._h, total_spp, out.ctypes.data))
        return {"albedo": out[..., 0:3], "normal": out[..., 3:6], "depth": out[..., 6], "coverage": out[..., 7]}

    def stats(self) -> dict:
        st = rt_stats()
        self._check(self.lib.rt_get_stats(self._h, C.byref(st)))
        return st.as_dict()

    def measure_fp32_peak(self) -> float:
        v = C.c_double()
        self._check(self.lib.rt_measure_fp32_peak(self._h, C.byref(v)))
        return v.value

    def measure_l1_peak(self) -> float:
        v = C.c_double()
        self._check(self.lib.rt_measure_l1_peak(self._h, C.byref(v)))
        return v.value

    def probe_texture(self, texture: int, uvp: np.ndarray) -> np.ndarray:
        uvp = np.ascontiguousarray(uvp, dtype=np.float32).reshape(-1, 5)
        out = np.empty((uvp.shape[0], 3), dtype=np.float32)
        self._check(self.lib.rt_probe_texture(self._h, texture, uvp.shape[0], uvp.ctypes.data, out.ctypes.data))
        return out

    def probe_scatter(self, material: int, records: np.ndarray, uniforms: np.ndarray) -> np.ndarray:
        records = np.ascontiguousarray(records, dtype=np.float32).reshape(-1, 16)
        uniforms = np.ascontiguousarray(uniforms, dtype=np.float32).reshape(-1, 4)
        out = np.empty((records.shape[0], 16), dtype=np.float32)
        self._check(self.lib.rt_probe_scatter(self._h, material, records.shape[0], records.ctypes.data, uniforms.ctypes.data, out.ctypes.data))
        return out

    def probe_hit(self, rays: np.ndarray) -> dict:
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 9)
        n = rays.shape[0]
        out = {"prim_id": np.empty(n, dtype=np.int32), "t": np.empty(n, dtype=np.float32),
               "normal": np.empty((n, 3), dtype=np.float32), "uv": np.empty((n, 2), dtype=np.float32)}
        self._check(self.lib.rt_probe_hit(self._h, n, rays.ctypes.data, *[out[k].ctypes.data for k in ("prim_id", "t", "normal", "uv")]))
        return out

    def close(self):
        if self._h:
            self.lib.rt_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
