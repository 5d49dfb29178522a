"""rtnw-b200: ctypes bindings over the two C-ABI libraries of this package.

    lib/librtnw_host.so  host scene API, flattener and chapter scene builders (include/rtnw_host.h)
    lib/librtnw.so       sm_100a kernels + C-ABI (include/rtnw.h)

The package directory name contains hyphens, so import it with
``importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")`` (tests/conftest.py does that once and
exposes it as ``rtnw``).  Nothing here computes: every call forwards to the CUDA library, and loading fails loudly
when the library is missing (there is no CPU fallback and nothing under oracle/ is ever imported from here).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
REPO_ROOT = PKG_DIR.parent
LIB_DIR = PKG_DIR / "lib"

RTNW_ABI_VERSION = 5
RTNW_OK = 0
RTNW_ERR_INVALID, RTNW_ERR_CUDA, RTNW_ERR_UNSUPPORTED, RTNW_ERR_NOMEM = -1, -2, -3, -4
BG_BLACK, BG_SKY = 0, 1
TEXF_BILINEAR = 1
F_DE_NAN, F_EMIT, F_FAST_BVH, F_COUNTERS, F_ACCUMULATE, F_ROTATE_SAMPLES, F_LIGHT_SAMPLING = 1, 2, 4, 8, 16, 32, 64
F_NEXT_EVENT = 128
FLT_MAX = float(np.finfo(np.float32).max)


class RtnwError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rtnw status {code}: {msg}")
        self.code = code


# ------------------------------------------------------------------------------------------------ C structs
class Prim(C.Structure):
    _fields_ = [("f", C.c_float * 6), ("kx", C.c_uint32), ("mat", C.c_int32)]


class XformOp(C.Structure):
    _fields_ = [("a", C.c_float), ("b", C.c_float), ("c", C.c_float), ("kind", C.c_uint32)]


class BvhNode(C.Structure):
    _fields_ = [("lmin", C.c_float * 3), ("left", C.c_int32), ("lmax", C.c_float * 3), ("right", C.c_int32),
                ("rmin", C.c_float * 3), ("lcount", C.c_int32), ("rmax", C.c_float * 3), ("rcount", C.c_int32)]


class Item(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("xform", C.c_uint32), ("first", C.c_int32), ("count", C.c_int32),
                ("bmin", C.c_float * 3), ("flip", C.c_uint32), ("bmax", C.c_float * 3), ("pad", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("tex", C.c_int32), ("f", C.c_float), ("pad0", C.c_uint32),
                ("albedo", C.c_float * 3), ("pad1", C.c_uint32)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("i0", C.c_int32), ("i1", C.c_int32), ("i2", C.c_int32),
                ("c", C.c_float * 3), ("flags", C.c_uint32)]


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32),
                ("n_items", C.c_int32), ("items", C.POINTER(Item)),
                ("n_nodes", C.c_int32), ("nodes", C.POINTER(BvhNode)),
                ("n_prim_slots", C.c_int32), ("prims", C.POINTER(Prim)),
                ("prim_ids", C.POINTER(C.c_int32)),
                ("n_xform_ops", C.c_int32), ("xforms", C.POINTER(XformOp)),
                ("n_materials", C.c_int32), ("materials", C.POINTER(Material)),
                ("n_textures", C.c_int32), ("textures", C.POINTER(Texture)),
                ("image_bytes", C.c_uint64), ("images", C.POINTER(C.c_uint8)),
                ("perlin_ranvec", C.POINTER(C.c_float)),
                ("perlin_perm_x", C.POINTER(C.c_int32)),
                ("perlin_perm_y", C.POINTER(C.c_int32)),
                ("perlin_perm_z", C.POINTER(C.c_int32))]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("lower_left_corner", C.c_float * 3), ("horizontal", C.c_float * 3),
                ("vertical", C.c_float * 3), ("u", C.c_float * 3), ("v", C.c_float * 3), ("w", C.c_float * 3),
                ("lens_radius", C.c_float), ("time0", C.c_float), ("time1", C.c_float)]


class RenderParams(C.Structure):
    _fields_ = [("nx", C.c_int32), ("ny", C.c_int32), ("sample_begin", C.c_int32), ("sample_count", C.c_int32),
                ("sample_stride", C.c_int32), ("max_depth", C.c_int32), ("t_min", C.c_float), ("t_max", C.c_float),
                ("background", C.c_uint32), ("flags", C.c_uint32), ("seed", C.c_uint64),
                ("pixel_begin", C.c_int32), ("pixel_stride", C.c_int32), ("pixel_count", C.c_int32), ("sample_ranges", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("box_tests", C.c_uint64), ("prim_tests", C.c_uint64),
                ("kernel_ms", C.c_float), ("total_ms", C.c_float), ("kernel_launches", C.c_int32), ("sample_ranges", C.c_int32)]


class Aov(C.Structure):
    """rtnw_aov: the host buffers rtnw_render_aov fills"""
    _fields_ = [("albedo", C.c_void_p), ("normal", C.c_void_p), ("depth", C.c_void_p), ("hits", C.c_void_p), ("prim_id", C.c_void_p)]


class DenoiseParams(C.Structure):
    """rtnw_denoise_params; the defaults are RTNW_DENOISE_DEFAULTS"""
    _fields_ = [("iterations", C.c_int32), ("sigma_luminance", C.c_float), ("sigma_depth", C.c_float),
                ("normal_power_log2", C.c_int32)]


class HostView(C.Structure):
    _fields_ = [("nx", C.c_int32), ("ny", C.c_int32), ("ns", C.c_int32), ("t_min", C.c_float),
                ("background", C.c_uint32), ("flags", C.c_uint32)]


# numpy views of the two array-of-struct types that cross the ABI in bulk
RAY_DTYPE = np.dtype([("origin", np.float32, 3), ("direction", np.float32, 3), ("time", np.float32), ("key", np.uint32)])
HIT_DTYPE = np.dtype([("prim_id", np.int32), ("sub_id", np.int32), ("t", np.float32), ("p", np.float32, 3),
                      ("normal", np.float32, 3), ("u", np.float32), ("v", np.float32), ("mat_id", np.int32)])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 48

# every symbol include/rtnw.h and include/rtnw_host.h declare (tests check the libraries export all of them)
DEVICE_SYMBOLS = ["rtnw_last_error", "rtnw_abi_version", "rtnw_device_count", "rtnw_ctx_create", "rtnw_ctx_destroy",
                  "rtnw_ctx_info", "rtnw_measure_fp32_peak", "rtnw_selftest_recip", "rtnw_quantize_device", "rtnw_scene_upload", "rtnw_scene_free", "rtnw_render", "rtnw_render_device", "rtnw_trace",
                  "rtnw_eval_texture", "rtnw_eval_perlin", "rtnw_scatter", "rtnw_camera_rays", "rtnw_camera_get_rays", "rtnw_plan_sample_ranges",
                  "rtnw_scene_inspect", "rtnw_ctx_create_multi", "rtnw_ctx_destroy_multi", "rtnw_multi_device_count",
                  "rtnw_scene_upload_multi", "rtnw_scene_free_multi", "rtnw_render_multi", "rtnw_scene_prepare", "rtnw_prepared_bytes",
                  "rtnw_scene_upload_prepared", "rtnw_prepared_free", "rtnw_render_aov", "rtnw_denoise", "rtnw_render_aov_device",
                  "rtnw_denoise_device", "rtnw_render_aov_multi"]
HOST_SYMBOLS = ["rtnw_host_last_error", "rtnw_host_scene_build", "rtnw_host_scene_free", "rtnw_host_scene_desc",
                "rtnw_host_scene_leaf_count", "rtnw_host_scene_camera", "rtnw_host_scene_view", "rtnw_host_make_camera",
                "rtnw_host_quantize", "rtnw_host_write_ppm", "rtnw_host_load_png", "rtnw_host_free_image", "rtnw_host_write_pfm"]


def build_native(device: bool = True, host: bool = True) -> None:
    """(Re)build the in-tree shared libraries with the package Makefile (nvcc cross-compiles sm_100a without a GPU)."""
    targets = (["host"] if host else []) + (["device"] if device else [])
    subprocess.run(["make", "-C", str(PKG_DIR), "-s"] + targets, check=True)


_host = None
_dev = None


def host_lib() -> C.CDLL:
    global _host
    if _host is None:
        path = LIB_DIR / "librtnw_host.so"
        if not path.exists():
            raise RtnwError(RTNW_ERR_INVALID, f"{path} is missing: run __graft_entry__.build() (make -C {PKG_DIR})")
        L = C.CDLL(str(path))
        L.rtnw_host_last_error.restype = C.c_char_p
        L.rtnw_host_scene_build.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.rtnw_host_scene_free.argtypes = [C.c_void_p]
        L.rtnw_host_scene_free.restype = None
        L.rtnw_host_scene_desc.argtypes = [C.c_void_p]
        L.rtnw_host_scene_desc.restype = C.POINTER(SceneDesc)
        L.rtnw_host_scene_leaf_count.argtypes = [C.c_void_p]
        L.rtnw_host_scene_camera.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(Camera)]
        L.rtnw_host_scene_view.argtypes = [C.c_void_p, C.POINTER(HostView)]
        L.rtnw_host_make_camera.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                            C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(Camera)]
        L.rtnw_host_quantize.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        L.rtnw_host_write_ppm.argtypes = [C.c_char_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
        L.rtnw_host_write_pfm.argtypes = [C.c_char_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
        L.rtnw_host_load_png.argtypes = [C.c_char_p, C.POINTER(C.POINTER(C.c_ubyte)), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.rtnw_host_free_image.argtypes = [C.POINTER(C.c_ubyte)]
        L.rtnw_host_free_image.restype = None
        _host = L
    return _host


def device_lib() -> C.CDLL:
    """Load librtnw.so.  Fails loudly when it is missing: the product path has no CPU fallback."""
    global _dev
    if _dev is None:
        path = Path(os.environ.get("RTNW_LIB", LIB_DIR / "librtnw.so"))  # RTNW_LIB: A/B builds while tuning
        if not path.exists():
            raise RtnwError(RTNW_ERR_CUDA, f"{path} is missing: the CUDA extension must be built "
                                           f"(__graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(str(path))
        L.rtnw_last_error.restype = C.c_char_p
        L.rtnw_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.rtnw_ctx_destroy.argtypes = [C.c_void_p]
        L.rtnw_ctx_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_int32)] * 4
        L.rtnw_measure_fp32_peak.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.rtnw_selftest_recip.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]
        L.rtnw_quantize_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        L.rtnw_plan_sample_ranges.argtypes = [C.POINTER(RenderParams), C.POINTER(C.c_int32), C.c_int32]
        L.rtnw_scene_inspect.argtypes = [C.POINTER(SceneDesc), C.c_int32, C.c_void_p, C.c_size_t]
        L.rtnw_scene_inspect.restype = C.c_int64
        L.rtnw_scene_upload.argtypes = [C.c_void_p, C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
        L.rtnw_scene_free.argtypes = [C.c_void_p, C.c_void_p]
        L.rtnw_render.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_void_p, C.POINTER(Stats)]
        L.rtnw_render_device.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_void_p,
                                         C.c_void_p, C.POINTER(Stats)]
        L.rtnw_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float, C.c_uint32, C.c_uint64,
                                 C.c_void_p]
        L.rtnw_render_aov.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.POINTER(Aov),
                                      C.POINTER(Stats)]
        L.rtnw_denoise.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Aov), C.c_int32, C.c_int32, C.c_int32, C.POINTER(DenoiseParams),
                                   C.c_void_p, C.POINTER(Stats)]
        L.rtnw_render_aov_device.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.POINTER(Aov),
                                             C.c_void_p, C.POINTER(Stats)]
        L.rtnw_denoise_device.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Aov), C.c_int32, C.c_int32, C.c_int32,
                                          C.POINTER(DenoiseParams), C.c_void_p, C.c_void_p, C.POINTER(Stats)]
        L.rtnw_eval_texture.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
        L.rtnw_eval_perlin.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]
        L.rtnw_scatter.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
        L.rtnw_camera_rays.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                       C.c_uint64, C.c_void_p]
        L.rtnw_camera_get_rays.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_void_p]
        L.rtnw_scene_prepare.argtypes = [C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
        L.rtnw_prepared_bytes.argtypes = [C.c_void_p]
        L.rtnw_prepared_bytes.restype = C.c_int64
        L.rtnw_scene_upload_prepared.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.rtnw_prepared_free.argtypes = [C.c_void_p]
        L.rtnw_ctx_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
        L.rtnw_ctx_destroy_multi.argtypes = [C.c_void_p]
        L.rtnw_multi_device_count.argtypes = [C.c_void_p]
        L.rtnw_scene_upload_multi.argtypes = [C.c_void_p, C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
        L.rtnw_scene_free_multi.argtypes = [C.c_void_p, C.c_void_p]
        L.rtnw_render_multi.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_void_p, C.POINTER(Stats)]
        L.rtnw_render_aov_multi.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_void_p,
                                            C.POINTER(Aov), C.POINTER(DenoiseParams), C.c_void_p, C.POINTER(Stats)]
        _dev = L
    return _dev


def _check_dev(rc):
    if rc != RTNW_OK:
        raise RtnwError(rc, device_lib().rtnw_last_error().decode())


def _check_host(rc):
    if rc != RTNW_OK:
        raise RtnwError(rc, host_lib().rtnw_host_last_error().decode())


# ------------------------------------------------------------------------------------------------ host scenes
class HostScene:
    """A chapter scene built by the C++ host library and flattened to the tables of include/rtnw.h."""

    def __init__(self, name: str):
        self.name = name
        self._h = C.c_void_p()
        _check_host(host_lib().rtnw_host_scene_build(name.encode(), C.byref(self._h)))
        self.desc_ptr = host_lib().rtnw_host_scene_desc(self._h)
        self.desc = self.desc_ptr.contents
        v = HostView()
        _check_host(host_lib().rtnw_host_scene_view(self._h, C.byref(v)))
        self.view = v

    @property
    def leaf_count(self) -> int:
        return host_lib().rtnw_host_scene_leaf_count(self._h)

    def camera(self, nx: int, ny: int) -> Camera:
        cam = Camera()
        _check_host(host_lib().rtnw_host_scene_camera(self._h, nx, ny, C.byref(cam)))
        return cam

    def params(self, nx=None, ny=None, ns=None, seed=1, sample_begin=0, sample_stride=1, flags_extra=0, pixel_begin=0,
               pixel_stride=1, pixel_count=0, sample_ranges=0) -> RenderParams:
        v = self.view
        return RenderParams(v.nx if nx is None else nx, v.ny if ny is None else ny, sample_begin, v.ns if ns is None else ns,
                            sample_stride, 50, v.t_min, FLT_MAX, v.background, v.flags | flags_extra, seed, pixel_begin,
                            pixel_stride, pixel_count, sample_ranges)

    def close(self):
        if self._h:
            host_lib().rtnw_host_scene_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def make_camera(lookfrom, lookat, vfov, aspect, aperture, focus_dist, t0, t1, vup=(0, 1, 0)) -> Camera:
    cam = Camera()
    f3 = C.c_float * 3
    _check_host(host_lib().rtnw_host_make_camera(f3(*lookfrom), f3(*lookat), f3(*vup), vfov, aspect, aperture, focus_dist, t0, t1,
                                                 C.byref(cam)))
    return cam


def quantize(sums: np.ndarray, ns: int, clamp255: bool = True) -> np.ndarray:
    """PSC/main.cpp:315-325 on the host: mean, sqrt gamma, int(255.99*c); returns (ny, nx, 3) int32, top row first."""
    ny, nx, _ = sums.shape
    sums = np.ascontiguousarray(sums, dtype=np.float32)
    out = np.empty((ny, nx, 3), dtype=np.int32)
    _check_host(host_lib().rtnw_host_quantize(sums.ctypes.data, nx, ny, ns, int(clamp255), out.ctypes.data))
    return out


def load_png(path) -> np.ndarray:
    """Texture ingest (replaces stbi_load, PSC/main.cpp:93): a PNG file as the (ny, nx, 3) uint8 array image_texture indexes."""
    px = C.POINTER(C.c_ubyte)()
    nx, ny = C.c_int32(), C.c_int32()
    _check_host(host_lib().rtnw_host_load_png(str(path).encode(), C.byref(px), C.byref(nx), C.byref(ny)))
    try:
        return np.ctypeslib.as_array(px, shape=(ny.value, nx.value, 3)).copy()
    finally:
        host_lib().rtnw_host_free_image(px)


def write_ppm(path: str, sums: np.ndarray, ns: int, clamp255: bool = True, binary: bool = False) -> None:
    ny, nx, _ = sums.shape
    sums = np.ascontiguousarray(sums, dtype=np.float32)
    _check_host(host_lib().rtnw_host_write_ppm(str(path).encode(), sums.ctypes.data, nx, ny, ns, int(clamp255), int(binary)))


def write_pfm(path, array: np.ndarray) -> None:
    """Write a float image as a Portable Float Map: (ny, nx, 3) as colour "PF", (ny, nx) as greyscale "Pf"; row 0 of the
    array (the library's bottom row, j = 0) is the first row of the file, as PFM wants."""
    a = np.ascontiguousarray(array, dtype=np.float32)
    channels = a.shape[2] if a.ndim == 3 else 1
    _check_host(host_lib().rtnw_host_write_pfm(str(path).encode(), a.ctypes.data, a.shape[1], a.shape[0], channels))


def device_tables(desc_ptr) -> dict:
    """The tables rtnw_scene_upload derives from a scene_desc, built on the host (no GPU needed): record stream, leaf ids,
    gates, the 4-wide gate tree and the light table of F_LIGHT_SAMPLING (include/rtnw.h: rtnw_scene_inspect)."""
    out = {}
    for table, (name, dtype, width) in enumerate([("recs", np.float32, 8), ("rec_leaf", np.int32, 1), ("gates", np.int32, 2),
                                                    ("wnodes", np.float32, 32), ("lights", np.float32, 8)]):
        n = device_lib().rtnw_scene_inspect(desc_ptr, table, None, 0)
        _check_dev(min(n, 0))
        a = np.empty(n // np.dtype(dtype).itemsize, dtype=dtype)
        device_lib().rtnw_scene_inspect(desc_ptr, table, a.ctypes.data, a.nbytes)
        out[name] = a.reshape(-1, width) if width > 1 else a
    return out


def plan_sample_ranges(params) -> np.ndarray:
    """Cumulative sample-range boundaries rtnw_render uses for `params` (host arithmetic; works without a GPU)."""
    cum = (C.c_int32 * 65)()
    n = device_lib().rtnw_plan_sample_ranges(C.byref(params), cum, 64)
    _check_dev(min(n, 0))
    return np.array(cum[:n + 1], dtype=np.int64)


AOV_KEYS = ("albedo", "normal", "depth", "hits", "prim_id")


def _aov_arrays(params):
    """host arrays for the five AOV buffers of a frame, and the rtnw_aov pointing at them"""
    ny, nx = params.ny, params.nx
    out = dict(albedo=np.empty((ny, nx, 3), np.float32), normal=np.empty((ny, nx, 3), np.float32),
               depth=np.empty((ny, nx), np.float32), hits=np.empty((ny, nx), np.int32), prim_id=np.empty((ny, nx), np.int32))
    return out, Aov(*(out[k].ctypes.data for k in AOV_KEYS))


# ------------------------------------------------------------------------------------------------ device
class Context:
    """One GPU + its stream (rtnw_ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check_dev(device_lib().rtnw_ctx_create(device, C.byref(self._h)))
        self.device = device

    def info(self) -> dict:
        v = [C.c_int32() for _ in range(4)]
        _check_dev(device_lib().rtnw_ctx_info(self._h, *[C.byref(x) for x in v]))
        return dict(sm_count=v[0].value, clock_khz=v[1].value, smem_optin=v[2].value, l2_bytes=v[3].value)

    def fp32_peak_tflops(self) -> float:
        v = C.c_float()
        _check_dev(device_lib().rtnw_measure_fp32_peak(self._h, C.byref(v)))
        return float(v.value)

    def selftest_recip(self, n: int, seed: int = 1) -> dict:
        """rtnw_selftest_recip: n random box / sphere / ray cases through the reciprocal shortcut and through the IEEE form."""
        out = (C.c_uint64 * 6)()
        _check_dev(device_lib().rtnw_selftest_recip(self._h, n, seed, out))
        return dict(zip(("box_mismatch", "sphere_mismatch", "quotient_mismatch", "box_shortcut", "sphere_hits", "box_hits"), map(int, out)))

    def quantize_device(self, dev_ptr: int, nx: int, ny: int, ns: int, clamp255: bool = True) -> np.ndarray:
        """PSC/main.cpp:315-325 on the GPU from a device buffer of sums; returns (ny, nx, 3) int32, top row first."""
        out = np.empty((ny, nx, 3), dtype=np.int32)
        _check_dev(device_lib().rtnw_quantize_device(self._h, C.c_void_p(dev_ptr), nx, ny, ns, int(clamp255), out.ctypes.data))
        return out

    def upload(self, desc) -> "DeviceScene":
        return DeviceScene(self, desc)

    def denoise(self, sums: np.ndarray, aov: dict, ns: int, iterations: int = 5, sigma_luminance: float = 4.0,
                sigma_depth: float = 1.0, normal_power_log2: int = 7, stats: Stats | None = None) -> np.ndarray:
        """Denoise a frame on the GPU from its first-hit feature buffers (include/rtnw.h: rtnw_denoise): `sums` as
        DeviceScene.render returns them and `aov` as DeviceScene.render_aov returns it for the same params, ns = their
        sample_count.  Returns the denoised MEAN colour, (ny, nx, 3) float32, row j = 0 at the bottom.  Pass a Stats to
        receive the call's statistics."""
        ny, nx, _ = sums.shape
        sums = np.ascontiguousarray(sums, dtype=np.float32)
        bufs = {k: np.ascontiguousarray(aov[k], dtype=np.int32 if k == "hits" else np.float32)
                for k in ("albedo", "normal", "depth", "hits")}
        for k, shape in (("albedo", (ny, nx, 3)), ("normal", (ny, nx, 3)), ("depth", (ny, nx)), ("hits", (ny, nx))):
            if bufs[k].shape != shape:
                raise RtnwError(RTNW_ERR_INVALID, f"aov[{k!r}] has shape {bufs[k].shape}, expected {shape}")
        feats = Aov(bufs["albedo"].ctypes.data, bufs["normal"].ctypes.data, bufs["depth"].ctypes.data, bufs["hits"].ctypes.data, None)
        out = np.empty((ny, nx, 3), np.float32)
        dp = DenoiseParams(iterations, sigma_luminance, sigma_depth, normal_power_log2)
        st = Stats() if stats is None else stats
        _check_dev(device_lib().rtnw_denoise(self._h, sums.ctypes.data, C.byref(feats), nx, ny, ns, C.byref(dp), out.ctypes.data,
                                             C.byref(st)))
        return out

    def denoise_device(self, color_ptr: int, aov_ptrs: dict, nx: int, ny: int, ns: int, out_ptr: int, stream: int = 0,
                       iterations: int = 5, sigma_luminance: float = 4.0, sigma_depth: float = 1.0, normal_power_log2: int = 7,
                       stats: Stats | None = None) -> Stats:
        """Context.denoise on device buffers (include/rtnw.h: rtnw_denoise_device), e.g. torch tensors' data_ptr(): the colour
        sums at color_ptr, aov_ptrs["albedo" | "normal" | "depth" | "hits"] (a "prim_id" entry is ignored), the denoised mean
        colour written to out_ptr (nx*ny*3 floats, not overlapping an input).  Ordered on `stream` (0 = the legacy default
        stream); returns the call's Stats."""
        feats = Aov(*(aov_ptrs[k] for k in ("albedo", "normal", "depth", "hits")), None)
        dp = DenoiseParams(iterations, sigma_luminance, sigma_depth, normal_power_log2)
        st = Stats() if stats is None else stats
        _check_dev(device_lib().rtnw_denoise_device(self._h, C.c_void_p(color_ptr), C.byref(feats), nx, ny, ns, C.byref(dp),
                                                    C.c_void_p(out_ptr), C.c_void_p(stream), C.byref(st)))
        return st

    def close(self):
        if self._h:
            device_lib().rtnw_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PreparedScene:
    """The device image of a scene_desc built once on the host (rtnw_scene_prepare); upload it with Context.upload()."""

    def __init__(self, desc):
        self._h = C.c_void_p()
        ptr = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
        _check_dev(device_lib().rtnw_scene_prepare(ptr, C.byref(self._h)))

    @property
    def nbytes(self) -> int:
        return int(device_lib().rtnw_prepared_bytes(self._h))

    def close(self):
        if self._h:
            device_lib().rtnw_prepared_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceScene:
    """Device-resident copy of a scene_desc (rtnw_scene)."""

    def __init__(self, ctx: Context, desc):
        self.ctx = ctx
        self._h = C.c_void_p()
        if isinstance(desc, PreparedScene):
            _check_dev(device_lib().rtnw_scene_upload_prepared(ctx._h, desc._h, C.byref(self._h)))
            return
        ptr = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
        _check_dev(device_lib().rtnw_scene_upload(ctx._h, ptr, C.byref(self._h)))

    def close(self):
        if self._h and self.ctx._h:
            device_lib().rtnw_scene_free(self.ctx._h, self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- the sample loop, PSC/main.cpp:299-313
    def render(self, cam: Camera, params: RenderParams, out: np.ndarray | None = None):
        """Host-buffer entry point: returns (sums[ny,nx,3] with row j=0 at the bottom, Stats)."""
        if out is None:
            out = np.empty((params.ny, params.nx, 3), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == params.nx * params.ny * 3
        st = Stats()
        _check_dev(device_lib().rtnw_render(self.ctx._h, self._h, C.byref(cam), C.byref(params), out.ctypes.data, C.byref(st)))
        return out, st

    def render_device(self, cam: Camera, params: RenderParams, dev_ptr: int, stream: int = 0) -> Stats:
        """Render into caller-owned device memory (e.g. a torch tensor's data_ptr())."""
        st = Stats()
        _check_dev(device_lib().rtnw_render_device(self.ctx._h, self._h, C.byref(cam), C.byref(params), C.c_void_p(dev_ptr),
                                                   C.c_void_p(stream), C.byref(st)))
        return st

    def render_aov(self, cam: Camera, params: RenderParams, stats: Stats | None = None) -> dict:
        """First-hit feature buffers of the frame rtnw_render draws for the same camera and params (include/rtnw.h:
        rtnw_render_aov): dict of per-pixel SUMS albedo (ny,nx,3), normal (ny,nx,3), depth (ny,nx), and int32 hits (ny,nx) and
        prim_id (ny,nx), row j = 0 at the bottom.  Divide albedo by sample_count, normal and depth by hits.  Pass a Stats to
        receive the call's statistics."""
        out, bufs = _aov_arrays(params)
        st = Stats() if stats is None else stats
        _check_dev(device_lib().rtnw_render_aov(self.ctx._h, self._h, C.byref(cam), C.byref(params), C.byref(bufs), C.byref(st)))
        return out

    def render_aov_device(self, cam: Camera, params: RenderParams, bufs: dict, stream: int = 0, stats: Stats | None = None) -> Stats:
        """render_aov into caller-owned device memory (include/rtnw.h: rtnw_render_aov_device): bufs maps "albedo", "normal",
        "depth", "hits" and "prim_id" to device pointers (e.g. torch tensors' data_ptr()) of the shapes render_aov returns.
        Ordered on `stream` (0 = the legacy default stream).  Takes params.flags | F_ROTATE_SAMPLES for one rank's share of
        a multi-GPU frame.  Returns the call's Stats."""
        aov = Aov(*(bufs[k] for k in AOV_KEYS))
        st = Stats() if stats is None else stats
        _check_dev(device_lib().rtnw_render_aov_device(self.ctx._h, self._h, C.byref(cam), C.byref(params), C.byref(aov),
                                                       C.c_void_p(stream), C.byref(st)))
        return st

    # -- one world->hit() per ray, PSC/main.cpp:27
    def trace(self, rays: np.ndarray, t_min: float = 0.001, t_max: float = FLT_MAX, flags: int = 0, seed: int = 1) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = np.zeros(rays.shape[0], dtype=HIT_DTYPE)
        _check_dev(device_lib().rtnw_trace(self.ctx._h, self._h, rays.ctypes.data, rays.shape[0], t_min, t_max, flags, seed,
                                           out.ctypes.data))
        return out

    def eval_texture(self, tex_id: int, uvp: np.ndarray) -> np.ndarray:
        uvp = np.ascontiguousarray(uvp, dtype=np.float32).reshape(-1, 5)
        out = np.zeros((uvp.shape[0], 3), dtype=np.float32)
        _check_dev(device_lib().rtnw_eval_texture(self.ctx._h, self._h, tex_id, uvp.ctypes.data, uvp.shape[0], out.ctypes.data))
        return out

    def eval_perlin(self, which: int, xyz: np.ndarray) -> np.ndarray:
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        out = np.zeros(xyz.shape[0], dtype=np.float32)
        _check_dev(device_lib().rtnw_eval_perlin(self.ctx._h, self._h, which, xyz.ctypes.data, xyz.shape[0], out.ctypes.data))
        return out

    def scatter(self, rays_in: np.ndarray, hits: np.ndarray, seed: int = 1):
        rays_in = np.ascontiguousarray(rays_in, dtype=RAY_DTYPE)
        hits = np.ascontiguousarray(hits, dtype=HIT_DTYPE)
        n = rays_in.shape[0]
        sc = np.zeros(n, dtype=RAY_DTYPE)
        att = np.zeros((n, 3), dtype=np.float32)
        em = np.zeros((n, 3), dtype=np.float32)
        flag = np.zeros(n, dtype=np.int32)
        _check_dev(device_lib().rtnw_scatter(self.ctx._h, self._h, rays_in.ctypes.data, hits.ctypes.data, n, seed, sc.ctypes.data,
                                             att.ctypes.data, em.ctypes.data, flag.ctypes.data))
        return sc, att, em, flag


class MultiContext:
    """N GPUs of one box behind one handle (rtnw_ctx_create_multi): spp split + one sum on device 0, in one process."""

    def __init__(self, devices):
        devices = list(devices)
        self._h = C.c_void_p()
        _check_dev(device_lib().rtnw_ctx_create_multi((C.c_int * len(devices))(*devices), len(devices), C.byref(self._h)))
        self.devices = devices

    def upload(self, desc) -> "MultiScene":
        return MultiScene(self, desc)

    def close(self):
        if self._h:
            device_lib().rtnw_ctx_destroy_multi(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiScene:
    def __init__(self, mctx: MultiContext, desc):
        self.mctx = mctx
        self._h = C.c_void_p()
        ptr = desc if isinstance(desc, C.POINTER(SceneDesc)) else C.pointer(desc)
        _check_dev(device_lib().rtnw_scene_upload_multi(mctx._h, ptr, C.byref(self._h)))

    def render(self, cam: Camera, params: RenderParams, out: np.ndarray | None = None):
        if out is None:
            out = np.empty((params.ny, params.nx, 3), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == params.nx * params.ny * 3
        st = Stats()
        _check_dev(device_lib().rtnw_render_multi(self.mctx._h, self._h, C.byref(cam), C.byref(params), out.ctypes.data, C.byref(st)))
        return out, st

    def render_aov(self, cam: Camera, params: RenderParams, denoise: DenoiseParams | None = None):
        """One frame and its first-hit feature buffers on every device of the handle (include/rtnw.h: rtnw_render_aov_multi),
        denoised on the first device when `denoise` is given.  Returns (sums, aov, denoised or None, Stats) in the shapes of
        DeviceScene.render, DeviceScene.render_aov and Context.denoise."""
        sums = np.empty((params.ny, params.nx, 3), dtype=np.float32)
        aov, bufs = _aov_arrays(params)
        den = None if denoise is None else np.empty((params.ny, params.nx, 3), dtype=np.float32)
        st = Stats()
        _check_dev(device_lib().rtnw_render_aov_multi(self.mctx._h, self._h, C.byref(cam), C.byref(params), sums.ctypes.data,
                                                      C.byref(bufs), None if denoise is None else C.byref(denoise),
                                                      None if den is None else den.ctypes.data, C.byref(st)))
        return sums, aov, den, st

    def close(self):
        if self._h and self.mctx._h:
            device_lib().rtnw_scene_free_multi(self.mctx._h, self._h)
        self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def camera_rays(ctx: Context, cam: Camera, nx: int, ny: int, ij: np.ndarray, sample: np.ndarray, seed: int = 1) -> np.ndarray:
    ij = np.ascontiguousarray(ij, dtype=np.int32).reshape(-1, 2)
    sample = np.ascontiguousarray(sample, dtype=np.int32)
    out = np.zeros(ij.shape[0], dtype=RAY_DTYPE)
    _check_dev(device_lib().rtnw_camera_rays(ctx._h, C.byref(cam), nx, ny, ij.ctypes.data, sample.ctypes.data, ij.shape[0], seed,
                                             out.ctypes.data))
    return out


def camera_get_rays(ctx: Context, cam: Camera, st: np.ndarray, seed: int = 1, key_base: int = 0) -> np.ndarray:
    """camera::get_ray(s, t) for n pairs (PSC/camera.h:41-47); draws from the path stream (seed, key_base + q, 0)"""
    st = np.ascontiguousarray(st, dtype=np.float32).reshape(-1, 2)
    out = np.zeros(st.shape[0], dtype=RAY_DTYPE)
    _check_dev(device_lib().rtnw_camera_get_rays(ctx._h, C.byref(cam), st.ctypes.data, st.shape[0], seed, key_base, out.ctypes.data))
    return out


def device_count() -> int:
    return device_lib().rtnw_device_count()
