"""raytracing-practice_b200 — Python plumbing over the C-ABI of the B200 path tracer.

The product is the CUDA library `librt_b200.so` (csrc/) behind include/rt_b200.h and the C++
host mirror of the reference's scene API (host/).  This module is only the ctypes binding the
tests and bench.py use: it loads the in-tree shared libraries, wraps named scenes
(`Scene`) and a device context (`Context`).  There is NO CPU fallback: if the CUDA
library is missing, or there is no GPU, every entry point raises.

The directory name contains a hyphen, so import it with
    rtb = importlib.import_module("raytracing-practice_b200")
"""
import ctypes as C
import os

import numpy as np

from . import _abi
from ._abi import *  # noqa: F401,F403

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)
CUDA_LIB_PATH = os.environ.get("RT_B200_LIB") or os.path.join(_HERE, "librt_b200.so")  # RT_B200_LIB: A/B variant builds
SCENES_LIB_PATH = os.path.join(_HERE, "librtb200_scenes.so")

_cuda_lib = None
_scenes_lib = None


class RtError(RuntimeError):
    pass


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def cuda_lib():
    """The C-ABI library.  Fails loudly when it has not been built (no fallback)."""
    global _cuda_lib
    if _cuda_lib is None:
        if not os.path.exists(CUDA_LIB_PATH):
            raise RtError(
                f"{CUDA_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)"
            )
        lib = C.CDLL(CUDA_LIB_PATH)
        lib.rt_last_error.restype = C.c_char_p
        lib.rt_last_error.argtypes = [C.c_void_p]
        lib.rt_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.rt_shutdown.argtypes = [C.c_void_p]
        lib.rt_shutdown.restype = None
        lib.rt_upload_scene.argtypes = [C.c_void_p, C.POINTER(_abi.rt_scene_desc)]
        lib.rt_render.argtypes = [C.c_void_p, C.POINTER(_abi.rt_camera_desc), C.POINTER(_abi.rt_render_opts)]
        lib.rt_render_views.argtypes = [C.c_void_p, C.c_int32, C.POINTER(_abi.rt_camera_desc), C.POINTER(_abi.rt_render_opts)]
        lib.rt_synchronize.argtypes = [C.c_void_p]
        lib.rt_accum_device_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        lib.rt_reduce_buffer.argtypes = [C.c_void_p, C.POINTER(_abi.rt_camera_desc), C.POINTER(C.c_void_p), C.POINTER(_abi.rt_ipc_handle)]
        lib.rt_peer_open.argtypes = [C.c_void_p, C.POINTER(_abi.rt_ipc_handle), C.POINTER(C.c_void_p)]
        lib.rt_peer_close.argtypes = [C.c_void_p, C.c_void_p]
        lib.rt_adopt_reduce_buffer.argtypes = [C.c_void_p]
        lib.rt_download.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_void_p, C.c_size_t]
        lib.rt_upload_accum.argtypes = [C.c_void_p, C.POINTER(_abi.rt_camera_desc), C.c_void_p, C.c_size_t]
        lib.rt_get_stats.argtypes = [C.c_void_p, C.POINTER(_abi.rt_stats)]
        lib.rt_camera_initialize.argtypes = [C.POINTER(_abi.rt_camera_desc), C.POINTER(_abi.rt_camera_frame)]
        dp, ip, bp, fp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.POINTER(C.c_float)
        lib.rt_trace_rays.argtypes = [C.c_void_p, C.c_int64, dp, dp, dp, C.c_double, C.c_double, C.c_int32, ip, dp, dp, bp]
        lib.rt_trace_rays_from.argtypes = [C.c_void_p, C.c_int64, dp, dp, dp, ip, C.c_double, C.c_double, C.c_int32, ip, dp, dp, bp]
        lib.rt_primary_visibility.argtypes = [C.c_void_p, C.POINTER(_abi.rt_camera_desc), C.c_int32, ip, dp, dp]
        lib.rt_bounce_visibility.argtypes = [C.c_void_p, C.POINTER(_abi.rt_camera_desc), C.c_uint64, ip, dp, fp, fp, ip, dp, dp, bp]
        lib.rt_medium_spans.argtypes = [C.c_void_p, C.c_int32, C.c_int64, dp, dp, dp, dp, dp]
        lib.rt_eval_texture.argtypes = [C.c_void_p, C.c_int32, C.c_int64, dp, fp]
        lib.rt_eval_scatter.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, dp, dp, bp, fp, fp, bp]
        _cuda_lib = lib
    return _cuda_lib


def scenes_lib():
    global _scenes_lib
    if _scenes_lib is None:
        if not os.path.exists(SCENES_LIB_PATH):
            raise RtError(f"{SCENES_LIB_PATH} is missing: run __graft_entry__.build()")
        lib = C.CDLL(SCENES_LIB_PATH)
        lib.rth_scene_count.restype = C.c_int
        lib.rth_scene_name.restype = C.c_char_p
        lib.rth_scene_name.argtypes = [C.c_int]
        lib.rth_scene_build.restype = C.c_void_p
        lib.rth_scene_build.argtypes = [C.c_char_p, C.c_long]
        lib.rth_scene_free.argtypes = [C.c_void_p]
        lib.rth_scene_free.restype = None
        lib.rth_scene_desc.restype = C.POINTER(_abi.rt_scene_desc)
        lib.rth_scene_desc.argtypes = [C.c_void_p]
        lib.rth_scene_camera.restype = C.POINTER(_abi.rt_camera_desc)
        lib.rth_scene_camera.argtypes = [C.c_void_p]
        lib.rth_load_texture.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.rth_free.argtypes = [C.c_void_p]
        lib.rth_free.restype = None
        _scenes_lib = lib
    return _scenes_lib


def default_image_dir():
    """Where earthmap.jpg lives on this machine (the reference's image asset is not committed)."""
    for d in (os.environ.get("RTW_IMAGES"), os.path.join(REPO_ROOT, "baseline", "_ref", "images"), "/root/reference/images"):
        if d and os.path.exists(os.path.join(d, "earthmap.jpg")):
            return d
    return None


def scene_names():
    lib = scenes_lib()
    return [lib.rth_scene_name(i).decode() for i in range(lib.rth_scene_count())]


class Scene:
    """A named scene built by the C++ host API (host/scenes.hpp) and flattened to rt_scene_desc."""

    def __init__(self, name, rand_seed=1):
        if "RTW_IMAGES" not in os.environ and default_image_dir():
            os.environ["RTW_IMAGES"] = default_image_dir()
        self._lib = scenes_lib()
        self._h = self._lib.rth_scene_build(name.encode(), rand_seed)
        if not self._h:
            raise RtError(f"unknown scene {name!r}; known: {scene_names()}")
        self.name = name
        self.desc = self._lib.rth_scene_desc(self._h)  # POINTER(rt_scene_desc)
        self.cam = self._lib.rth_scene_camera(self._h)  # POINTER(rt_camera_desc), mutable

    def camera_copy(self, **overrides):
        cam = _abi.rt_camera_desc()
        C.memmove(C.byref(cam), self.cam, C.sizeof(cam))
        for k, v in overrides.items():
            setattr(cam, k, v)
        return cam

    def close(self):
        if self._h:
            self._lib.rth_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def camera_frame(cam, lib=None):
    """camera::initialize in double (host arithmetic inside the C-ABI library)."""
    f = _abi.rt_camera_frame()
    (lib or cuda_lib()).rt_camera_initialize(C.byref(cam), C.byref(f))
    return f


def image_height(cam):
    h = int(cam.image_width / cam.aspect_ratio)
    return max(h, 1)


class Context:
    """One rt_ctx = one CUDA device = one rank."""

    def __init__(self, device=0):
        self._lib = cuda_lib()
        self._h = C.c_void_p()
        rc = self._lib.rt_init(device, C.byref(self._h))
        if rc != RT_OK:
            raise RtError(f"rt_init({device}) failed ({rc}): {self._lib.rt_last_error(None).decode()}")
        self.device = device
        self._views = False  # the accumulator holds a batch of rt_render_views: downloads are (V, H, W, 3)

    def _check(self, rc, what):
        if rc != RT_OK:
            raise RtError(f"{what} failed ({rc}): {self._lib.rt_last_error(self._h).decode()}")

    def upload_scene(self, desc):
        self._check(self._lib.rt_upload_scene(self._h, desc), "rt_upload_scene")

    def render(self, cam, seed=0, sample_begin=0, sample_count=0, clear=True, peer_accum=None, flags=0, push_accum=None):
        o = _abi.rt_render_opts(seed, sample_begin, sample_count, 1 if clear else 0, flags, peer_accum, push_accum)
        self._views = False
        self._check(self._lib.rt_render(self._h, C.byref(cam), C.byref(o)), "rt_render")

    def render_views(self, cams, seed=0, sample_begin=0, sample_count=0, clear=True, flags=0):
        """Render several views of the uploaded scene in one launch (rt_render_views).  `cams`: a sequence of
        rt_camera_desc of one image size and spp.  View v gets the bits render(cams[v], seed, ...) gives; the downloads
        then return (V, H, W, 3)."""
        cams = list(cams)
        arr = (_abi.rt_camera_desc * max(len(cams), 1))(*cams)
        o = _abi.rt_render_opts(seed, sample_begin, sample_count, 1 if clear else 0, flags, None, None)
        self._check(self._lib.rt_render_views(self._h, len(cams), arr if cams else None, C.byref(o)), "rt_render_views")
        self._views = True

    def reduce_buffer(self, cam):
        """Allocate / zero this context's reduce buffer for `cam`; returns (device pointer, 64-byte IPC handle)."""
        p, h = C.c_void_p(), _abi.rt_ipc_handle()
        self._check(self._lib.rt_reduce_buffer(self._h, C.byref(cam), C.byref(p), C.byref(h)), "rt_reduce_buffer")
        return p.value, bytes(h.bytes)

    def peer_open(self, handle_bytes):
        h = _abi.rt_ipc_handle()
        C.memmove(h.bytes, handle_bytes, 64)
        p = C.c_void_p()
        self._check(self._lib.rt_peer_open(self._h, C.byref(h), C.byref(p)), "rt_peer_open")
        return p.value

    def peer_close(self, ptr):
        self._check(self._lib.rt_peer_close(self._h, ptr), "rt_peer_close")

    def adopt_reduce_buffer(self):
        self._check(self._lib.rt_adopt_reduce_buffer(self._h), "rt_adopt_reduce_buffer")

    def synchronize(self):
        self._check(self._lib.rt_synchronize(self._h), "rt_synchronize")

    def accum_ptr(self):
        p, n = C.c_void_p(), C.c_size_t()
        self._check(self._lib.rt_accum_device_ptr(self._h, C.byref(p), C.byref(n)), "rt_accum_device_ptr")
        return p.value, n.value

    def accum_tensor(self):
        """The int64 accumulator as a torch tensor aliasing device memory (for NCCL)."""
        import torch

        ptr, nbytes = self.accum_ptr()

        class _Alias:
            __cuda_array_interface__ = {"shape": (nbytes // 8,), "typestr": "<i8", "data": (ptr, False), "version": 3}

        return torch.as_tensor(_Alias(), device=f"cuda:{self.device}")

    def stats(self):
        s = _abi.rt_stats()
        self._check(self._lib.rt_get_stats(self._h, C.byref(s)), "rt_get_stats")
        return s

    def _download(self, kind, spp, arr):
        self._check(self._lib.rt_download(self._h, kind, spp, arr.ctypes.data_as(C.c_void_p), arr.nbytes), "rt_download")
        return arr

    def _image_shape(self):
        """(H, W, 3) after render / upload_accum; (V, H, W, 3) after render_views, also for V = 1."""
        s = self.stats()
        shape = (s.image_height, s.image_width, 3)
        return (s.n_views,) + shape if self._views or s.n_views > 1 else shape

    def download_accum(self):
        return self._download(RT_BUF_ACCUM_I64, 1, np.empty(self._image_shape(), np.int64))

    def upload_accum(self, cam, sums):
        """Replace the accumulator with saved int64 sums (H x W x 3): the inverse of download_accum."""
        a = np.ascontiguousarray(sums, dtype=np.int64)
        self._views = False
        self._check(self._lib.rt_upload_accum(self._h, C.byref(cam), a.ctypes.data_as(C.c_void_p), a.nbytes), "rt_upload_accum")

    def download_radiance(self, spp):
        return self._download(RT_BUF_RADIANCE_F32, spp, np.empty(self._image_shape(), np.float32))

    def download_rgb8(self, spp):
        return self._download(RT_BUF_RGB8, spp, np.empty(self._image_shape(), np.uint8))

    def trace_rays(self, origin, direction, time=None, tmin=0.001, tmax=float("inf"), flags=RT_TRACE_FP32, start_prim=None):
        """start_prim: per ray the primitive id it starts on (-1: none), for rays that leave a surface as rt_render's
        bounce rays do (rt_trace_rays_from; fp32 mode only)."""
        origin = np.ascontiguousarray(origin, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = origin.shape[0]
        time = np.zeros(n) if time is None else np.ascontiguousarray(time, np.float64)
        ids = np.empty(n, np.int32)
        t = np.empty(n, np.float64)
        nrm = np.empty((n, 3), np.float64)
        ff = np.empty(n, np.uint8)
        ip = C.POINTER(C.c_int32)
        sp = None
        if start_prim is not None:
            start_prim = np.ascontiguousarray(start_prim, np.int32)
            if start_prim.shape != (n,):
                raise ValueError(f"start_prim must hold one id per ray: shape {start_prim.shape}, {n} rays")
            sp = start_prim.ctypes.data_as(ip)
        rc = self._lib.rt_trace_rays_from(
            self._h, n, _dptr(origin), _dptr(direction), _dptr(time), sp, tmin, tmax, flags,
            ids.ctypes.data_as(ip), _dptr(t), _dptr(nrm), ff.ctypes.data_as(C.POINTER(C.c_uint8)))
        self._check(rc, "rt_trace_rays_from")
        return ids, t, nrm, ff

    def primary_visibility(self, cam, flags=RT_TRACE_EXACT | RT_TRACE_SKIP_MEDIA):
        w, h = cam.image_width, image_height(cam)
        ids = np.empty((h, w), np.int32)
        t = np.empty((h, w), np.float64)
        nrm = np.empty((h, w, 3), np.float64)
        rc = self._lib.rt_primary_visibility(self._h, C.byref(cam), flags, ids.ctypes.data_as(C.POINTER(C.c_int32)), _dptr(t), _dptr(nrm))
        self._check(rc, "rt_primary_visibility")
        return ids, t, nrm

    def bounce_visibility(self, cam, seed=0):
        """The render kernel's first two segments of every pixel-centre path (rt_bounce_visibility), as a dict of H x W
        arrays: id, t (primary hit); o1, d1 (fp32 bounce ray); id1, t1, n1, front1 (its hit; id1 = RT_NO_BOUNCE without one)."""
        w, h = cam.image_width, image_height(cam)
        out = dict(id=np.empty((h, w), np.int32), t=np.empty((h, w)), o1=np.empty((h, w, 3), np.float32), d1=np.empty((h, w, 3), np.float32),
                   id1=np.empty((h, w), np.int32), t1=np.empty((h, w)), n1=np.empty((h, w, 3)), front1=np.empty((h, w), np.uint8))
        ip, fp = C.POINTER(C.c_int32), C.POINTER(C.c_float)
        rc = self._lib.rt_bounce_visibility(self._h, C.byref(cam), seed, out["id"].ctypes.data_as(ip), _dptr(out["t"]), out["o1"].ctypes.data_as(fp),
                                            out["d1"].ctypes.data_as(fp), out["id1"].ctypes.data_as(ip), _dptr(out["t1"]), _dptr(out["n1"]),
                                            out["front1"].ctypes.data_as(C.POINTER(C.c_uint8)))
        self._check(rc, "rt_bounce_visibility")
        return out

    def medium_spans(self, medium_index, origin, direction, time=None):
        origin = np.ascontiguousarray(origin, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = origin.shape[0]
        time = np.zeros(n) if time is None else np.ascontiguousarray(time, np.float64)
        t1, t2 = np.empty(n), np.empty(n)
        self._check(self._lib.rt_medium_spans(self._h, medium_index, n, _dptr(origin), _dptr(direction), _dptr(time), _dptr(t1), _dptr(t2)), "rt_medium_spans")
        return t1, t2

    def eval_texture(self, texture, uvp):
        uvp = np.ascontiguousarray(uvp, np.float64)
        out = np.empty((uvp.shape[0], 3), np.float32)
        self._check(self._lib.rt_eval_texture(self._h, texture, uvp.shape[0], _dptr(uvp), out.ctypes.data_as(C.POINTER(C.c_float))), "rt_eval_texture")
        return out

    def eval_scatter(self, material, dir_in, normal, front_face, seed=0):
        dir_in = np.ascontiguousarray(dir_in, np.float64)
        normal = np.ascontiguousarray(normal, np.float64)
        front_face = np.ascontiguousarray(front_face, np.uint8)
        n = dir_in.shape[0]
        d = np.empty((n, 3), np.float32)
        a = np.empty((n, 3), np.float32)
        s = np.empty(n, np.uint8)
        fp, bp = C.POINTER(C.c_float), C.POINTER(C.c_uint8)
        rc = self._lib.rt_eval_scatter(self._h, material, n, seed, _dptr(dir_in), _dptr(normal), front_face.ctypes.data_as(bp),
                                       d.ctypes.data_as(fp), a.ctypes.data_as(fp), s.ctypes.data_as(bp))
        self._check(rc, "rt_eval_scatter")
        return d, a, s

    def close(self):
        if self._h:
            self._lib.rt_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def write_ppm_p3(path, rgb8):
    """The reference's P3 text format (camera.hpp:36-37, color.hpp:57)."""
    h, w, _ = rgb8.shape
    with open(path, "w") as f:
        f.write(f"P3\n{w} {h}\n255\n")
        f.write("".join(f"{r} {g} {b}\n" for r, g, b in rgb8.reshape(-1, 3).tolist()))
