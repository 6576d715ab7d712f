"""toymeshpathtracer_b200 -- B200-native Trace() hot path of pr0g/ToyMeshPathTracer.

The product is the C-ABI library ``libtmpt.so`` (include/tmpt.h; CUDA kernels for sm_100a in
csrc/kernels.cu, C++ host glue in csrc/host.cpp) and the drop-in command line
``bin/TrimeshTracer``.  This module is the thin ctypes binding the tests and ``bench.py``
drive it through; it mirrors the reference's own interface names:

    Scene(tris)                      Scene::Scene + BuildOctree      (scene.h:19, 26)
    Scene.HitScene(rays, tMin, tMax) Scene::HitScene, batched        (scene.h:36-37)
    Scene.render(camera, w, h, spp)  TraceImageBody over all rows    (main.cpp:180-246, 329-331)
    Scene.render_outputs(...)        the same frame plus linear radiance and first-hit AOVs (beyond the reference)
    Scene.denoise(...)               an a-trous filter over the radiance, guided by the AOVs (beyond the reference)
    load_scene(path)                 LoadScene                       (main.cpp:122-170)
    camera_for_scene(...)            camera placement of main()      (main.cpp:296-307)

There is no CPU fallback: importing works anywhere (so symbols can be checked), but every
compute call raises ``TmptError`` unless a CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtmpt.so")
CLI_PATH = os.path.join(HERE, "bin", "TrimeshTracer")

TMPT_OK, TMPT_ERR_ARG, TMPT_ERR_CUDA, TMPT_ERR_IO, TMPT_ERR_OOM = 0, -1, -2, -3, -4
HOST, DEVICE = 0, 1
HIT_CLOSEST, HIT_ANY, HIT_BRUTE, HIT_SUN = 0, 1, 2, 3
BUILD_DEFAULT, BUILD_LBVH = 0, 1
K_MIN_T, K_MAX_T = 0.001, 1.0e7  # main.cpp:30-31

# every symbol include/tmpt.h declares (tests check the library exports exactly these)
ABI_SYMBOLS = [
    "tmpt_scene_create", "tmpt_scene_destroy", "tmpt_scene_get_info", "tmpt_hit_scene", "tmpt_render",
    "tmpt_render_stripes", "tmpt_stripe_rows", "tmpt_local_width", "tmpt_unpack_stripes", "tmpt_load_obj", "tmpt_free",
    "tmpt_camera_make", "tmpt_camera_for_scene", "tmpt_write_png", "tmpt_main", "tmpt_last_error",
    "tmpt_device_count", "tmpt_launch_count", "tmpt_render_stats", "tmpt_hit_scene_stats",
    "tmpt_frame_alloc", "tmpt_frame_open", "tmpt_frame_close", "tmpt_frame_free", "tmpt_render_multi",
    "tmpt_scene_refit", "tmpt_progressive_begin", "tmpt_progressive_pass", "tmpt_render_kernel_choice",
    "tmpt_render_outputs", "tmpt_progressive_pass_outputs", "tmpt_progressive_pass_adaptive", "tmpt_denoise",
]


class TmptError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"tmpt status {status}: {message}")
        self.status = status


OUTPUTS = ("rgba", "radiance", "normal", "depth", "triangle")  # the members of tmpt_outputs, in order


class Outputs(C.Structure):
    """tmpt_outputs: one pointer per buffer, NULL = not produced."""
    _fields_ = [(name, C.c_void_p) for name in OUTPUTS]


def _output_arrays(names, width: int, height: int) -> dict:
    """Host arrays for the named outputs: rgba [h,w,4] uint8, radiance / normal [h,w,4] float32, depth [h,w] float32,
    triangle [h,w] int32."""
    unknown = set(names) - set(OUTPUTS)
    if unknown:
        raise ValueError(f"unknown outputs {sorted(unknown)}; choose from {OUTPUTS}")
    shapes = {"rgba": ((height, width, 4), np.uint8), "radiance": ((height, width, 4), np.float32),
              "normal": ((height, width, 4), np.float32), "depth": ((height, width), np.float32), "triangle": ((height, width), np.int32)}
    return {n: np.zeros(*shapes[n]) for n in OUTPUTS if n in names}


class Adaptive(C.Structure):
    """tmpt_adaptive: the stop rule of an adaptive progressive pass."""
    _fields_ = [("tolerance", C.c_float), ("minChunks", C.c_int32)]


class DenoiseParams(C.Structure):
    """tmpt_denoise_params: the a-trous filter's iterations and edge-stopping parameters."""
    _fields_ = [("iterations", C.c_int32), ("sigmaLuminance", C.c_float), ("sigmaDepth", C.c_float), ("normalPowerLog2", C.c_int32)]


class SceneInfo(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("tri_count", C.c_int32), ("node_count", C.c_int32),
                ("leaf_count", C.c_int32), ("max_leaf_tris", C.c_int32), ("max_depth", C.c_int32), ("builder", C.c_int32),
                ("bounds_min", C.c_float * 3), ("bounds_max", C.c_float * 3), ("sah_cost", C.c_float), ("build_ms", C.c_float),
                ("device_bytes", C.c_uint64)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["bounds_min"] = list(self.bounds_min)
        d["bounds_max"] = list(self.bounds_max)
        return d


_lib = None


def lib() -> C.CDLL:
    """Load libtmpt.so (building it in-tree first if the sources are newer and nvcc is here)."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    path = os.environ.get("TMPT_LIB") or LIB_PATH  # TMPT_LIB: another build of the same ABI (build.build_variant), for A/B runs
    if path == LIB_PATH:
        try:
            _build.build()
        except Exception:
            if not os.path.exists(LIB_PATH):
                raise
    L = C.CDLL(path)
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    L.tmpt_scene_create.argtypes = [vp, i32, i32, C.c_uint, C.POINTER(vp)]
    L.tmpt_scene_destroy.argtypes = [vp]
    L.tmpt_scene_destroy.restype = None
    L.tmpt_scene_get_info.argtypes = [vp, C.POINTER(SceneInfo)]
    L.tmpt_scene_refit.argtypes = [vp, vp, i32, C.POINTER(C.c_double)]
    L.tmpt_hit_scene.argtypes = [vp, vp, i64, f32, f32, i32, i32, vp, vp, vp, vp, vp]
    L.tmpt_render.argtypes = [vp, vp, i32, i32, i32, i32, vp, C.POINTER(C.c_uint64), C.POINTER(C.c_double), vp]
    L.tmpt_render_outputs.argtypes = [vp, vp, i32, i32, i32, i32, C.POINTER(Outputs), C.POINTER(C.c_uint64), C.POINTER(C.c_double), vp]
    L.tmpt_progressive_pass_outputs.argtypes = [vp, vp, i32, i32, C.POINTER(Outputs), C.POINTER(C.c_uint64), C.POINTER(C.c_double),
                                                C.POINTER(i32), vp]
    L.tmpt_progressive_pass_adaptive.argtypes = [vp, vp, i32, C.POINTER(Adaptive), i32, C.POINTER(Outputs), vp, C.POINTER(C.c_uint64),
                                                 C.POINTER(C.c_double), C.POINTER(i64), vp]
    L.tmpt_denoise.argtypes = [vp, i32, i32, i32, C.POINTER(Outputs), C.POINTER(DenoiseParams), C.POINTER(Outputs), C.POINTER(C.c_double), vp]
    L.tmpt_progressive_begin.argtypes = [vp, i32, i32]
    L.tmpt_progressive_pass.argtypes = [vp, vp, i32, i32, vp, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(i32), vp]
    L.tmpt_render_stripes.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp]
    L.tmpt_stripe_rows.argtypes = [i32, i32, i32, i32]
    L.tmpt_local_width.argtypes = [i32, i32, i32]
    L.tmpt_unpack_stripes.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp]
    L.tmpt_render_stats.argtypes = [vp, vp, i32, i32, i32, vp]
    L.tmpt_hit_scene_stats.argtypes = [vp, vp, i64, f32, f32, i32, vp]
    L.tmpt_render_multi.argtypes = [vp, i32, vp, i32, i32, i32, vp, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]
    L.tmpt_frame_alloc.argtypes = [i32, C.c_size_t, C.POINTER(vp), vp]
    L.tmpt_frame_open.argtypes = [i32, vp, C.POINTER(vp)]
    L.tmpt_frame_close.argtypes = [i32, vp]
    L.tmpt_frame_free.argtypes = [i32, vp]
    L.tmpt_load_obj.argtypes = [C.c_char_p, C.POINTER(C.POINTER(C.c_float)), C.POINTER(i32), vp, vp]
    L.tmpt_free.argtypes = [vp]
    L.tmpt_free.restype = None
    L.tmpt_camera_make.argtypes = [vp, vp, vp, f32, f32, f32, f32, vp]
    L.tmpt_camera_make.restype = None
    L.tmpt_camera_for_scene.argtypes = [C.c_char_p, vp, vp, i32, i32, vp]
    L.tmpt_camera_for_scene.restype = None
    L.tmpt_write_png.argtypes = [C.c_char_p, i32, i32, vp, i32]
    L.tmpt_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.tmpt_render_kernel_choice.argtypes = [vp, vp, vp]
    L.tmpt_last_error.restype = C.c_char_p
    L.tmpt_launch_count.restype = C.c_uint64
    _lib = L
    return L


def _check(rc):
    if rc != TMPT_OK:
        raise TmptError(rc, lib().tmpt_last_error().decode(errors="replace"))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


STATS_COUNT = 16  # TMPT_STATS_COUNT


def _stats_dict(st) -> dict:
    """Counters of an instrumented pass (include/tmpt.h) -> per-ray figures and how the warps spent their iterations."""
    v = [int(x) for x in st]
    rays, witers = max(v[0], 1), max(v[9], 1)
    return {"rays": v[0], "node_visits_per_ray": v[1] / rays, "box_tests_per_ray": 4.0 * v[1] / rays, "tri_tests_per_ray": v[2] / rays,
            "lane_iters_per_ray": v[4] / rays, "culled_pops_per_ray": v[5] / rays, "leaf_waits_per_ray": v[6] / rays,
            "warp_iters_per_ray": v[9] / rays,
            "lanes_with_a_ray": v[4] / witers,                       # of 32, averaged over warp iterations
            "lanes_per_node_step": v[1] / max(v[7], 1), "lanes_per_tri_test": v[2] / max(v[8], 1),
            "warp_iters_with_node_step": v[7] / witers, "warp_iters_with_tri_test": v[8] / witers,
            "stack_overflow_rays": v[10] / rays, "stack_deeper_than": {str(k): v[11 + i] / rays for i, k in enumerate((4, 8, 12, 16, 24))}}


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def device_count() -> int:
    return lib().tmpt_device_count()


def launch_count() -> int:
    return int(lib().tmpt_launch_count())


def load_scene(path: str):
    """LoadScene (main.cpp:122-170): (tris[n,9] incl. the two floor triangles, boundsMin, boundsMax)."""
    L = lib()
    out = C.POINTER(C.c_float)()
    n = C.c_int(0)
    mn, mx = np.zeros(3, np.float32), np.zeros(3, np.float32)
    _check(L.tmpt_load_obj(os.fsencode(path), C.byref(out), C.byref(n), _ptr(mn), _ptr(mx)))
    try:
        tris = np.ctypeslib.as_array(out, shape=(n.value, 9)).copy()
    finally:
        L.tmpt_free(out)
    return tris, mn, mx


def camera_make(look_from, look_at, vup, vfov, aspect, aperture, focus_dist) -> np.ndarray:
    """Camera::Camera (maths.cpp:40-59) -> the 22 floats of maths.h:106-111."""
    cam = np.zeros(22, np.float32)
    lib().tmpt_camera_make(_ptr(_f32(look_from)), _ptr(_f32(look_at)), _ptr(_f32(vup)), vfov, aspect, aperture, focus_dist, _ptr(cam))
    return cam


def camera_for_scene(obj_path: str, bounds_min, bounds_max, width: int, height: int) -> np.ndarray:
    cam = np.zeros(22, np.float32)
    lib().tmpt_camera_for_scene(os.fsencode(obj_path), _ptr(_f32(bounds_min)), _ptr(_f32(bounds_max)), width, height, _ptr(cam))
    return cam


def write_png(path: str, rgba: np.ndarray, flip_vertically: bool = True) -> None:
    rgba = np.ascontiguousarray(rgba, np.uint8)
    h, w = rgba.shape[:2]
    _check(lib().tmpt_write_png(os.fsencode(path), w, h, _ptr(rgba), int(flip_vertically)))


def stripe_rows(height: int, stripe: int, rank: int, world: int) -> int:
    return lib().tmpt_stripe_rows(height, stripe, rank, world)


def local_width(width: int, stripe: int, world: int) -> int:
    return lib().tmpt_local_width(width, stripe, world)


def main(argv) -> int:
    """tmpt_main: the reference command line inside this process."""
    args = [b"TrimeshTracer"] + [os.fsencode(a) for a in argv]
    arr = (C.c_char_p * len(args))(*args)
    return lib().tmpt_main(len(args), arr)


def render_multi(scenes, camera, width: int, height: int, spp: int):
    """One frame on several GPUs from this process: scenes[i] is the replica on device i (tmpt_render_multi)."""
    cam = _f32(camera).reshape(22)
    rgba = np.zeros((height, width, 4), np.uint8)
    rays, sec = C.c_uint64(0), C.c_double(0.0)
    handles = (C.c_void_p * len(scenes))(*[s.handle for s in scenes])
    _check(lib().tmpt_render_multi(handles, len(scenes), _ptr(cam), width, height, spp, _ptr(rgba), C.byref(rays), C.byref(sec)))
    return rgba, rays.value, sec.value


class Scene:
    """``Scene`` (scene.h:17-43) on one GPU: triangle replica + BVH resident in HBM."""

    def __init__(self, tris, device: int = 0, flags: int = BUILD_DEFAULT):
        tris = _f32(tris).reshape(-1, 9)
        self._h = C.c_void_p()
        self.device = device
        _check(lib().tmpt_scene_create(_ptr(tris), tris.shape[0], device, flags, C.byref(self._h)))

    def refit(self, tris) -> float:
        """Same triangles, moved (tmpt_scene_refit): the BVH keeps its topology, boxes / slots / payload follow -> seconds."""
        tris = _f32(tris).reshape(-1, 9)
        sec = C.c_double(0.0)
        _check(lib().tmpt_scene_refit(self._h, _ptr(tris), tris.shape[0], C.byref(sec)))
        return sec.value

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals may be gone at interpreter exit)
            _lib.tmpt_scene_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        return self._h

    def info(self) -> dict:
        si = SceneInfo()
        _check(lib().tmpt_scene_get_info(self._h, C.byref(si)))
        return si.as_dict()

    def HitScene(self, rays, tMin: float = K_MIN_T, tMax: float = K_MAX_T, mode: int = HIT_CLOSEST, payload: bool = True):
        """Batched Scene::HitScene on host arrays -> (id, t, pos, normal); misses keep id = -1 and zeros."""
        rays = _f32(rays).reshape(-1, 6)
        n = rays.shape[0]
        ids = np.full(n, -1, np.int32)
        want = payload and mode not in (HIT_ANY, HIT_SUN)
        t = np.zeros(n, np.float32) if want else None
        pos = np.zeros((n, 3), np.float32) if want else None
        nrm = np.zeros((n, 3), np.float32) if want else None
        _check(lib().tmpt_hit_scene(self._h, _ptr(rays), n, tMin, tMax, mode, HOST, _ptr(ids), _ptr(t), _ptr(pos), _ptr(nrm), None))
        return ids, t, pos, nrm

    def hit_scene_device(self, rays_ptr: int, n: int, ids_ptr: int, t_ptr: int = 0, pos_ptr: int = 0, nrm_ptr: int = 0,
                         tMin: float = K_MIN_T, tMax: float = K_MAX_T, mode: int = HIT_CLOSEST, stream: int = 0):
        """Device-pointer form (asynchronous on `stream`); pointers are raw addresses, e.g. torch ``data_ptr()``."""
        _check(lib().tmpt_hit_scene(self._h, rays_ptr, n, tMin, tMax, mode, DEVICE, ids_ptr, t_ptr or None, pos_ptr or None,
                                    nrm_ptr or None, stream or None))

    def render(self, camera, width: int, height: int, spp: int):
        """One frame into host memory -> (rgba[h,w,4] with row 0 = bottom, rayCount, seconds)."""
        cam = _f32(camera).reshape(22)
        rgba = np.zeros((height, width, 4), np.uint8)
        rays, sec = C.c_uint64(0), C.c_double(0.0)
        _check(lib().tmpt_render(self._h, _ptr(cam), width, height, spp, HOST, _ptr(rgba), C.byref(rays), C.byref(sec), None))
        return rgba, rays.value, sec.value

    def render_outputs(self, camera, width: int, height: int, spp: int, outputs=OUTPUTS):
        """One frame with the named outputs (tmpt_render_outputs) -> ({name: host array}, rayCount, seconds).  rgba is
        render()'s frame; radiance the linear mean before sqrt / quantise; normal / depth / triangle the camera rays' first
        hits (include/tmpt.h)."""
        cam = _f32(camera).reshape(22)
        arrays = _output_arrays(outputs, width, height)
        out = Outputs(**{n: a.ctypes.data for n, a in arrays.items()})
        rays, sec = C.c_uint64(0), C.c_double(0.0)
        _check(lib().tmpt_render_outputs(self._h, _ptr(cam), width, height, spp, HOST, C.byref(out), C.byref(rays), C.byref(sec), None))
        return arrays, rays.value, sec.value

    def render_outputs_device(self, camera, width: int, height: int, spp: int, rgba_ptr: int = 0, radiance_ptr: int = 0,
                              normal_ptr: int = 0, depth_ptr: int = 0, triangle_ptr: int = 0, stream: int = 0):
        """tmpt_render_outputs into device buffers (raw addresses, e.g. torch ``data_ptr()``; 0 = not produced) -> (rayCount, seconds)."""
        cam = _f32(camera).reshape(22)
        out = Outputs(rgba_ptr or None, radiance_ptr or None, normal_ptr or None, depth_ptr or None, triangle_ptr or None)
        rays, sec = C.c_uint64(0), C.c_double(0.0)
        _check(lib().tmpt_render_outputs(self._h, _ptr(cam), width, height, spp, DEVICE, C.byref(out), C.byref(rays), C.byref(sec),
                                         stream or None))
        return rays.value, sec.value

    def progressive_begin(self, width: int, height: int):
        """Start (or restart) a progressive render of a width x height frame (tmpt_progressive_begin)."""
        _check(lib().tmpt_progressive_begin(self._h, width, height))
        self._prog = (width, height)

    def progressive_pass(self, camera, n_chunks: int = 1):
        """n_chunks more 8-sample chunks per pixel -> (rgba mean so far, rays of this pass, seconds, samples so far)."""
        width, height = self._prog
        cam = _f32(camera).reshape(22)
        rgba = np.zeros((height, width, 4), np.uint8)
        rays, sec, spp = C.c_uint64(0), C.c_double(0.0), C.c_int32(0)
        _check(lib().tmpt_progressive_pass(self._h, _ptr(cam), n_chunks, HOST, _ptr(rgba), C.byref(rays), C.byref(sec), C.byref(spp), None))
        return rgba, rays.value, sec.value, spp.value

    def progressive_pass_outputs(self, camera, n_chunks: int = 1, radiance: bool = True):
        """A progressive pass that also returns the linear mean so far -> ({"rgba", "radiance"}, rays of this pass, seconds,
        samples so far)."""
        width, height = self._prog
        cam = _f32(camera).reshape(22)
        arrays = _output_arrays(("rgba", "radiance") if radiance else ("rgba",), width, height)
        out = Outputs(**{n: a.ctypes.data for n, a in arrays.items()})
        rays, sec, spp = C.c_uint64(0), C.c_double(0.0), C.c_int32(0)
        _check(lib().tmpt_progressive_pass_outputs(self._h, _ptr(cam), n_chunks, HOST, C.byref(out), C.byref(rays), C.byref(sec),
                                                   C.byref(spp), None))
        return arrays, rays.value, sec.value, spp.value

    def progressive_pass_adaptive(self, camera, n_chunks: int = 1, tolerance: float = 0.5, min_chunks: int = 4, radiance: bool = True):
        """An adaptive progressive pass (tmpt_progressive_pass_adaptive): only pixels whose estimated error is above `tolerance`
        8-bit codes trace n_chunks more chunks -> ({"rgba", ["radiance"], "samples"}, rays of this pass, seconds, pixels still
        active after the pass)."""
        width, height = self._prog
        cam = _f32(camera).reshape(22)
        arrays = _output_arrays(("rgba", "radiance") if radiance else ("rgba",), width, height)
        out = Outputs(**{n: a.ctypes.data for n, a in arrays.items()})
        arrays["samples"] = np.zeros((height, width), np.int32)
        params = Adaptive(tolerance, min_chunks)
        rays, sec, active = C.c_uint64(0), C.c_double(0.0), C.c_int64(0)
        _check(lib().tmpt_progressive_pass_adaptive(self._h, _ptr(cam), n_chunks, C.byref(params), HOST, C.byref(out),
                                                    _ptr(arrays["samples"]), C.byref(rays), C.byref(sec), C.byref(active), None))
        return arrays, rays.value, sec.value, active.value

    def denoise(self, radiance, normal, depth, iterations: int = 5, sigma_luminance: float = 4.0, sigma_depth: float = 1.0,
                normal_power_log2: int = 7, outputs=("rgba", "radiance")):
        """tmpt_denoise on host arrays: radiance / normal [h,w,4] float32 and depth [h,w] float32 as render_outputs returns them (the
        guides may come from a frame at another spp) -> ({"rgba", "radiance"} as named in `outputs`, seconds)."""
        radiance, normal, depth = _f32(radiance), _f32(normal), _f32(depth)
        height, width = depth.shape
        if radiance.shape != (height, width, 4) or normal.shape != (height, width, 4):
            raise ValueError(f"radiance {radiance.shape} and normal {normal.shape} must be {(height, width, 4)} for depth {depth.shape}")
        if set(outputs) - {"rgba", "radiance"}:
            raise ValueError(f"denoise outputs are rgba and radiance, not {sorted(set(outputs) - {'rgba', 'radiance'})}")
        arrays = _output_arrays(outputs, width, height)
        inp = Outputs(radiance=radiance.ctypes.data, normal=normal.ctypes.data, depth=depth.ctypes.data)
        out = Outputs(**{n: a.ctypes.data for n, a in arrays.items()})
        params = DenoiseParams(iterations, sigma_luminance, sigma_depth, normal_power_log2)
        sec = C.c_double(0.0)
        _check(lib().tmpt_denoise(self._h, width, height, HOST, C.byref(inp), C.byref(params), C.byref(out), C.byref(sec), None))
        return arrays, sec.value

    def denoise_device(self, width: int, height: int, radiance_ptr: int, normal_ptr: int, depth_ptr: int, rgba_out_ptr: int = 0,
                       radiance_out_ptr: int = 0, iterations: int = 5, sigma_luminance: float = 4.0, sigma_depth: float = 1.0,
                       normal_power_log2: int = 7, stream: int = 0) -> float:
        """tmpt_denoise on device buffers (raw addresses, e.g. torch ``data_ptr()``; an output 0 = not produced; radiance_out_ptr may
        be radiance_ptr) -> seconds."""
        inp = Outputs(radiance=radiance_ptr, normal=normal_ptr, depth=depth_ptr)
        out = Outputs(rgba=rgba_out_ptr or None, radiance=radiance_out_ptr or None)
        params = DenoiseParams(iterations, sigma_luminance, sigma_depth, normal_power_log2)
        sec = C.c_double(0.0)
        _check(lib().tmpt_denoise(self._h, width, height, DEVICE, C.byref(inp), C.byref(params), C.byref(out), C.byref(sec), stream or None))
        return sec.value

    def render_into(self, camera, width: int, height: int, spp: int, host_ptr: int):
        """One frame into caller-owned HOST memory (w*h*4 bytes, e.g. a pinned buffer) -> (rayCount, seconds): tmpt_render as a
        C caller uses it, without this binding allocating the frame."""
        cam = _f32(camera).reshape(22)
        rays, sec = C.c_uint64(0), C.c_double(0.0)
        _check(lib().tmpt_render(self._h, _ptr(cam), width, height, spp, HOST, host_ptr, C.byref(rays), C.byref(sec), None))
        return rays.value, sec.value

    def render_kernel_choice(self):
        """-> (kernel of the last frame: 0 k_render, 1 k_render_paths, -1 none yet; the probe's escape fraction)."""
        k, e = C.c_int(-1), C.c_float(0.0)
        _check(lib().tmpt_render_kernel_choice(self._h, C.byref(k), C.byref(e)))
        return k.value, e.value

    def traversal_stats(self, camera, width: int, height: int, spp: int) -> dict:
        """Instrumented render pass -> mean box / triangle tests per ray (bench.py's roofline figures)."""
        cam = _f32(camera).reshape(22)
        st = np.zeros(STATS_COUNT, np.uint64)
        _check(lib().tmpt_render_stats(self._h, _ptr(cam), width, height, spp, _ptr(st)))
        return _stats_dict(st)

    def hit_scene_stats(self, rays_ptr: int, n: int, mode: int = HIT_CLOSEST, tMin: float = K_MIN_T, tMax: float = K_MAX_T) -> dict:
        st = np.zeros(STATS_COUNT, np.uint64)
        _check(lib().tmpt_hit_scene_stats(self._h, rays_ptr, n, tMin, tMax, mode, _ptr(st)))
        d = _stats_dict(st)
        d["hit_rate"] = int(st[3]) / max(int(st[0]), 1)
        return d

    def render_device(self, camera, width: int, height: int, spp: int, frame_ptr: int, stream: int = 0):
        """One frame into a device buffer (w*h*4 bytes) -> (rayCount, seconds)."""
        cam = _f32(camera).reshape(22)
        rays, sec = C.c_uint64(0), C.c_double(0.0)
        _check(lib().tmpt_render(self._h, _ptr(cam), width, height, spp, DEVICE, frame_ptr, C.byref(rays), C.byref(sec), stream or None))
        return rays.value, sec.value

    def render_stripes(self, camera, width: int, height: int, spp: int, stripe: int, rank: int, world: int, out_ptr: int,
                       ray_count_ptr: int, peer_frame_ptr: int = 0, stream: int = 0):
        """This rank's row stripes (asynchronous); see tmpt_render_stripes."""
        cam = _f32(camera).reshape(22)
        _check(lib().tmpt_render_stripes(self._h, _ptr(cam), width, height, spp, stripe, rank, world, out_ptr or None,
                                         peer_frame_ptr or None, ray_count_ptr, stream or None))
