"""ctypes binding of the adaptive-pass checkers -- TEST INFRASTRUCTURE, never the product path.

``AdaptiveOracle`` -> tests/adaptive/liboracle_adaptive.so: orc_pass_adaptive, oracle/oracle.c's restatement of one adaptive pass
``AdaptiveEmu``    -> tests/adaptive/libemu_adaptive.so:    tests/emu plus emu_pass_adaptive, the product's integrator.cuh helpers

Both run one pass of tmpt_progressive_pass_adaptive over a ``State`` (the per-pixel n, colour sum, Welford mean and M2 a session
keeps) and return what Scene.progressive_pass_adaptive returns: ({"rgba", "radiance", "samples"}, rays, active pixels)."""
import ctypes as C
import os
import subprocess

import numpy as np

from aov_binding import CUDA_INC, _p, _stale

HERE = os.path.dirname(os.path.abspath(__file__))
ADAPTIVE = os.path.join(HERE, "adaptive")
ROOT = os.path.dirname(HERE)


class State:
    """A session's per-pixel state after tmpt_progressive_begin: every pixel at n = 0."""

    def __init__(self, w, h):
        self.w, self.h = w, h
        self.n = np.zeros((h, w), np.uint32)
        self.sum = np.zeros((h, w, 4), np.float32)
        self.mean = np.zeros((h, w), np.float32)
        self.m2 = np.zeros((h, w), np.float32)

    def copy(self):
        c = State(self.w, self.h)
        for k in ("n", "sum", "mean", "m2"):
            setattr(c, k, getattr(self, k).copy())
        return c


def _outputs(w, h):
    return {"rgba": np.zeros((h, w, 4), np.uint8), "radiance": np.zeros((h, w, 4), np.float32), "samples": np.zeros((h, w), np.int32)}


def build_oracle():
    so, src = os.path.join(ADAPTIVE, "liboracle_adaptive.so"), os.path.join(ADAPTIVE, "oracle_adaptive.c")
    deps = [src, os.path.join(ROOT, "oracle", "oracle.c"), os.path.join(ROOT, "oracle", "oracle.h")]
    if _stale(so, deps):
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread", "-Wall",
                        "-o", so, src, "-lm"], check=True)
    return so


def build_emu():
    so, src = os.path.join(ADAPTIVE, "libemu_adaptive.so"), os.path.join(ADAPTIVE, "emu_adaptive.cpp")
    csrc = os.path.join(ROOT, "toymeshpathtracer_b200", "csrc")
    deps = [src, os.path.join(HERE, "emu", "emu.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if _stale(so, deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                        "-I" + CUDA_INC, "-o", so, src], check=True)
    return so


class AdaptiveOracle:
    def __init__(self):
        self.L = C.CDLL(build_oracle())
        self.L.orc_adaptive_converged.argtypes = [C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_int]
        self.threads = int(os.environ.get("ORACLE_THREADS", os.cpu_count() or 1))

    def converged(self, n, mean, m2, tolerance, min_chunks):
        return bool(self.L.orc_adaptive_converged(n, mean, m2, tolerance, min_chunks))

    def pass_(self, tris9, cam22, state, n_chunks, tolerance, min_chunks, rows=None, threads=None):
        """One pass over `state` (updated in place); with rows=(r0, r1) only those rows (the others stay zero)."""
        tris9 = np.ascontiguousarray(tris9, np.float32).reshape(-1, 9)
        out = _outputs(state.w, state.h)
        rays, active = C.c_int64(0), C.c_int64(0)
        r0, r1 = rows if rows else (0, state.h)
        self.L.orc_pass_adaptive(_p(tris9), tris9.shape[0], _p(np.ascontiguousarray(cam22, np.float32)), state.w, state.h, n_chunks,
                                 C.c_float(tolerance), min_chunks, r0, r1, _p(state.n), _p(state.sum), _p(state.mean), _p(state.m2),
                                 _p(out["rgba"]), _p(out["radiance"]), _p(out["samples"]), C.byref(active), C.byref(rays),
                                 threads or self.threads)
        return out, rays.value, active.value


class AdaptiveEmu:
    def __init__(self):
        from emu_binding import EmuScene
        self.L = C.CDLL(build_emu())
        self.L.emu_scene_create2.restype = C.c_void_p
        self.L.emu_adaptive_converged.argtypes = [C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_int]
        self._scene = EmuScene

    def scene(self, tris):
        return self._scene(self.L, tris)

    def converged(self, n, mean, m2, tolerance, min_chunks):
        return bool(self.L.emu_adaptive_converged(n, mean, m2, tolerance, min_chunks))

    def pass_(self, scene, cam22, state, n_chunks, tolerance, min_chunks, rows=None):
        out = _outputs(state.w, state.h)
        rays, active = C.c_longlong(0), C.c_longlong(0)
        r0, r1 = rows if rows else (0, state.h)
        self.L.emu_pass_adaptive(scene.h, _p(np.ascontiguousarray(cam22, np.float32)), state.w, state.h, n_chunks, C.c_float(tolerance),
                                 min_chunks, r0, r1, _p(state.n), _p(state.sum), _p(state.mean), _p(state.m2), _p(out["rgba"]),
                                 _p(out["radiance"]), _p(out["samples"]), C.byref(active), C.byref(rays))
        return out, rays.value, active.value
