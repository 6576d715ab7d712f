"""ctypes binding of the AOV checkers -- TEST INFRASTRUCTURE, never the product path.

``AovOracle``  -> tests/aov/liboracle_aov.so: orc_render_aov, oracle/oracle.c's restatement plus the buffers of tmpt_outputs
``AovEmu``     -> tests/aov/libemu_aov.so:    tests/emu plus emu_render_aov, the product's integrator compiled for the host

Both return the outputs as Scene.render_outputs does: {"rgba", "radiance", "normal", "depth", "triangle"} -> host arrays."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
AOV = os.path.join(HERE, "aov")
ROOT = os.path.dirname(HERE)
CUDA_INC = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
RNG_ROW, RNG_PIXEL = 0, 1
TRIG_LIBM, TRIG_SPEC = 0, 1


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _stale(so, deps):
    return not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps)


def _outputs(w, h):
    return {"rgba": np.zeros((h, w, 4), np.uint8), "radiance": np.zeros((h, w, 4), np.float32), "normal": np.zeros((h, w, 4), np.float32),
            "depth": np.zeros((h, w), np.float32), "triangle": np.full((h, w), -2, np.int32)}


def build_oracle():
    so, src = os.path.join(AOV, "liboracle_aov.so"), os.path.join(AOV, "oracle_aov.c")
    deps = [src, os.path.join(ROOT, "oracle", "oracle.c"), os.path.join(ROOT, "oracle", "oracle.h")]
    if _stale(so, deps):
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread", "-Wall",
                        "-o", so, src, "-lm"], check=True)
    return so


def build_emu():
    so, src = os.path.join(AOV, "libemu_aov.so"), os.path.join(AOV, "emu_aov.cpp")
    csrc = os.path.join(ROOT, "toymeshpathtracer_b200", "csrc")
    deps = [src, os.path.join(HERE, "emu", "emu.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if _stale(so, deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                        "-I" + CUDA_INC, "-o", so, src], check=True)
    return so


class AovOracle:
    def __init__(self):
        self.L = C.CDLL(build_oracle())
        self.threads = int(os.environ.get("ORACLE_THREADS", os.cpu_count() or 1))

    def render_aov(self, tris9, cam22, w, h, spp, rng=RNG_PIXEL, trig=TRIG_SPEC, rows=None, threads=None):
        """-> (outputs dict, rayCount); with rows=(r0, r1) only those rows are rendered (the others stay zero / -2)."""
        tris9 = np.ascontiguousarray(tris9, np.float32).reshape(-1, 9)
        out = _outputs(w, h)
        rc = C.c_int64(0)
        r0, r1 = rows if rows else (0, h)
        self.L.orc_render_aov(_p(tris9), tris9.shape[0], _p(np.ascontiguousarray(cam22, np.float32)), w, h, spp, rng, trig, r0, r1,
                              _p(out["rgba"]), _p(out["radiance"]), _p(out["normal"]), _p(out["depth"]), _p(out["triangle"]),
                              C.byref(rc), threads or self.threads)
        return out, rc.value


class AovEmu:
    def __init__(self):
        from emu_binding import EmuScene
        self.L = C.CDLL(build_emu())
        self.L.emu_scene_create2.restype = C.c_void_p
        self._scene = EmuScene

    def scene(self, tris):
        """The product's default build (binned SAH), as tests/emu_binding.Emu.scene makes it."""
        return self._scene(self.L, tris)

    def render_aov(self, scene, cam22, w, h, spp, rows=None):
        out = _outputs(w, h)
        rc = C.c_longlong(0)
        r0, r1 = rows if rows else (0, h)
        self.L.emu_render_aov(scene.h, _p(np.ascontiguousarray(cam22, np.float32)), w, h, spp, r0, r1, _p(out["rgba"]), _p(out["radiance"]),
                              _p(out["normal"]), _p(out["depth"]), _p(out["triangle"]), C.byref(rc))
        return out, rc.value
