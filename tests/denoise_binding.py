"""ctypes binding of the denoiser checkers -- TEST INFRASTRUCTURE, never the product path.

``DenoiseOracle`` -> tests/denoise/liboracle_denoise.so: orc_denoise, a plain-C restatement of tmpt_denoise from include/tmpt.h
``DenoiseEmu``    -> tests/denoise/libemu_denoise.so:    emu_denoise, the product's denoise.cuh compiled for the host

Both take the host arrays Scene.denoise takes (radiance / normal [h,w,4], depth [h,w], float32) and return what it returns:
{"rgba", "radiance"}."""
import ctypes as C
import os
import subprocess

import numpy as np

from aov_binding import CUDA_INC, _p, _stale

HERE = os.path.dirname(os.path.abspath(__file__))
DENOISE = os.path.join(HERE, "denoise")
ROOT = os.path.dirname(HERE)
DEFAULTS = {"iterations": 5, "sigma_luminance": 4.0, "sigma_depth": 1.0, "normal_power_log2": 7}  # Scene.denoise's


def _inputs(radiance, normal, depth):
    radiance, normal, depth = (np.ascontiguousarray(a, np.float32) for a in (radiance, normal, depth))
    h, w = depth.shape
    assert radiance.shape == (h, w, 4) and normal.shape == (h, w, 4)
    return radiance, normal, depth, w, h


def _outputs(w, h):
    return {"rgba": np.zeros((h, w, 4), np.uint8), "radiance": np.zeros((h, w, 4), np.float32)}


def build_oracle():
    so, src = os.path.join(DENOISE, "liboracle_denoise.so"), os.path.join(DENOISE, "oracle_denoise.c")
    if _stale(so, [src]):
        subprocess.run(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread", "-Wall",
                        "-o", so, src, "-lm"], check=True)
    return so


def build_emu():
    so, src = os.path.join(DENOISE, "libemu_denoise.so"), os.path.join(DENOISE, "emu_denoise.cpp")
    csrc = os.path.join(ROOT, "toymeshpathtracer_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if _stale(so, deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-I" + CUDA_INC,
                        "-o", so, src], check=True)
    return so


class DenoiseOracle:
    def __init__(self):
        self.L = C.CDLL(build_oracle())
        self.L.orc_expneg.argtypes = [C.c_float]
        self.L.orc_expneg.restype = C.c_float
        self.threads = int(os.environ.get("ORACLE_THREADS", os.cpu_count() or 1))

    def expneg(self, x):
        return self.L.orc_expneg(x)

    def denoise(self, radiance, normal, depth, iterations=5, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=7, threads=None):
        radiance, normal, depth, w, h = _inputs(radiance, normal, depth)
        out = _outputs(w, h)
        self.L.orc_denoise(w, h, _p(radiance), _p(normal), _p(depth), iterations, C.c_float(sigma_luminance), C.c_float(sigma_depth),
                           normal_power_log2, _p(out["rgba"]), _p(out["radiance"]), threads or self.threads)
        return out


class DenoiseEmu:
    def __init__(self):
        self.L = C.CDLL(build_emu())
        self.L.emu_expneg.argtypes = [C.c_float]
        self.L.emu_expneg.restype = C.c_float

    def expneg(self, x):
        return self.L.emu_expneg(x)

    def denoise(self, radiance, normal, depth, iterations=5, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=7):
        radiance, normal, depth, w, h = _inputs(radiance, normal, depth)
        out = _outputs(w, h)
        self.L.emu_denoise(w, h, _p(radiance), _p(normal), _p(depth), iterations, C.c_float(sigma_luminance), C.c_float(sigma_depth),
                           normal_power_log2, _p(out["rgba"]), _p(out["radiance"]))
        return out
