"""tmpt_denoise on the CPU: the product's denoise.cuh compiled for the host (tests/denoise/emu_denoise.cpp) against the plain-C
restatement of include/tmpt.h's filter (tests/denoise/oracle_denoise.c), bit for bit, on rendered AOV frames and synthetic buffers;
expneg against float64 exp; the identity at 0 iterations; class separation; the argument checks of tmpt_denoise."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from aov_binding import AovOracle
from conftest import ROOT, load_scene
from denoise_binding import DenoiseEmu, DenoiseOracle


def same_bits(a, b):
    """Float arrays equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


@pytest.fixture(scope="module")
def dn_oracle():
    return DenoiseOracle()


@pytest.fixture(scope="module")
def dn_emu():
    return DenoiseEmu()


_FRAMES = {}


def rendered(name, w, h, spp):
    """orc_render_aov's frame of a golden scene: (outputs dict) -- cached per module run."""
    key = (name, w, h, spp)
    if key not in _FRAMES:
        sc = load_scene(name)
        from oracle.pyoracle import Oracle
        cam = Oracle().camera_for_scene(sc["bounds_min"], sc["bounds_max"], w, h)
        _FRAMES[key] = AovOracle().render_aov(sc["tris"], cam, w, h, spp)[0]
    return _FRAMES[key]


def check_equal(dn_oracle, dn_emu, radiance, normal, depth, **params):
    want = dn_oracle.denoise(radiance, normal, depth, **params)
    got = dn_emu.denoise(radiance, normal, depth, **params)
    assert (got["rgba"] == want["rgba"]).all(), params
    assert same_bits(got["radiance"], want["radiance"]), params
    assert (want["radiance"][..., 3] == 1.0).all() and (want["rgba"][..., 3] == 255).all()
    return want


PARAMS = [dict(iterations=5, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=7),
          dict(iterations=0, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=7),
          dict(iterations=1, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=0),
          dict(iterations=8, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=8),
          dict(iterations=5, sigma_luminance=1e-30, sigma_depth=1e-30, normal_power_log2=7),
          dict(iterations=5, sigma_luminance=3.0e38, sigma_depth=3.0e38, normal_power_log2=8),
          dict(iterations=3, sigma_luminance=0.5, sigma_depth=100.0, normal_power_log2=1)]


@pytest.mark.parametrize("name,w,h", [("cube", 24, 14), ("suzanne", 20, 12), ("teapot", 22, 13), ("triangle", 17, 9)])
@pytest.mark.parametrize("spp", [1, 4, 64])
def test_emulation_equals_the_oracle_on_rendered_frames(dn_oracle, dn_emu, name, w, h, spp):
    f = rendered(name, w, h, spp)
    for prm in PARAMS:
        check_equal(dn_oracle, dn_emu, f["radiance"], f["normal"], f["depth"], **prm)


def synthetic(w, h, seed, sky=0.3, nan=0.0, inf=0.0, zero_normal=0.0):
    rng = np.random.default_rng(seed)
    rad = rng.gamma(0.6, 0.4, (h, w, 4)).astype(np.float32)
    rad[..., 3] = 1.0
    nrm = rng.normal(size=(h, w, 4)).astype(np.float32)
    nrm[..., 3] = rng.choice(np.float32([0.125, 0.5, 1.0]), (h, w))  # fractional coverage
    skym = rng.random((h, w)) < sky
    nrm[skym] = 0.0
    dep = rng.uniform(0.5, 20.0, (h, w)).astype(np.float32)
    dep[skym] = np.inf
    rad[rng.random((h, w)) < nan, rng.integers(0, 3)] = np.nan
    rad[rng.random((h, w)) < inf, rng.integers(0, 3)] = np.inf
    zm = (rng.random((h, w)) < zero_normal) & ~skym
    nrm[zm, :3] = 0.0
    return rad, nrm, dep


@pytest.mark.parametrize("w,h", [(1, 1), (1, 13), (13, 1), (3, 2), (4, 4), (5, 3), (37, 29)])
@pytest.mark.parametrize("kind", ["mixed", "all_sky", "nan_inf", "zero_normals"])
def test_emulation_equals_the_oracle_on_synthetic_buffers(dn_oracle, dn_emu, w, h, kind):
    """1x1, 1xN and Nx1 frames, frames smaller than the widest tap (2 * 128 pixels at iteration 8), all-sky frames, NaN and inf
    radiance, zero normal sums and fractional coverage."""
    args = {"mixed": {}, "all_sky": {"sky": 1.0}, "nan_inf": {"nan": 0.15, "inf": 0.05}, "zero_normals": {"zero_normal": 0.3}}[kind]
    rad, nrm, dep = synthetic(w, h, w * 131 + h, **args)
    for prm in PARAMS:
        check_equal(dn_oracle, dn_emu, rad, nrm, dep, **prm)


def test_extreme_values(dn_oracle, dn_emu):
    """Huge, tiny, negative and subnormal radiance; huge normals (dot(N, N) overflows); zero and negative depth; NaN coverage."""
    rad, nrm, dep = synthetic(19, 11, 5, nan=0.05)
    rad[0, :5, :3] = np.float32([[3e38, 1e-42, 0.0], [-1.0, 2.0, 0.5], [1e30, 1e30, 1e30], [-0.0, 0.0, 1e-45], [0.25, 0.25, 0.25]])[:, :]
    nrm[1, :3, :3] = np.float32(1e30)
    nrm[2, :2, 3] = np.nan
    dep[3, :4] = np.float32([0.0, -1.0, 1e-40, 3e38])
    for prm in PARAMS:
        check_equal(dn_oracle, dn_emu, rad, nrm, dep, **prm)


def test_nan_pixels_become_the_mean_of_their_valid_neighbours(dn_oracle, dn_emu):
    rad, nrm, dep = synthetic(16, 10, 9, nan=0.1)
    assert np.isnan(rad[..., :3]).any()
    want = check_equal(dn_oracle, dn_emu, rad, nrm, dep, iterations=1)
    assert np.isfinite(want["radiance"]).all()
    # a NaN pixel with no valid pixel of its class in reach keeps its input
    rad2, nrm2, dep2 = rad.copy(), nrm.copy(), dep.copy()
    nrm2[...] = 0.0
    dep2[...] = np.inf
    nrm2[4, 4] = (0.0, 1.0, 0.0, 1.0)
    dep2[4, 4] = 2.0
    rad2[4, 4, 0] = np.nan
    out = check_equal(dn_oracle, dn_emu, rad2, nrm2, dep2, iterations=3)
    assert np.isnan(out["radiance"][4, 4, 0]) and out["rgba"][4, 4, 0] == 0


def test_expneg_is_within_one_ulp_of_exp(dn_oracle, dn_emu):
    xs = np.concatenate([np.linspace(0.0, 110.0, 400001, dtype=np.float32),
                         np.float32(2.0) ** -np.arange(1, 150, dtype=np.float32),
                         np.random.default_rng(3).uniform(0.0, 104.0, 20000).astype(np.float32),
                         np.float32([103.9, 103.97, 103.972, 103.98, 104.0, 87.3, 88.7, 1e-45])])
    got = np.array([dn_emu.expneg(float(x)) for x in xs], np.float32)
    want = np.array([dn_oracle.expneg(float(x)) for x in xs], np.float32)
    assert (got.view(np.uint32) == want.view(np.uint32)).all()
    ref = np.exp(-xs.astype(np.float64)).astype(np.float32)
    ulps = np.abs(got.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, xs[np.argmax(ulps)]
    specials = {0.0: 1.0, -0.0: 1.0, -5.0: 1.0, -math.inf: 1.0, math.inf: 0.0, math.nan: 0.0, 104.0: 0.0, 3e38: 0.0}
    for x, v in specials.items():
        assert dn_emu.expneg(x) == v and dn_oracle.expneg(x) == v, x


@pytest.mark.parametrize("name,w,h,spp", [("cube", 24, 14, 4), ("suzanne", 20, 12, 64), ("triangle", 17, 9, 1)])
def test_zero_iterations_is_the_identity(dn_oracle, dn_emu, name, w, h, spp):
    f = rendered(name, w, h, spp)
    out = check_equal(dn_oracle, dn_emu, f["radiance"], f["normal"], f["depth"], iterations=0)
    assert same_bits(out["radiance"], f["radiance"]) and (out["rgba"] == f["rgba"]).all()


def test_classes_do_not_mix(dn_oracle, dn_emu):
    """Changing every hit-class radiance leaves every sky-class output bit-identical (and the other way round)."""
    f = rendered("suzanne", 24, 14, 4)
    hit = f["normal"][..., 3] > 0
    assert hit.any() and (~hit).any()
    base = dn_emu.denoise(f["radiance"], f["normal"], f["depth"], iterations=5)
    for cls in (hit, ~hit):
        rad = f["radiance"].copy()
        rad[cls, :3] = rad[cls, :3] * np.float32(3.0) + np.float32(0.25)
        rad[np.argwhere(cls)[0][0], np.argwhere(cls)[0][1], 1] = np.nan
        got = check_equal(dn_oracle, dn_emu, rad, f["normal"], f["depth"], iterations=5)
        assert same_bits(got["radiance"][~cls], base["radiance"][~cls]) and (got["rgba"][~cls] == base["rgba"][~cls]).all()
        assert not same_bits(got["radiance"][cls], base["radiance"][cls])


def test_denoise_checks_its_arguments():
    """Each argument error returns TMPT_ERR_ARG and leaves a message, before any device work (no GPU needed)."""
    L = tm.lib()
    N = None
    fake_scene = C.create_string_buffer(4096)  # never dereferenced: every call below fails its argument checks first
    rad, nrm = (C.c_float * 64)(), (C.c_float * 64)()
    dep, rgba = (C.c_float * 16)(), (C.c_uint8 * 64)()
    s = C.cast(fake_scene, C.c_void_p)
    full_in = tm.Outputs(radiance=C.addressof(rad), normal=C.addressof(nrm), depth=C.addressof(dep))
    only_rgba = tm.Outputs(rgba=C.addressof(rgba))
    ok = tm.DenoiseParams(5, 4.0, 1.0, 7)

    def call(scene=s, w=4, h=4, mem=tm.HOST, inp=full_in, params=ok, out=only_rgba):
        return L.tmpt_denoise(scene, w, h, mem, C.byref(inp) if inp is not None else N, C.byref(params) if params is not None else N,
                              C.byref(out) if out is not None else N, N, N)

    calls = {
        "NULL scene": (lambda: call(scene=N), "NULL scene"),
        "NULL in": (lambda: call(inp=None), "in is NULL"),
        "NULL params": (lambda: call(params=None), "params is NULL"),
        "NULL out": (lambda: call(out=None), "out is NULL"),
        "no radiance": (lambda: call(inp=tm.Outputs(normal=C.addressof(nrm), depth=C.addressof(dep))), "are required"),
        "no normal": (lambda: call(inp=tm.Outputs(radiance=C.addressof(rad), depth=C.addressof(dep))), "are required"),
        "no depth": (lambda: call(inp=tm.Outputs(radiance=C.addressof(rad), normal=C.addressof(nrm))), "are required"),
        "nothing requested": (lambda: call(out=tm.Outputs()), "no output requested"),
        "an AOV out": (lambda: call(out=tm.Outputs(rgba=C.addressof(rgba), depth=C.addressof(dep))), "rgba and radiance only"),
        "only an AOV out": (lambda: call(out=tm.Outputs(normal=C.addressof(nrm))), "no output requested"),
        "bad mem": (lambda: call(mem=2), "mem 2"),
        "width 0": (lambda: call(w=0), "0 x 4 out of range"),
        "height 10001": (lambda: call(h=10001), "4 x 10001 out of range"),
        "iterations -1": (lambda: call(params=tm.DenoiseParams(-1, 4.0, 1.0, 7)), "iterations -1"),
        "iterations 9": (lambda: call(params=tm.DenoiseParams(9, 4.0, 1.0, 7)), "iterations 9"),
        "normalPowerLog2 -1": (lambda: call(params=tm.DenoiseParams(5, 4.0, 1.0, -1)), "normalPowerLog2 -1"),
        "normalPowerLog2 9": (lambda: call(params=tm.DenoiseParams(5, 4.0, 1.0, 9)), "normalPowerLog2 9"),
        "sigmaLuminance 0": (lambda: call(params=tm.DenoiseParams(5, 0.0, 1.0, 7)), "sigmaLuminance"),
        "sigmaLuminance < 0": (lambda: call(params=tm.DenoiseParams(5, -1.0, 1.0, 7)), "sigmaLuminance"),
        "sigmaLuminance NaN": (lambda: call(params=tm.DenoiseParams(5, math.nan, 1.0, 7)), "sigmaLuminance"),
        "sigmaLuminance inf": (lambda: call(params=tm.DenoiseParams(5, math.inf, 1.0, 7)), "sigmaLuminance"),
        "sigmaDepth 0": (lambda: call(params=tm.DenoiseParams(5, 4.0, 0.0, 7)), "sigmaDepth"),
        "sigmaDepth NaN": (lambda: call(params=tm.DenoiseParams(5, 4.0, math.nan, 7)), "sigmaDepth"),
        "sigmaDepth inf": (lambda: call(params=tm.DenoiseParams(5, 4.0, math.inf, 7)), "sigmaDepth"),
    }
    for name, (fn, message) in calls.items():
        assert fn() == tm.TMPT_ERR_ARG, name
        assert message in L.tmpt_last_error().decode(), (name, L.tmpt_last_error())


def test_header_declares_the_denoiser():
    hdr = open(os.path.join(ROOT, "include", "tmpt.h")).read()
    assert "#define TMPT_ABI_VERSION 3" in hdr and "tmpt_denoise" in tm.ABI_SYMBOLS
    assert "int tmpt_denoise(tmpt_scene* scene, int width, int height, int mem, const tmpt_outputs* in" in hdr
    assert [f[0] for f in tm.DenoiseParams._fields_] == ["iterations", "sigmaLuminance", "sigmaDepth", "normalPowerLog2"]
    assert C.sizeof(tm.DenoiseParams) == 16
    assert [getattr(tm.DenoiseParams, f[0]).offset for f in tm.DenoiseParams._fields_] == [0, 4, 8, 12]
