"""Adaptive progressive passes on the CPU: the product's integrator.cuh helpers compiled for the host (tests/adaptive/emu_adaptive.cpp)
against the oracle's serial restatement (tests/adaptive/oracle_adaptive.c), bit for bit over multi-pass sessions; the stop rule
against a numpy float32 restatement; the argument checks of tmpt_progressive_pass_adaptive."""
import ctypes as C
import math

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from adaptive_binding import AdaptiveEmu, AdaptiveOracle, State
from conftest import load_scene


def same_bits(a, b):
    """Float arrays equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


@pytest.fixture(scope="module")
def ad_oracle():
    return AdaptiveOracle()


@pytest.fixture(scope="module")
def ad_emu():
    return AdaptiveEmu()


@pytest.mark.parametrize("name,w,h", [("cube", 24, 14), ("suzanne", 16, 9), ("triangle", 21, 11)])
@pytest.mark.parametrize("schedule", [(1, 1, 1, 1), (4, 2, 8), (16, 16, 16)])
@pytest.mark.parametrize("tolerance", [0.0, 0.25, 2.0, 1e6])
@pytest.mark.parametrize("min_chunks", [2, 5])
def test_emulated_session_equals_the_oracle(oracle, ad_oracle, ad_emu, name, w, h, schedule, tolerance, min_chunks):
    sc = load_scene(name)
    cam = oracle.camera_for_scene(sc["bounds_min"], sc["bounds_max"], w, h)
    es = ad_emu.scene(sc["tris"])
    want_state, got_state = State(w, h), State(w, h)
    prefix = 0
    for k in schedule:
        want, wrays, wactive = ad_oracle.pass_(sc["tris"], cam, want_state, k, tolerance, min_chunks)
        got, rays, active = ad_emu.pass_(es, cam, got_state, k, tolerance, min_chunks)
        assert (rays, active) == (wrays, wactive)
        assert (got["rgba"] == want["rgba"]).all() and (got["samples"] == want["samples"]).all()
        assert same_bits(got["radiance"], want["radiance"])
        assert (got_state.n == want_state.n).all()
        for f in ("sum", "mean", "m2"):
            assert same_bits(getattr(got_state, f), getattr(want_state, f)), f
        prefix += k
        # with fixed params a stopped pixel stays stopped: every n is a prefix sum of the pass sizes
        assert set(np.unique(want_state.n)) <= set(np.cumsum(schedule)), np.unique(want_state.n)
        if tolerance == 0.0:
            assert (want_state.n == prefix).all() and active == w * h
    es.close()
    if tolerance == 0.0 and prefix >= 32:  # a uniform session after P >= 32 chunks is tmpt_render(spp = 8 P)
        img, _, lin = oracle.render(sc["tris"], cam, w, h, 8 * prefix, linear=True)
        assert (got["rgba"] == img).all() and same_bits(got["radiance"][..., :3], lin)
    if tolerance == 1e6:  # everything stops at minChunks
        assert (want_state.n <= max(min_chunks + max(schedule), schedule[0])).all()


def _np_converged(n, mean, m2, tol, min_chunks):
    """The stop rule of include/tmpt.h in numpy float32, one rounding per operation."""
    f = np.float32
    n32 = np.asarray(n, np.uint32)
    a = np.asarray(m2, f) * f(65025.0)
    nm1 = (n32 - np.uint32(1)).astype(f)  # (n - 1 wraps for n = 0, as the uint32 expression does; such n fail n >= minChunks)
    b = ((n32.astype(f) * nm1) * (f(4.0) * np.fmax(np.asarray(mean, f), f(2.0 ** -16)))) * (f(tol) * f(tol))
    with np.errstate(invalid="ignore"):
        return (f(tol) != f(0.0)) & (n32 >= np.uint32(min_chunks)) & ~(a > b)


def test_stop_rule_equals_a_float32_restatement(ad_oracle, ad_emu):
    rng = np.random.default_rng(7)
    cases = []
    for _ in range(4000):
        n = int(rng.choice([0, 1, 2, 3, 5, 64, 1000, 1 << 21, (1 << 24) + 1]))
        mean = float(np.float32(rng.choice([rng.uniform(-0.1, 2.0), 0.0, -0.5, 1e-9, 2.0 ** -17, math.nan])))
        m2 = float(np.float32(rng.choice([rng.uniform(0, 1e-2) * n, 0.0, 1e-12, math.nan, math.inf])))
        tol = float(np.float32(rng.choice([0.0, 0.1, 0.5, 1.0, 2.0, rng.uniform(0, 4)])))
        cases.append((n, mean, m2, tol, int(rng.choice([2, 4, 5, 1 << 21]))))
    cases += [(1, 0.5, 0.0, 1.0, 2), (2, 0.5, 0.0, 0.0, 2), (2, 0.5, 0.0, 1.0, 2), (10, math.nan, math.nan, 1.0, 2),
              (10, math.nan, math.nan, 1.0, 11), (10, 0.3, math.nan, 1.0, 2), (10, -1.0, 1e-3, 1.0, 2), (10, 0.0, 0.0, 1e-30, 2)]
    want = [bool(_np_converged(*c)) for c in cases]
    assert [ad_emu.converged(*c) for c in cases] == want
    assert [ad_oracle.converged(*c) for c in cases] == want
    assert any(want) and not all(want)
    assert ad_emu.converged(10, math.nan, math.nan, 1.0, 2) and not ad_emu.converged(10, math.nan, math.nan, 1.0, 11)
    assert not ad_emu.converged(100, 0.5, 0.0, 0.0, 2)  # tolerance 0: never converged, even with M2 = 0
    assert ad_emu.converged(100, 0.5, 0.0, 0.01, 2) and not ad_emu.converged(1, 0.5, 0.0, 1.0, 2)


def test_adaptive_pass_checks_its_arguments():
    """Each argument error returns TMPT_ERR_ARG and leaves a message, before any device work (no GPU needed)."""
    L = tm.lib()
    L.tmpt_last_error.restype = C.c_char_p
    N = None
    fake_scene = C.create_string_buffer(4096)  # never dereferenced: every call below fails its argument checks first
    cam = (C.c_float * 22)()
    rgba = (C.c_uint8 * 64)()
    depth = (C.c_float * 16)()
    s, c = C.cast(fake_scene, C.c_void_p), C.cast(cam, C.c_void_p)
    only_rgba = tm.Outputs(rgba=C.addressof(rgba))
    none = tm.Outputs()
    aov = tm.Outputs(rgba=C.addressof(rgba), depth=C.addressof(depth))
    ok = tm.Adaptive(0.5, 4)

    def call(scene=s, camera=c, n=1, params=ok, mem=tm.HOST, out=only_rgba):
        return L.tmpt_progressive_pass_adaptive(scene, camera, n, C.byref(params) if params is not None else N, mem,
                                                C.byref(out) if out is not None else N, N, N, N, N, N)

    calls = {
        "NULL scene": (lambda: call(scene=N), "NULL scene"),
        "NULL camera": (lambda: call(camera=N), "NULL scene / camera"),
        "NULL out": (lambda: call(out=None), "out is NULL"),
        "nothing requested": (lambda: call(out=none), "no output requested"),
        "bad mem": (lambda: call(mem=3), "mem 3"),
        "an AOV": (lambda: call(out=aov), "rgba and radiance only"),
        "NULL params": (lambda: call(params=None), "params is NULL"),
        "negative tolerance": (lambda: call(params=tm.Adaptive(-0.5, 4)), "tolerance"),
        "NaN tolerance": (lambda: call(params=tm.Adaptive(math.nan, 4)), "tolerance"),
        "infinite tolerance": (lambda: call(params=tm.Adaptive(math.inf, 4)), "tolerance"),
        "minChunks 1": (lambda: call(params=tm.Adaptive(0.5, 1)), "minChunks 1"),
        "minChunks 2^21 + 1": (lambda: call(params=tm.Adaptive(0.5, (1 << 21) + 1)), "minChunks 2097153"),
        "nChunks 0": (lambda: call(n=0), "nChunks 0"),
        "nChunks 129": (lambda: call(n=129), "nChunks 129"),
    }
    for name, (fn, message) in calls.items():
        assert fn() == tm.TMPT_ERR_ARG, name
        assert message in L.tmpt_last_error().decode(), (name, L.tmpt_last_error())


def test_header_declares_the_adaptive_pass():
    import os
    from conftest import ROOT
    hdr = open(os.path.join(ROOT, "include", "tmpt.h")).read()
    assert "#define TMPT_ABI_VERSION 3" in hdr and "tmpt_progressive_pass_adaptive" in tm.ABI_SYMBOLS
    assert [f[0] for f in tm.Adaptive._fields_] == ["tolerance", "minChunks"] and C.sizeof(tm.Adaptive) == 8
