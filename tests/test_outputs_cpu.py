"""tmpt_outputs (linear radiance and first-hit AOVs) on the CPU: the product's integrator compiled for the host (tests/aov/emu_aov.cpp)
against the oracle's restatement (tests/aov/oracle_aov.c), bit for bit, and the argument checks of the two entry points."""
import ctypes as C

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from aov_binding import AovEmu, AovOracle
from conftest import load_scene

FLOATS = ("radiance", "normal", "depth")


def same_bits(a, b):
    """Float buffers equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


@pytest.fixture(scope="module")
def aov_oracle():
    return AovOracle()


@pytest.fixture(scope="module")
def aov_emu():
    return AovEmu()


def _camera(oracle, sc, w, h):
    return oracle.camera_for_scene(sc["bounds_min"], sc["bounds_max"], w, h)


# spp 1: one chunk; 9: one-sample chunks; 100: 3-sample chunks, the last one ragged; 256: 8-sample chunks
@pytest.mark.parametrize("name,w,h", [("cube", 24, 14), ("suzanne", 16, 9), ("triangle", 21, 11)])
@pytest.mark.parametrize("spp", [1, 9, 100, 256])
def test_emulated_outputs_equal_the_oracle(oracle, aov_oracle, aov_emu, name, w, h, spp):
    sc = load_scene(name)
    cam = _camera(oracle, sc, w, h)
    want, orays = aov_oracle.render_aov(sc["tris"], cam, w, h, spp)
    es = aov_emu.scene(sc["tris"])
    got, rays = aov_emu.render_aov(es, cam, w, h, spp)
    es.close()
    assert rays == orays
    assert (got["rgba"] == want["rgba"]).all() and (got["triangle"] == want["triangle"]).all()
    for k in FLOATS:
        assert same_bits(got[k], want[k]), k
    _, _, lin = oracle.render(sc["tris"], cam, w, h, spp, linear=True)
    assert same_bits(got["radiance"][..., :3], lin) and (got["radiance"][..., 3] == 1.0).all()
    hit = got["triangle"] >= 0
    assert hit.any() and (got["normal"][..., 3][hit] > 0).all()  # sample 0 hit: coverage > 0
    cov = got["normal"][..., 3]
    assert np.isinf(got["depth"][cov == 0]).all() and np.isfinite(got["depth"][cov > 0]).all()
    assert ((cov >= 0) & (cov <= 1)).all()


@pytest.mark.parametrize("rng", [0, 1])
def test_oracle_aov_frame_is_orc_render_frame(oracle, aov_oracle, rng):
    """orc_render_aov traces the paths orc_render traces: same rgba, linear mean and ray count, both RNG layouts, a row range."""
    sc = load_scene("cube")
    w, h, spp = 20, 12, 40
    cam = _camera(oracle, sc, w, h)
    for rows in (None, (3, 8)):
        want, wrays, lin = oracle.render(sc["tris"], cam, w, h, spp, rng=rng, rows=rows, linear=True)
        got, rays = aov_oracle.render_aov(sc["tris"], cam, w, h, spp, rng=rng, rows=rows)
        r0, r1 = rows or (0, h)
        assert rays == wrays
        assert (got["rgba"] == want).all()
        assert same_bits(got["radiance"][r0:r1, :, :3], lin[r0:r1])


def test_depth_and_normal_restate_the_hit_query(oracle, aov_oracle):
    """At spp = 1 the AOVs are the oracle's HitScene answer for the sample's camera ray: the triangle id, t as depth, the normal."""
    sc = load_scene("suzanne")
    w, h = 12, 8
    cam = _camera(oracle, sc, w, h)
    out, _ = aov_oracle.render_aov(sc["tris"], cam, w, h, 1)
    tri = out["triangle"]
    assert (tri >= 0).any() and (tri < 0).any()
    hit = tri >= 0
    assert (out["normal"][..., 3][hit] == 1.0).all() and (out["normal"][..., 3][~hit] == 0.0).all()
    assert np.allclose(np.linalg.norm(out["normal"][..., :3][hit], axis=-1), 1.0, atol=1e-5)
    assert np.isinf(out["depth"][~hit]).all() and (out["depth"][hit] > 0).all()


def test_output_entry_points_check_their_arguments():
    """Each argument error returns TMPT_ERR_ARG and leaves a message, before any device work (no GPU needed)."""
    L = tm.lib()
    L.tmpt_last_error.restype = C.c_char_p
    N = None
    fake_scene = C.create_string_buffer(4096)  # never dereferenced: every call below fails its argument checks first
    cam = (C.c_float * 22)()
    rgba = (C.c_uint8 * 64)()
    radiance = (C.c_float * 64)()
    depth = (C.c_float * 16)()
    s, c = C.cast(fake_scene, C.c_void_p), C.cast(cam, C.c_void_p)
    none = tm.Outputs()
    only_rgba = tm.Outputs(rgba=C.addressof(rgba))
    aov = tm.Outputs(rgba=C.addressof(rgba), radiance=C.addressof(radiance), depth=C.addressof(depth))
    calls = {
        "render: NULL scene": (lambda: L.tmpt_render_outputs(N, c, 4, 4, 1, tm.HOST, C.byref(only_rgba), N, N, N), "NULL scene"),
        "render: NULL camera": (lambda: L.tmpt_render_outputs(s, N, 4, 4, 1, tm.HOST, C.byref(only_rgba), N, N, N), "NULL scene / camera"),
        "render: width 0": (lambda: L.tmpt_render_outputs(s, c, 0, 4, 1, tm.HOST, C.byref(only_rgba), N, N, N), "out of range"),
        "render: height 10001": (lambda: L.tmpt_render_outputs(s, c, 4, 10001, 1, tm.HOST, C.byref(only_rgba), N, N, N), "out of range"),
        "render: spp 1025": (lambda: L.tmpt_render_outputs(s, c, 4, 4, 1025, tm.HOST, C.byref(only_rgba), N, N, N), "out of range"),
        "render: NULL out": (lambda: L.tmpt_render_outputs(s, c, 4, 4, 1, tm.HOST, N, N, N, N), "out is NULL"),
        "render: nothing requested": (lambda: L.tmpt_render_outputs(s, c, 4, 4, 1, tm.HOST, C.byref(none), N, N, N), "no output requested"),
        "render: bad mem": (lambda: L.tmpt_render_outputs(s, c, 4, 4, 1, 7, C.byref(aov), N, N, N), "mem 7"),
        "pass: NULL scene": (lambda: L.tmpt_progressive_pass_outputs(N, c, 1, tm.HOST, C.byref(only_rgba), N, N, N, N), "NULL scene"),
        "pass: NULL out": (lambda: L.tmpt_progressive_pass_outputs(s, c, 1, tm.HOST, N, N, N, N, N), "out is NULL"),
        "pass: nothing requested": (lambda: L.tmpt_progressive_pass_outputs(s, c, 1, tm.HOST, C.byref(none), N, N, N, N), "no output requested"),
        "pass: bad mem": (lambda: L.tmpt_progressive_pass_outputs(s, c, 1, -1, C.byref(only_rgba), N, N, N, N), "mem -1"),
        "pass: an AOV": (lambda: L.tmpt_progressive_pass_outputs(s, c, 1, tm.HOST, C.byref(aov), N, N, N, N), "rgba and radiance only"),
    }
    for name, (call, message) in calls.items():
        assert call() == tm.TMPT_ERR_ARG, name
        assert message in L.tmpt_last_error().decode(), (name, L.tmpt_last_error())


def test_header_states_the_outputs_contract():
    import os
    from conftest import ROOT
    hdr = open(os.path.join(ROOT, "include", "tmpt.h")).read()
    assert "#define TMPT_ABI_VERSION 3" in hdr
    assert [f[0] for f in tm.Outputs._fields_] == ["rgba", "radiance", "normal", "depth", "triangle"] == list(tm.OUTPUTS)
    with pytest.raises(ValueError):
        tm._output_arrays(("rgba", "albedo"), 2, 2)
