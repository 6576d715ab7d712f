"""The build's two level loops (the binned-SAH build and the collapse to wide nodes) run in one cooperative launch each, or, on a
device without cooperative launch and under TMPT_BUILD_HOSTLOOP=1, as one launch and one read-back per level.  Both forms share
the build's scratch layout and geometry steps, so a scene built either way is the same scene: the same tree statistics, the same
bounds bit for bit and the same HitScene answers; and a refit of either leaves what a fresh scene has."""
import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from conftest import bits, load_rays, load_scene, sponza_scene

pytestmark = pytest.mark.gpu


def first_triangles(k):
    return load_scene("triangle")["tris"][:k]


SCENES = {
    "cube": lambda: load_scene("cube")["tris"],
    "suzanne": lambda: load_scene("suzanne")["tris"],
    "teapot": lambda: load_scene("teapot")["tris"],
    "sponza": lambda: sponza_scene()[0],
    "one_triangle": lambda: first_triangles(1),
    "two_triangles": lambda: first_triangles(2),
    "coincident_100": lambda: np.repeat(first_triangles(1), 100, 0),
}
BUILDERS = {"default": tm.BUILD_DEFAULT, "lbvh": tm.BUILD_LBVH}
INFO_KEYS = ("node_count", "leaf_count", "max_depth", "builder", "tri_count", "device_bytes")


def tris_of(name):
    return np.ascontiguousarray(SCENES[name](), np.float32)


def rays_of(name):
    return load_rays(name if name in ("cube", "suzanne", "teapot", "sponza") else "triangle")["rays"]


def create(tris, flags, hostloop, monkeypatch):
    """(scene, kernel launches of its creation), built with the level loops on the host or in cooperative launches."""
    if hostloop:
        monkeypatch.setenv("TMPT_BUILD_HOSTLOOP", "1")
    else:
        monkeypatch.delenv("TMPT_BUILD_HOSTLOOP", raising=False)
    before = tm.launch_count()
    s = tm.Scene(tris, flags=flags)
    return s, tm.launch_count() - before


def refit(s, tris):
    before = tm.launch_count()
    s.refit(tris)
    return tm.launch_count() - before


def answers(s, rays):
    """CLOSEST (ids, t, position, normal), ANY and SUN (ids): integers and float bits."""
    out = []
    for mode in (tm.HIT_CLOSEST, tm.HIT_ANY, tm.HIT_SUN):
        out += [a if a.dtype == np.int32 else bits(a) for a in s.HitScene(rays, mode=mode) if a is not None]
    return out


def assert_same_bounds(a, b):
    for k in ("bounds_min", "bounds_max"):
        assert (bits(a[k]) == bits(b[k])).all(), (k, a[k], b[k])


def assert_same_answers(a, b):
    assert len(a) == len(b)
    for k, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and (x == y).all(), k


@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("name", SCENES)
def test_host_loop_build_equals_cooperative_build(monkeypatch, name, builder):
    tris, rays = tris_of(name), rays_of(name)
    coop, coopLaunches = create(tris, BUILDERS[builder], False, monkeypatch)
    host, hostLaunches = create(tris, BUILDERS[builder], True, monkeypatch)
    with coop, host:
        a, b = coop.info(), host.info()
        for k in INFO_KEYS:
            assert a[k] == b[k], k
        assert_same_bounds(a, b)
        assert a["sah_cost"] == pytest.approx(b["sah_cost"], rel=1e-5)  # (sums of float atomics, in another order)
        assert_same_answers(answers(coop, rays), answers(host, rays))
    # the host loops launch once per level where the cooperative kernels launch once
    assert hostLaunches >= coopLaunches


@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("name", ["suzanne", "teapot", "two_triangles", "coincident_100"])
def test_refit_of_either_build_equals_a_fresh_scene(monkeypatch, name, builder):
    tris, rays = tris_of(name), rays_of(name)
    rng = np.random.default_rng(11)
    moved = (tris * np.float32(1.3) + rng.normal(0.0, 0.02, tris.shape).astype(np.float32)).astype(np.float32)
    refitLaunches = []
    for hostloop in (False, True):
        s, launches = create(tris, BUILDERS[builder], hostloop, monkeypatch)
        fresh, freshLaunches = create(tris, BUILDERS[builder], hostloop, monkeypatch)
        with s, fresh:
            assert launches == freshLaunches
            want, wantAnswers = fresh.info(), answers(fresh, rays)
            refitLaunches.append(refit(s, tris))  # to its own triangles
            assert_same_bounds(s.info(), want)
            assert_same_answers(answers(s, rays), wantAnswers)
            refitLaunches.append(refit(s, moved))
            refitLaunches.append(refit(s, tris))  # and back
            assert_same_bounds(s.info(), want)
            assert_same_answers(answers(s, rays), wantAnswers)
    assert len(set(refitLaunches)) == 1, refitLaunches
