"""tmpt_progressive_pass_adaptive on the GPU, through both render kernels (TMPT_RENDER_PATHS=0 / 1 in a probe process): every pass of
multi-pass sessions bit for bit against the oracle's restatement (tests/adaptive/oracle_adaptive.c); each pixel equals the uniform
session's pixel after the same number of chunks (and tmpt_render_outputs from 32 chunks on); tolerance 0 is the uniform pass; the
active list split into several bands; determinism, session reset and kind mixing; fewer rays than a uniform session."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from adaptive_binding import AdaptiveOracle, State
from conftest import ROOT, load_scene, sponza_scene

pytestmark = pytest.mark.gpu
KERNELS = ("0", "1")  # TMPT_RENDER_PATHS: k_render, k_render_paths
ORACLE_STEPS = [["begin"], ["a", 2, 0.0, 2], ["a", 2, 1.0, 4], ["a", 3, 0.5, 4], ["a", 1, 2.0, 3], ["a", 2, 0.25, 5]]
ORACLE_CASES = [("cube", 160, 90), ("suzanne", 128, 72), ("teapot", 64, 36), ("cube", 7, 3)]
SPONZA_STEPS = [["begin"], ["a", 1, 0.5, 2], ["a", 1, 0.5, 2]]
PREFIX_STEPS = [["begin"]] + [["u", 1]] * 40 + [["begin"]] + [["a", 4, 1.0, 4]] * 10 + [["r", 256], ["r", 288], ["r", 320]]
TOL0_STEPS = [["begin"], ["a", 1, 0.0, 2], ["a", 3, 0.0, 2], ["a", 8, 0.0, 5], ["begin"], ["u", 1], ["u", 3], ["u", 8]]
# 0 begin, 1-2 adaptive, 3 a uniform pass (refused), 4 begin, 5 uniform, 6 an adaptive pass (refused), 7 begin, 8-9 = 1-2 again,
# 10 begin, 11 tolerance 0 (= step 5)
RESET_STEPS = [["begin"], ["a", 2, 0.5, 2], ["a", 2, 0.5, 2], ["ua", 1], ["begin"], ["u", 2], ["au", 1, 0.5, 2], ["begin"],
               ["a", 2, 0.5, 2], ["a", 2, 0.5, 2], ["begin"], ["a", 2, 0.0, 2]]
BAND_W, BAND_H, BAND_TOL = 2000, 3000, 0.05
BAND_STEPS = [["begin"], ["u", 128], ["begin"], ["a", 128, 0.0, 2], ["a", 128, BAND_TOL, 4]]
SAVE_STEPS = [["begin"], ["until", 4, 1.0, 4, 512], ["uto", 1]]
BAND_ENTRIES = (4 << 30) // (128 * 16)  # list entries per band of a 128-chunk pass (4 GB of float4 chunk sums)


def sessions():
    s = [{"name": f"oracle_{n}_{w}x{h}", "scene": n, "w": w, "h": h, "steps": ORACLE_STEPS} for n, w, h in ORACLE_CASES]
    s += [{"name": "oracle_sponza", "scene": "sponza", "w": 32, "h": 18, "steps": SPONZA_STEPS},
          {"name": "noprogress", "scene": "triangle", "w": 8, "h": 4, "steps": [["au", 1, 0.5, 2]]},
          {"name": "prefix", "scene": "cube", "w": 160, "h": 90, "steps": PREFIX_STEPS},
          {"name": "tol0", "scene": "suzanne", "w": 128, "h": 72, "steps": TOL0_STEPS},
          {"name": "reset", "scene": "cube", "w": 64, "h": 36, "steps": RESET_STEPS},
          {"name": "band", "scene": "cube", "w": BAND_W, "h": BAND_H, "steps": BAND_STEPS},
          {"name": "savings", "scene": "cube", "w": 320, "h": 180, "steps": SAVE_STEPS}]
    return s


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


def scene_data(name):
    if name == "sponza":
        t, mn, mx = sponza_scene()
        return {"tris": t, "bounds_min": mn, "bounds_max": mx}
    return load_scene(name)


def camera(name, w, h):
    sc = scene_data(name)
    return tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)


@pytest.fixture(scope="module")
def ad_oracle():
    return AdaptiveOracle()


@pytest.fixture(scope="module")
def probed(tmp_path_factory):
    """Every session run once per forced render kernel (one process per kernel)."""
    runs = {}
    spec = tmp_path_factory.mktemp("spec") / "sessions.json"
    spec.write_text(json.dumps(sessions()))
    for k in KERNELS:
        d = tmp_path_factory.mktemp(f"paths{k}")
        env = dict(os.environ, TMPT_RENDER_PATHS=k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "adaptive_probe.py"), str(d), str(spec)], env=env,
                           capture_output=True, text=True, timeout=1800)
        assert r.returncode == 0, r.stderr[-3000:]
        runs[k] = {s["name"]: dict(np.load(d / f"{s['name']}.npz")) for s in sessions()}
    return runs


def check_against_oracle(ad_oracle, res, name, w, h, steps, rows=None):
    sc = scene_data(name)
    cam = camera(name, w, h)
    state = State(w, h)
    r0, r1 = rows or (0, h)
    for i, step in enumerate(steps):
        if step[0] == "begin":
            continue
        want, rays, active = ad_oracle.pass_(sc["tris"], cam, state, step[1], step[2], step[3], rows=rows)
        assert (res[f"{i}_rgba"][r0:r1] == want["rgba"][r0:r1]).all(), i
        assert same_bits(res[f"{i}_radiance"][r0:r1], want["radiance"][r0:r1]), i
        assert (res[f"{i}_samples"][r0:r1] == want["samples"][r0:r1]).all(), i
        if rows is None:
            assert (int(res[f"{i}_rays"]), int(res[f"{i}_active"])) == (rays, active), i


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name,w,h", ORACLE_CASES)
def test_passes_equal_the_oracle(probed, ad_oracle, kernel, name, w, h):
    res = probed[kernel][f"oracle_{name}_{w}x{h}"]
    assert int(res["kernel"]) == int(kernel)
    check_against_oracle(ad_oracle, res, name, w, h, ORACLE_STEPS)
    assert len({int(res[f"{i}_active"]) for i in range(2, len(ORACLE_STEPS))}) > 1 or w * h < 32  # the tolerances matter


@pytest.mark.parametrize("kernel", KERNELS)
def test_sponza_passes_equal_the_oracle(probed, ad_oracle, kernel):
    res = probed[kernel]["oracle_sponza"]
    assert int(res["kernel"]) == int(kernel)
    check_against_oracle(ad_oracle, res, "sponza", 32, 18, SPONZA_STEPS)


@pytest.mark.parametrize("kernel", KERNELS)
def test_pixels_equal_the_uniform_session_at_their_chunk_count(probed, kernel):
    res = probed[kernel]["prefix"]
    last = len(PREFIX_STEPS) - 4  # the last adaptive pass
    for i in range(42, last + 1):
        n = res[f"{i}_samples"] // 8
        assert set(np.unique(n)) <= set(range(4, 41, 4)), np.unique(n)  # a stopped pixel stays stopped: prefix sums of the passes
        for c in np.unique(n):
            m = n == c
            assert (res[f"{i}_rgba"][m] == res[f"{c}_rgba"][m]).all(), (i, c)
            assert same_bits(res[f"{i}_radiance"][m], res[f"{c}_radiance"][m]), (i, c)
    n = res[f"{last}_samples"] // 8
    assert len(np.unique(n)) > 2 and (n >= 32).any()
    for j, c in zip(range(last + 1, last + 4), (32, 36, 40)):
        m = n == c
        assert (res[f"{last}_rgba"][m] == res[f"{j}_rgba"][m]).all(), c
        assert same_bits(res[f"{last}_radiance"][m], res[f"{j}_radiance"][m]), c


@pytest.mark.parametrize("kernel", KERNELS)
def test_tolerance_zero_is_the_uniform_pass(probed, kernel):
    res = probed[kernel]["tol0"]
    for a, u in ((1, 5), (2, 6), (3, 7)):
        assert (res[f"{a}_rgba"] == res[f"{u}_rgba"]).all() and same_bits(res[f"{a}_radiance"], res[f"{u}_radiance"])
        assert int(res[f"{a}_rays"]) == int(res[f"{u}_rays"]) and (res[f"{a}_samples"] == res[f"{u}_spp"]).all()
        assert int(res[f"{a}_active"]) == 128 * 72


@pytest.mark.parametrize("kernel", KERNELS)
def test_determinism_reset_and_session_kinds(probed, kernel):
    res = probed[kernel]["reset"]
    for a, b in ((1, 8), (2, 9)):
        for k in ("rgba", "radiance", "samples", "rays", "active"):
            assert (res[f"{a}_{k}"] == res[f"{b}_{k}"]).all(), k
    assert (res["5_rgba"] == res["11_rgba"]).all() and same_bits(res["5_radiance"], res["11_radiance"])
    assert int(res["5_rays"]) == int(res["11_rays"])
    assert int(res["3_status"]) == tm.TMPT_ERR_ARG and "adaptive" in str(res["3_message"])
    assert int(res["6_status"]) == tm.TMPT_ERR_ARG and "uniform" in str(res["6_message"])
    none = probed[kernel]["noprogress"]
    assert int(none["0_status"]) == tm.TMPT_ERR_ARG and "tmpt_progressive_begin first" in str(none["0_message"])


def tile_slots(w, h):
    """Each pixel's slot in the tile-ordered list: 8x4 tiles in row-major tile order, lane (x & 7) + 8 (y & 3)."""
    y, x = np.mgrid[0:h, 0:w]
    return (((y >> 2) * ((w + 7) // 8) + (x >> 3)) * 32 + (x & 7) + 8 * (y & 3))


@pytest.mark.parametrize("kernel", KERNELS)
def test_list_bands(probed, ad_oracle, kernel):
    res = probed[kernel]["band"]
    w, h = BAND_W, BAND_H
    assert (res["3_rgba"] == res["1_rgba"]).all() and same_bits(res["3_radiance"], res["1_radiance"])
    assert int(res["3_rays"]) == int(res["1_rays"])
    # pass 2's list: the pixels it traced, in tile order; the rows of the pixels on either side of every band boundary
    traced = res["4_samples"] > res["3_samples"]
    order = np.argsort(tile_slots(w, h)[traced])
    ys = np.nonzero(traced)[0][order]
    assert BAND_ENTRIES < len(ys) < w * h, len(ys)  # a partial list of more than one band
    rows = set()
    for b in range(BAND_ENTRIES, len(ys), BAND_ENTRIES):
        rows |= {int(ys[b - 1]), int(ys[b])}
    full = np.argsort(tile_slots(w, h).ravel())  # pass 1: every pixel
    for b in range(BAND_ENTRIES, w * h, BAND_ENTRIES):
        rows |= {int(full[b - 1] // w), int(full[b] // w)}
    steps = [s for i, s in enumerate(BAND_STEPS) if i >= 2]
    sub = {f"{i - 2}_{k}": res[f"{i}_{k}"] for i in (3, 4) for k in ("rgba", "radiance", "samples")}
    for r in sorted(rows):
        check_against_oracle(ad_oracle, sub, "cube", w, h, steps, rows=(r, r + 1))


@pytest.mark.parametrize("kernel", KERNELS)
def test_adaptive_session_traces_fewer_rays(probed, kernel):
    res = probed[kernel]["savings"]
    active = res["1_active"]
    assert active[-1] == 0 and len(active) < 512
    assert (np.diff(active) <= 0).all()  # fixed params: a stopped pixel stays stopped
    n = res["1_samples"] // 8
    assert n.min() == 4 and n.max() == int(res["1_maxn"]) > 4
    assert int(res["1_rays"].sum()) < int(res["2_rays"])
