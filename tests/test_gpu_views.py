"""tmpt_render_views on the GPU: a batch of views in one call, each view byte for byte the single tmpt_render_outputs frame of its
camera, through both render kernels, across accumulation bands and the 2^16-row limit of k_render_paths' packed item words, with
far cameras in the batch, in the device form, and without disturbing the scene's other frames and sessions."""
import os
import subprocess
import sys

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from aov_binding import AovOracle
from conftest import ROOT
from views_probe import case_file, cameras, orbit_cameras, scene_data

pytestmark = pytest.mark.gpu

KERNELS = ("0", "1")  # TMPT_RENDER_PATHS: k_render, k_render_paths
BUDGET = 4 << 30      # the accumulation buffer's budget (kernels.cu: prepare_accum)
MAX_VIEW_BAND = 65536 - 4  # kernels.cu: kMaxViewBandRows
OUTPUTS = tm.OUTPUTS

# (scene, w, h, spp, views, kind): the sizes of test_gpu_outputs.py's cases, H % 4 != 0 (tiles straddle two views), 128 chunks,
# a one-pixel view, a view smaller than a tile with a ragged last chunk, the closed hall, a batch of one; duplicate cameras and
# lens radii that differ from view to view; near cameras and the camera 10^5 scene sizes away in one batch
CASES = [("cube", 160, 90, 4, 6, "orbit"), ("suzanne", 33, 17, 5, 7, "orbit"), ("triangle", 40, 24, 1024, 3, "orbit"),
         ("cube", 1, 1, 1, 5, "orbit"), ("cube", 7, 3, 33, 4, "orbit"), ("sponza", 64, 36, 2, 4, "orbit"), ("teapot", 64, 36, 2, 1, "orbit"),
         ("cube", 32, 18, 4, 4, "dup"), ("suzanne", 40, 24, 6, 3, "lens"), ("suzanne", 64, 36, 3, 4, "far")]
# accumulation bands: all outputs (two plane sets) of 256-pixel rows at 32 one-sample chunks are 16384-row bands; 6144-row views put
# the first two band boundaries inside views 2 and 5 and the third on the boundary of views 7 and 8
BANDS = ("triangle", 256, 6144, 32, 9, "orbit")
BANDS_CHECKED = (0, 2, 5, 7, 8)
# 700 views of 100 rows are 70000 stacked rows: more than k_render_paths' 16-bit band row, so two bands (the boundary inside view 655)
PACKED = ("cube", 8, 100, 2, 700, "orbit")
PACKED_CHECKED = (0, 654, 655, 656, 699)


def chunk_count(spp):
    n = min(max(spp // 32, 1), 8)  # integ::chunk_len
    return (spp + n - 1) // n


def band_rows(w, rows, spp, planes):
    """Stacked rows per band of a batch: kernels.cu prepare_accum with plan_render's views cap."""
    return min(rows, MAX_VIEW_BAND, max(4, (BUDGET // (w * chunk_count(spp) * planes * 16)) & ~3))


def spec(case, checked=None):
    s = ":".join(map(str, case))
    return s + ":" + "-".join(map(str, checked)) if checked else s


def run_probe(script, args, env_set, env_pop=(), timeout=1800):
    env = dict(os.environ, **env_set)
    for k in env_pop:
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", script), *args], env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]


def same_bits(a, b):
    """Float buffers equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload, and the GPU's is canonical)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return a.shape == b.shape and (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


def same_bytes(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and (a.view(np.uint8) == b.view(np.uint8)).all()


@pytest.fixture(scope="module")
def probed(tmp_path_factory):
    """Every case, the band case and the packed-word case, once per forced render kernel (one process per kernel)."""
    specs = [spec(c) for c in CASES] + [spec(BANDS, BANDS_CHECKED), spec(PACKED, PACKED_CHECKED)]
    runs = {}
    for k in KERNELS:
        d = tmp_path_factory.mktemp(f"views{k}")
        run_probe("views_probe.py", [str(d), *specs], {"TMPT_RENDER_PATHS": k}, ("TMPT_RENDER_CFG",))
        for c in CASES + [BANDS, PACKED]:
            runs[(k, c)] = dict(np.load(d / case_file(spec(c, BANDS_CHECKED if c == BANDS else PACKED_CHECKED if c == PACKED else None))))
    return runs


def check_views_equal_single_frames(probed, case, all_checked):
    for k in KERNELS:
        z = probed[(k, case)]
        assert int(z["kernel"]) == (0 if case[5] == "far" else int(k)), k
        for key in OUTPUTS:
            assert same_bytes(z["batch_" + key], z["single_" + key]), (k, key)
        if all_checked:
            assert int(z["rays"]) == int(z["single_rays"]), k
        else:
            assert int(z["rays"]) > int(z["single_rays"]), k
    for key in OUTPUTS:
        assert same_bytes(probed[("0", case)]["batch_" + key], probed[("1", case)]["batch_" + key]), key


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s_%dx%dx%d_%d_%s" % c)
def test_every_view_equals_its_single_frame_under_both_kernels(probed, case):
    """Every output of every view is tmpt_render_outputs' for that view's camera, byte for byte; the batch's ray count is the sum
    of the single frames'; both kernels give the same bytes."""
    check_views_equal_single_frames(probed, case, True)
    z = probed[("0", case)]
    if case[5] == "dup":
        for key in OUTPUTS:
            assert same_bytes(z["batch_" + key][0::2], z["batch_" + key][:1].repeat(len(z["checked"][0::2]), 0)), key
            assert same_bytes(z["batch_" + key][1::2], z["batch_" + key][1:2].repeat(len(z["checked"][1::2]), 0)), key
        assert not same_bytes(z["batch_rgba"][0], z["batch_rgba"][1])
    if case[5] == "lens":  # every view has its own lens radius
        cams = cameras("lens", scene_data(case[0]), *case[1:3], case[4])
        assert len(set(cams[:, 21].tolist())) == case[4]
    if case[5] == "far":
        assert (z["batch_triangle"][1] >= 0).mean() > 0.2  # the far camera's model fills part of its view


def test_views_on_either_side_of_band_boundaries(probed):
    """A batch whose accumulation exceeds the 4 GB budget: band boundaries inside views 2 and 5 and between views 7 and 8; those
    views, the first and the last equal their single frames under both kernels."""
    name, w, h, spp, n, _ = BANDS
    band = band_rows(w, n * h, spp, 2)
    bounds = list(range(band, n * h, band))
    assert band == 16384 and bounds == [16384, 32768, 49152]
    assert [b // h for b in bounds] == [2, 5, 8] and [b % h for b in bounds] == [4096, 2048, 0]
    check_views_equal_single_frames(probed, BANDS, False)


def test_views_past_the_packed_row_limit(probed):
    """70000 stacked rows: k_render_paths packs a band's row in 16 bits, so a batch's bands stop below 2^16 rows.  The first and the
    last view and the views around the band boundary equal their single frames under both kernels."""
    name, w, h, spp, n, _ = PACKED
    rows = n * h
    band = band_rows(w, rows, spp, 2)
    assert rows > 65536 and band == MAX_VIEW_BAND and (BUDGET // (w * chunk_count(spp) * 2 * 16)) > rows
    assert band // h == 655 and band % h == 32
    check_views_equal_single_frames(probed, PACKED, False)


def test_two_views_equal_the_oracle(oracle):
    """Two views of a batch against the oracle's restatements directly: rgba, rays and radiance (oracle.render), normal, depth and
    triangle (AovOracle)."""
    aov = AovOracle()
    name, w, h, spp = "suzanne", 48, 28, 9
    sc = scene_data(name)
    cams = orbit_cameras(sc, w, h, 2)
    with tm.Scene(sc["tris"]) as s:
        outs, rays, sec = s.render_views(cams, w, h, spp)
    assert sec > 0 and set(outs) == set(OUTPUTS) and outs["rgba"].shape == (2, h, w, 4) and outs["depth"].shape == (2, h, w)
    total = 0
    for v in range(2):
        oimg, orays, lin = oracle.render(sc["tris"], cams[v], w, h, spp, linear=True)
        want, _ = aov.render_aov(sc["tris"], cams[v], w, h, spp)
        total += orays
        assert (outs["rgba"][v] == oimg).all(), v
        lin4 = np.concatenate([lin, np.ones(lin.shape[:2] + (1,), np.float32)], axis=-1)
        assert same_bits(outs["radiance"][v], lin4), v
        assert (outs["triangle"][v] == want["triangle"]).all() and (want["triangle"] >= 0).any(), v
        assert same_bits(outs["normal"][v], want["normal"]) and same_bits(outs["depth"][v], want["depth"]), v
    assert rays == total


@pytest.mark.parametrize("spp", [1, 6])
def test_device_form_and_subsets_give_the_host_buffers(spp):
    """Torch tensors [N, H, W, ...] on a non-default stream give the host form's buffers; any subset of the outputs gives the full
    set's values (radiance alone: the plain kernels with a resolve; triangle alone: the AOV kernels)."""
    import torch
    name, w, h, n = "suzanne", 45, 26, 5
    sc = scene_data(name)
    cams = orbit_cameras(sc, w, h, n)
    with tm.Scene(sc["tris"]) as s:
        full, rays, _ = s.render_views(cams, w, h, spp)
        for subset in (("radiance",), ("triangle",), ("depth", "rgba"), ("normal",), ("rgba",)):
            part, prays, _ = s.render_views(cams, w, h, spp, outputs=subset)
            assert prays == rays and set(part) == set(subset)
            for key in subset:
                assert same_bytes(part[key], full[key]), (subset, key)
        dev = torch.device("cuda", 0)
        stream = torch.cuda.Stream(dev)
        t = {"rgba": torch.zeros((n, h, w, 4), dtype=torch.uint8, device=dev), "radiance": torch.zeros((n, h, w, 4), dtype=torch.float32, device=dev),
             "normal": torch.zeros((n, h, w, 4), dtype=torch.float32, device=dev), "depth": torch.zeros((n, h, w), dtype=torch.float32, device=dev),
             "triangle": torch.zeros((n, h, w), dtype=torch.int32, device=dev)}
        torch.cuda.synchronize(dev)
        drays, _ = s.render_views_device(cams, w, h, spp, **{f"{k}_ptr": v.data_ptr() for k, v in t.items()}, stream=stream.cuda_stream)
        stream.synchronize()
        assert drays == rays
        for key, v in t.items():
            assert same_bytes(v.cpu().numpy(), full[key]), key


def test_a_batch_leaves_frames_and_sessions_alone():
    """A tmpt_render after a batch gives its old bytes; a batch between two progressive passes leaves the session's result as it is
    without the batch."""
    name, w, h, spp = "cube", 61, 35, 4
    sc = scene_data(name)
    cams = orbit_cameras(sc, w, h, 3)
    cam = tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)
    with tm.Scene(sc["tris"]) as s:
        before, rays0, _ = s.render(cam, w, h, spp)
        s.render_views(cams, 2 * w, h, 64)  # (larger scratch, other chunk counts)
        after, rays1, _ = s.render(cam, w, h, spp)
        assert rays1 == rays0 and (after == before).all()
        s.progressive_begin(w, h)
        s.progressive_pass_outputs(cam, 2)
        want, _, _, _ = s.progressive_pass_outputs(cam, 3)
        s.progressive_begin(w, h)
        s.progressive_pass_outputs(cam, 2)
        s.render_views(cams, w, h, 16)
        got, _, _, spp_so_far = s.progressive_pass_outputs(cam, 3)
        assert spp_so_far == 40
        for key in want:
            assert same_bytes(got[key], want[key]), key
