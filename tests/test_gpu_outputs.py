"""tmpt_render_outputs / tmpt_progressive_pass_outputs on the GPU: the linear radiance and the first-hit AOVs (normal, coverage,
depth, triangle) of a frame, bit for bit against the oracle's restatement, through both render kernels; the RGBA frame and the
ray count stay tmpt_render's."""
import os
import subprocess
import sys

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from aov_binding import AovOracle
from conftest import ROOT, load_scene, sponza_scene

pytestmark = pytest.mark.gpu

# the sizes of test_gpu_parity.py::test_frame_bit_exact_vs_oracle_pixel_mode (640x360: the 1024-thread configuration; 1x1; a frame
# smaller than one tile with a ragged last chunk; 128 chunks of 8 samples) plus a small Sponza frame (the closed hall)
CASES = [("cube", 160, 90, 4), ("suzanne", 128, 72, 3), ("teapot", 64, 36, 2), ("triangle", 33, 17, 5), ("cube", 70, 41, 20),
         ("suzanne", 48, 28, 9), ("cube", 640, 360, 8), ("cube", 640, 360, 4), ("suzanne", 640, 360, 4), ("triangle", 40, 24, 1024),
         ("cube", 1, 1, 1), ("cube", 7, 3, 33), ("sponza", 64, 36, 2)]
AOV_CASES = [("cube", 160, 90, 4), ("suzanne", 128, 72, 3), ("teapot", 64, 36, 2), ("cube", 70, 41, 20), ("cube", 7, 3, 33),
             ("triangle", 40, 24, 1024), ("sponza", 64, 36, 2)]
KERNELS = ("0", "1")  # TMPT_RENDER_PATHS: k_render, k_render_paths


def same_bits(a, b):
    """Float buffers equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload, and the GPU's is canonical)."""
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
def aov_oracle():
    return AovOracle()


@pytest.fixture(scope="module")
def probed(tmp_path_factory):
    """Every case rendered by tmpt_render and tmpt_render_outputs, once per forced render kernel (one process per kernel)."""
    runs = {}
    for k in KERNELS:
        d = tmp_path_factory.mktemp(f"paths{k}")
        env = dict(os.environ, TMPT_RENDER_PATHS=k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "outputs_probe.py"), str(d), *[":".join(map(str, c)) for c in CASES]],
                           env=env, capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stderr[-3000:]
        for c in CASES:
            name, w, h, spp = c
            runs[(k, c)] = dict(np.load(d / f"{name}_{w}x{h}x{spp}.npz"))
    return runs


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s_%dx%dx%d" % c)
def test_rgba_and_rays_are_tmpt_render_s_under_both_kernels(probed, case):
    for k in KERNELS:
        z = probed[(k, case)]
        assert int(z["kernel"]) == int(k)
        assert int(z["rays"]) == int(z["render_rays"]), k
        assert (z["rgba"] == z["render_rgba"]).all(), k
    assert (probed[("0", case)]["rgba"] == probed[("1", case)]["rgba"]).all()


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s_%dx%dx%d" % c)
def test_radiance_is_the_oracle_linear_mean(probed, oracle, case):
    """radiance = the oracle's linear mean bit for bit (NaN where it has NaN), A = 1; sqrt -> clamp -> *255 -> truncate of it
    (NaN -> 0) is the RGBA frame."""
    name, w, h, spp = case
    oimg, orays, lin = oracle.render(scene_data(name)["tris"], camera(name, w, h), w, h, spp, linear=True)
    for k in KERNELS:
        z = probed[(k, case)]
        assert int(z["rays"]) == orays and (z["rgba"] == oimg).all(), k
        assert same_bits(z["radiance"][..., :3], lin) and (z["radiance"][..., 3] == 1.0).all(), k
        with np.errstate(invalid="ignore"):
            q = np.minimum(np.maximum(np.sqrt(z["radiance"][..., :3]), np.float32(0)), np.float32(1)) * np.float32(255)
        q = np.where(np.isnan(q), 0, q).astype(np.uint8)
        assert (q == z["rgba"][..., :3]).all() and (z["rgba"][..., 3] == 255).all(), k


@pytest.mark.parametrize("case", AOV_CASES, ids=lambda c: "%s_%dx%dx%d" % c)
def test_aovs_equal_the_oracle(probed, aov_oracle, case):
    name, w, h, spp = case
    want, _ = aov_oracle.render_aov(scene_data(name)["tris"], camera(name, w, h), w, h, spp)
    for k in KERNELS:
        z = probed[(k, case)]
        assert (z["triangle"] == want["triangle"]).all(), k
        assert same_bits(z["normal"], want["normal"]), k
        assert same_bits(z["depth"], want["depth"]), k
    hit = want["triangle"] >= 0
    assert hit.any()


def test_band_boundaries_of_an_aov_frame(aov_oracle):
    """With AOVs the accumulation holds two plane sets, so a band has half the rows: 2000 x 3000 at 64 spp (32 chunks) is two
    bands of 2096 and 904 rows (one band without AOVs).  Rows either side of the boundary equal the oracle's; rgba and rays
    equal tmpt_render's."""
    name, w, h, spp = "cube", 2000, 3000, 64
    band = min(h, ((4 << 30) // (w * 32 * 2 * 16)) & ~3)
    assert band == 2096
    sc = load_scene(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        img, rays, _ = s.render(cam, w, h, spp)
        outs, orays, sec = s.render_outputs(cam, w, h, spp)
    assert orays == rays and (outs["rgba"] == img).all() and sec > 0
    for rows in ((0, 1), (band - 1, band + 1), (h - 1, h)):
        want, _ = aov_oracle.render_aov(sc["tris"], cam, w, h, spp, rows=rows)
        r0, r1 = rows
        for key in ("radiance", "normal", "depth"):
            assert same_bits(outs[key][r0:r1], want[key][r0:r1]), (rows, key)
        assert (outs["triangle"][r0:r1] == want["triangle"][r0:r1]).all() and (outs["rgba"][r0:r1] == want["rgba"][r0:r1]).all(), rows


@pytest.mark.parametrize("spp", [1, 6])
def test_device_form_and_subsets_give_the_same_buffers(spp):
    """Torch tensors on a non-default stream give the host form's buffers; any subset of the outputs gives the same values as the
    full set (radiance alone runs the plain kernels; triangle alone the AOV kernels without k_resolve at one chunk); a plain
    tmpt_render after AOV frames gives its old bytes."""
    import torch
    name, w, h = "suzanne", 203, 61
    sc = load_scene(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        before, rays0, _ = s.render(cam, w, h, spp)
        full, rays, _ = s.render_outputs(cam, w, h, spp)
        assert rays == rays0 and (full["rgba"] == before).all()
        for subset in (("radiance",), ("triangle",), ("depth", "rgba"), ("normal",)):
            part, prays, _ = s.render_outputs(cam, w, h, spp, outputs=subset)
            assert prays == rays and set(part) == set(subset)
            for key in subset:
                assert (part[key].view(np.uint8) == full[key].view(np.uint8)).all(), (subset, key)
        dev = torch.device("cuda", 0)
        stream = torch.cuda.Stream(dev)
        t = {"rgba": torch.zeros((h, w, 4), dtype=torch.uint8, device=dev), "radiance": torch.zeros((h, w, 4), dtype=torch.float32, device=dev),
             "normal": torch.zeros((h, w, 4), dtype=torch.float32, device=dev), "depth": torch.zeros((h, w), dtype=torch.float32, device=dev),
             "triangle": torch.zeros((h, w), dtype=torch.int32, device=dev)}
        torch.cuda.synchronize(dev)
        drays, _ = s.render_outputs_device(cam, w, h, spp, **{f"{k}_ptr": v.data_ptr() for k, v in t.items()}, stream=stream.cuda_stream)
        stream.synchronize()
        assert drays == rays
        for key, v in t.items():
            assert (v.cpu().numpy().view(np.uint8) == full[key].view(np.uint8)).all(), key
        after, rays2, _ = s.render(cam, w, h, spp)
        assert rays2 == rays0 and (after == before).all()


def test_progressive_radiance_converges_to_the_one_shot_radiance():
    """After passes totalling P >= 32 chunks the pass's radiance equals tmpt_render_outputs' at spp = 8 P bit for bit (and its
    rgba tmpt_render's); an AOV pointer on a pass is an argument error."""
    name, w, h = "suzanne", 85, 47
    sc = load_scene(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        want, want_rays, _ = s.render_outputs(cam, w, h, 272, outputs=("rgba", "radiance"))
        s.progressive_begin(w, h)
        total = 0
        for n in (1, 3, 12, 1, 17):  # 34 chunks = 272 samples
            got, rays, sec, spp = s.progressive_pass_outputs(cam, n)
            total += rays
            assert sec > 0 and set(got) == {"rgba", "radiance"} and (got["radiance"][..., 3] == 1.0).all()
        assert spp == 272 and total == want_rays
        assert (got["rgba"] == want["rgba"]).all() and same_bits(got["radiance"], want["radiance"])
        only, _, _, _ = s.progressive_pass_outputs(cam, 1, radiance=False)
        assert set(only) == {"rgba"}
        import ctypes as C
        rgba = np.zeros((h, w, 4), np.uint8)
        depth = np.zeros((h, w), np.float32)
        out = tm.Outputs(rgba=rgba.ctypes.data, depth=depth.ctypes.data)
        rc = tm.lib().tmpt_progressive_pass_outputs(s.handle, cam.ctypes.data, 1, tm.HOST, C.byref(out), None, None, None, None)
        assert rc == tm.TMPT_ERR_ARG and b"radiance only" in tm.lib().tmpt_last_error()
