"""tmpt_denoise on the GPU: bit for bit against the plain-C restatement (tests/denoise/oracle_denoise.c) on guides and radiance
from tmpt_render_outputs, including the 1920x1080 Sponza headline frame; host, device and in-place forms; the identity at 0
iterations; the adaptive workflow (8-spp guides, radiance from an adaptive session); NaN pixels; and the quality gate: at 16 spp
the denoised frame is closer to a 1024-spp frame than the noisy one on every bench.py scene."""
import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from conftest import load_scene, sponza_scene
from denoise_binding import DEFAULTS, DenoiseOracle

pytestmark = pytest.mark.gpu


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
def dn_oracle():
    return DenoiseOracle()


def rmse(a, b):
    d = a[..., :3].astype(np.float64) - b[..., :3].astype(np.float64)
    return float(np.sqrt((d * d).mean()))


def assert_matches(got, want):
    assert (got["rgba"] == want["rgba"]).all()
    assert same_bits(got["radiance"], want["radiance"])


@pytest.mark.parametrize("name", ["cube", "suzanne", "teapot"])
@pytest.mark.parametrize("w,h", [(160, 90), (7, 3)])
@pytest.mark.parametrize("spp", [1, 16])
def test_gpu_equals_the_oracle(dn_oracle, name, w, h, spp):
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        f, _, _ = s.render_outputs(cam, w, h, spp, outputs=("radiance", "normal", "depth"))
        for prm in (DEFAULTS, dict(iterations=1, sigma_luminance=4.0, sigma_depth=1.0, normal_power_log2=0),
                    dict(iterations=8, sigma_luminance=0.5, sigma_depth=3.0, normal_power_log2=8)):
            got, sec = s.denoise(f["radiance"], f["normal"], f["depth"], **prm)
            assert sec > 0
            assert_matches(got, dn_oracle.denoise(f["radiance"], f["normal"], f["depth"], **prm))


def test_sponza_headline_frame_equals_the_oracle(dn_oracle):
    w, h, spp = 1920, 1080, 64
    sc = scene_data("sponza")
    with tm.Scene(sc["tris"]) as s:
        f, _, _ = s.render_outputs(camera("sponza", w, h), w, h, spp, outputs=("rgba", "radiance", "normal", "depth"))
        got, sec = s.denoise(f["radiance"], f["normal"], f["depth"])
    want = dn_oracle.denoise(f["radiance"], f["normal"], f["depth"])
    assert_matches(got, want)
    print(f"sponza 1920x1080 64 spp: denoise {sec * 1e3:.3f} ms (host buffers, copies included)")


def test_host_device_and_in_place_forms_agree():
    """TMPT_HOST and TMPT_DEVICE (torch buffers, a non-default stream) give the same bytes; so do in-place and out-of-place
    radiance; two calls give the same bytes; the denoiser leaves the next frame of the scene unchanged."""
    import torch
    name, w, h, spp = "suzanne", 203, 61, 4
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        img0, _, _ = s.render(cam, w, h, spp)
        f, _, _ = s.render_outputs(cam, w, h, spp, outputs=("radiance", "normal", "depth"))
        host, _ = s.denoise(f["radiance"], f["normal"], f["depth"])
        again, _ = s.denoise(f["radiance"], f["normal"], f["depth"])
        assert (host["rgba"] == again["rgba"]).all() and (host["radiance"].view(np.uint32) == again["radiance"].view(np.uint32)).all()
        only_rgba, _ = s.denoise(f["radiance"], f["normal"], f["depth"], outputs=("rgba",))
        assert set(only_rgba) == {"rgba"} and (only_rgba["rgba"] == host["rgba"]).all()
        dev = torch.device("cuda", 0)
        stream = torch.cuda.Stream(dev)
        t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in f.items()}
        rgba = torch.zeros((h, w, 4), dtype=torch.uint8, device=dev)
        rad = torch.zeros((h, w, 4), dtype=torch.float32, device=dev)
        torch.cuda.synchronize(dev)
        sec = s.denoise_device(w, h, t["radiance"].data_ptr(), t["normal"].data_ptr(), t["depth"].data_ptr(), rgba.data_ptr(), rad.data_ptr(),
                               stream=stream.cuda_stream)
        stream.synchronize()
        assert sec > 0
        assert (rgba.cpu().numpy() == host["rgba"]).all()
        assert (rad.cpu().numpy().view(np.uint32) == host["radiance"].view(np.uint32)).all()
        inplace = t["radiance"].clone()
        torch.cuda.synchronize(dev)
        s.denoise_device(w, h, inplace.data_ptr(), t["normal"].data_ptr(), t["depth"].data_ptr(), 0, inplace.data_ptr(), stream=stream.cuda_stream)
        stream.synchronize()
        assert (inplace.cpu().numpy().view(np.uint32) == host["radiance"].view(np.uint32)).all()
        img1, _, _ = s.render(cam, w, h, spp)
        assert (img1 == img0).all()


@pytest.mark.parametrize("name,w,h,spp", [("cube", 160, 90, 16), ("teapot", 7, 3, 1), ("suzanne", 64, 36, 64)])
def test_zero_iterations_is_the_identity(name, w, h, spp):
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        img, _, _ = s.render(cam, w, h, spp)
        f, _, _ = s.render_outputs(cam, w, h, spp, outputs=("radiance", "normal", "depth"))
        got, _ = s.denoise(f["radiance"], f["normal"], f["depth"], iterations=0)
    assert same_bits(got["radiance"], f["radiance"]) and (got["rgba"] == img).all()


def test_adaptive_workflow_matches_the_oracle(dn_oracle):
    """Guides from an 8-spp tmpt_render_outputs, radiance from an adaptive session of the same camera and size."""
    name, w, h = "suzanne", 96, 54
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        g, _, _ = s.render_outputs(cam, w, h, 8, outputs=("normal", "depth"))
        s.progressive_begin(w, h)
        for _ in range(4):
            outs, _, _, active = s.progressive_pass_adaptive(cam, 4, 1.0, 4)
        assert len(np.unique(outs["samples"])) > 1  # the session really is adaptive
        got, _ = s.denoise(outs["radiance"], g["normal"], g["depth"])
    assert_matches(got, dn_oracle.denoise(outs["radiance"], g["normal"], g["depth"]))


def test_nan_pixels_match_the_oracle_and_come_out_finite(dn_oracle):
    name, w, h = "cube", 64, 40
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        f, _, _ = s.render_outputs(cam, w, h, 4, outputs=("radiance", "normal", "depth"))
        rad = f["radiance"].copy()
        rng = np.random.default_rng(11)
        mask = rng.random((h, w)) < 0.05
        rad[mask, rng.integers(0, 3)] = np.nan
        got, _ = s.denoise(rad, f["normal"], f["depth"])
    assert_matches(got, dn_oracle.denoise(rad, f["normal"], f["depth"]))
    assert mask.any() and np.isfinite(got["radiance"][mask]).all()


@pytest.mark.parametrize("name", ["sponza", "teapot", "suzanne", "cube"])
def test_quality_gate(name):
    """At 16 spp with the default parameters the denoised rgba is closer (RMSE of RGB in 8-bit codes) to a 1024-spp frame than
    the noisy rgba.  Only 'closer' is gated."""
    w, h = 320, 180
    sc = scene_data(name)
    cam = camera(name, w, h)
    with tm.Scene(sc["tris"]) as s:
        ref, _, _ = s.render(cam, w, h, 1024)
        f, _, _ = s.render_outputs(cam, w, h, 16, outputs=("rgba", "radiance", "normal", "depth"))
        got, _ = s.denoise(f["radiance"], f["normal"], f["depth"])
    noisy, denoised = rmse(f["rgba"], ref), rmse(got["rgba"], ref)
    print(f"{name} {w}x{h} 16 spp vs 1024 spp: RMSE noisy {noisy:.3f} codes, denoised {denoised:.3f} codes")
    assert denoised < noisy, (noisy, denoised)
