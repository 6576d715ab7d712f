"""A scene's scratch buffers grow on demand and are reused at smaller sizes: one scene runs a sequence that makes every buffer grow
and then serve a smaller call (staged outputs in host and device memory, accumulation, progressive sums, adaptive state, denoiser
state, HitScene staging, the sun grid after a refit), and every result equals, byte for byte with the same ray count, the same
call on a freshly created scene.  Creating, exercising and destroying a scene twenty times works each time."""
import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from conftest import load_rays, load_scene

pytestmark = pytest.mark.gpu

NAME = "suzanne"
SCENE = load_scene(NAME)
OUTPUTS = ("rgba", "radiance", "normal", "depth", "triangle")


def camera(w, h):
    return tm.camera_for_scene(f"{NAME}.obj", SCENE["bounds_min"], SCENE["bounds_max"], w, h)


def rays(n):
    r = load_rays(NAME)["rays"]
    return np.ascontiguousarray(np.tile(r, (-(-n // len(r)), 1))[:n])


def moved_tris():
    rng = np.random.default_rng(7)
    t = SCENE["tris"].astype(np.float32)
    return (t * np.float32(1.3) + rng.normal(0.0, 0.02, t.shape).astype(np.float32)).astype(np.float32)


def outputs_host(w, h, spp):
    def run(s):
        arrays, nrays, _ = s.render_outputs(camera(w, h), w, h, spp, outputs=OUTPUTS)
        return arrays, nrays
    return run


def outputs_device(w, h, spp):
    def run(s):
        import torch
        dev = torch.device("cuda", 0)
        shapes = {"rgba": ((h, w, 4), torch.uint8), "radiance": ((h, w, 4), torch.float32), "normal": ((h, w, 4), torch.float32),
                  "depth": ((h, w), torch.float32), "triangle": ((h, w), torch.int32)}
        t = {k: torch.zeros(shape, dtype=dt, device=dev) for k, (shape, dt) in shapes.items()}
        torch.cuda.synchronize(dev)
        nrays, _ = s.render_outputs_device(camera(w, h), w, h, spp, **{f"{k}_ptr": v.data_ptr() for k, v in t.items()})
        return {k: v.cpu().numpy() for k, v in t.items()}, nrays
    return run


def uniform_session(w, h, passes):
    def run(s):
        s.progressive_begin(w, h)
        out = []
        for n in passes:
            arrays, nrays, _, spp = s.progressive_pass_outputs(camera(w, h), n)
            out.append((arrays, nrays, spp))
        return out
    return run


def adaptive_session(w, h, passes):
    def run(s):
        s.progressive_begin(w, h)
        out = []
        for n in passes:
            arrays, nrays, _, active = s.progressive_pass_adaptive(camera(w, h), n, tolerance=1.0, min_chunks=2)
            out.append((arrays, nrays, active))
        return out
    return run


def denoise(w, h):
    def run(s):
        f, nrays, _ = s.render_outputs(camera(w, h), w, h, 8, outputs=("radiance", "normal", "depth"))
        got, _ = s.denoise(f["radiance"], f["normal"], f["depth"])
        return f, nrays, got
    return run


def hit_scene(n):
    def run(s):
        return s.HitScene(rays(n))
    return run


def refit_then_frame(w, h, spp):
    def run(s):
        s.refit(moved_tris())
        rgba, nrays, _ = s.render(camera(w, h), w, h, spp)
        return rgba, nrays
    return run


# Each buffer first grows, then serves a smaller call.  The refit comes last: it moves the scene's geometry.
STEPS = [
    ("outputs host 160x90", outputs_host(160, 90, 16)),
    ("outputs host 640x360", outputs_host(640, 360, 16)),
    ("outputs host 7x3", outputs_host(7, 3, 16)),
    ("outputs device 160x90", outputs_device(160, 90, 16)),
    ("outputs device 640x360", outputs_device(640, 360, 16)),
    ("outputs device 7x3", outputs_device(7, 3, 16)),
    ("uniform session 200x120", uniform_session(200, 120, (1, 3, 2))),
    ("adaptive session 256x144", adaptive_session(256, 144, (2, 2, 4, 4))),
    ("adaptive session 64x36", adaptive_session(64, 36, (2, 3, 4))),
    ("denoise 320x180", denoise(320, 180)),
    ("denoise 100x50", denoise(100, 50)),
    ("HitScene 1k", hit_scene(1000)),
    ("HitScene 100k", hit_scene(100_000)),
    ("HitScene 10", hit_scene(10)),
    ("refit, then a frame", refit_then_frame(160, 90, 8)),
]


def same(a, b):
    """Equal structure, equal integers, and arrays equal byte for byte."""
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        return a is not None and b is not None and a.dtype == b.dtype and a.shape == b.shape and \
            np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return isinstance(b, (list, tuple)) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return a == b


def exercise(s):
    return [run(s) for _, run in STEPS]


def test_reused_buffers_give_a_fresh_scenes_results():
    with tm.Scene(SCENE["tris"]) as s:
        reused = exercise(s)
    for (label, run), got in zip(STEPS, reused):
        with tm.Scene(SCENE["tris"]) as fresh:
            want = run(fresh)
        assert same(got, want), label


def test_create_exercise_destroy_cycles():
    device_bytes = []
    for _ in range(20):
        with tm.Scene(SCENE["tris"]) as s:
            exercise(s)
            device_bytes.append(s.info()["device_bytes"])
    assert len(set(device_bytes)) == 1, device_bytes
