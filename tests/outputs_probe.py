"""Helper of tests/test_gpu_outputs.py (TEST INFRASTRUCTURE): in a fresh process -- the render kernel is read from the environment
once per process (TMPT_RENDER_PATHS) -- render each case with tmpt_render and with tmpt_render_outputs (every output), and save
both frames, both ray counts, the outputs and the kernel that ran as <out_dir>/<scene>_<w>x<h>x<spp>.npz.

    python tests/outputs_probe.py <out_dir> <scene>:<w>:<h>:<spp> ...
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import toymeshpathtracer_b200 as tm  # noqa: E402
from conftest import load_scene, sponza_scene  # noqa: E402

out_dir = sys.argv[1]
scenes = {}
for case in sys.argv[2:]:
    name, w, h, spp = case.split(":")
    w, h, spp = int(w), int(h), int(spp)
    if name not in scenes:
        if name == "sponza":
            t, mn, mx = sponza_scene()
            sc = {"tris": t, "bounds_min": mn, "bounds_max": mx}
        else:
            sc = load_scene(name)
        scenes[name] = (sc, tm.Scene(sc["tris"]))
    sc, s = scenes[name]
    cam = tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)
    img, rays, _ = s.render(cam, w, h, spp)
    outs, orays, _ = s.render_outputs(cam, w, h, spp)
    kernel, _ = s.render_kernel_choice()
    np.savez(os.path.join(out_dir, f"{name}_{w}x{h}x{spp}.npz"), render_rgba=img, render_rays=np.int64(rays), rays=np.int64(orays),
             kernel=np.int64(kernel), **outs)
for _, s in scenes.values():
    s.close()
