"""Helper of tests/test_gpu_adaptive.py (TEST INFRASTRUCTURE): in a fresh process -- the render kernel is read from the environment
once per process (TMPT_RENDER_PATHS) -- run scripted progressive sessions and save every step's outputs as <out_dir>/<name>.npz.

    python tests/adaptive_probe.py <out_dir> <sessions.json>

sessions.json: [{"name", "scene", "w", "h", "steps": [[op, ...], ...]}, ...] with the ops
    ["begin"]                          tmpt_progressive_begin(w, h)
    ["a", nChunks, tolerance, minChunks]  an adaptive pass: rgba, radiance, samples, rays, active
    ["u", nChunks]                     a uniform pass (tmpt_progressive_pass_outputs): rgba, radiance, rays, samples so far
    ["r", spp]                         tmpt_render_outputs(rgba, radiance): rgba, radiance, rays
    ["ua", nChunks] / ["au", ...]      the pass of the other kind, expected to fail: its status and message
    ["until", nChunks, tolerance, minChunks, maxPasses]  adaptive passes until no pixel is active: per-pass rays / active, the
                                       last pass's outputs; "<i>_maxn" = the largest chunk count reached
    ["uto", i]                         a fresh uniform session to step i's maxn chunks (passes of at most 128): total rays
Step i's arrays are saved as "<i>_rgba", "<i>_radiance", ...; "kernel" is the render kernel of the last frame."""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import toymeshpathtracer_b200 as tm  # noqa: E402
from conftest import load_scene, sponza_scene  # noqa: E402

out_dir, spec = sys.argv[1], json.load(open(sys.argv[2]))
L = tm.lib()
L.tmpt_last_error.restype = C.c_char_p
scenes = {}
for sess in spec:
    name, w, h = sess["scene"], sess["w"], sess["h"]
    if name not in scenes:
        if name == "sponza":
            t, mn, mx = sponza_scene()
            sc = {"tris": t, "bounds_min": mn, "bounds_max": mx}
        else:
            sc = load_scene(name)
        scenes[name] = (sc, tm.Scene(sc["tris"]))
    sc, s = scenes[name]
    cam = tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)
    res = {}
    for i, step in enumerate(sess["steps"]):
        op = step[0]
        if op == "begin":
            s.progressive_begin(w, h)
        elif op == "a":
            outs, rays, sec, active = s.progressive_pass_adaptive(cam, step[1], step[2], step[3])
            res.update({f"{i}_{k}": v for k, v in outs.items()})
            res.update({f"{i}_rays": np.int64(rays), f"{i}_active": np.int64(active), f"{i}_seconds": np.float64(sec)})
        elif op == "u":
            outs, rays, sec, spp = s.progressive_pass_outputs(cam, step[1])
            res.update({f"{i}_{k}": v for k, v in outs.items()})
            res.update({f"{i}_rays": np.int64(rays), f"{i}_spp": np.int64(spp)})
        elif op == "r":
            outs, rays, _ = s.render_outputs(cam, w, h, step[1], ("rgba", "radiance"))
            res.update({f"{i}_{k}": v for k, v in outs.items()})
            res[f"{i}_rays"] = np.int64(rays)
        elif op == "until":
            rays, active = [], []
            while len(rays) < step[4] and (not active or active[-1] > 0):
                outs, r, _, a = s.progressive_pass_adaptive(cam, step[1], step[2], step[3])
                rays.append(r)
                active.append(a)
            res.update({f"{i}_{k}": v for k, v in outs.items()})
            res.update({f"{i}_rays": np.array(rays, np.int64), f"{i}_active": np.array(active, np.int64),
                        f"{i}_maxn": np.int64(outs["samples"].max() // 8)})
        elif op == "uto":
            s.progressive_begin(w, h)
            left, total = int(res[f"{step[1]}_maxn"]), 0
            while left > 0:
                _, r, _, _ = s.progressive_pass(cam, min(left, 128))
                total += r
                left -= min(left, 128)
            res[f"{i}_rays"] = np.int64(total)
        elif op in ("ua", "au"):
            camf = np.ascontiguousarray(cam, np.float32)
            rgba = np.zeros((h, w, 4), np.uint8)
            out = tm.Outputs(rgba=rgba.ctypes.data)
            if op == "ua":
                st = L.tmpt_progressive_pass_outputs(s._h, camf.ctypes.data, step[1], tm.HOST, C.byref(out), None, None, None, None)
            else:
                st = L.tmpt_progressive_pass_adaptive(s._h, camf.ctypes.data, step[1], C.byref(tm.Adaptive(step[2], step[3])), tm.HOST,
                                                      C.byref(out), None, None, None, None, None)
            res[f"{i}_status"] = np.int64(st)
            res[f"{i}_message"] = np.array(L.tmpt_last_error().decode())
    res["kernel"] = np.int64(s.render_kernel_choice()[0])
    np.savez(os.path.join(out_dir, f"{sess['name']}.npz"), **res)
for _, s in scenes.values():
    s.close()
