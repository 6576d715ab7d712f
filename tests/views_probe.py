"""Helper of tests/test_gpu_views.py (TEST INFRASTRUCTURE): in a fresh process -- the render kernel is read from the environment once
per process (TMPT_RENDER_PATHS) -- render each case as one tmpt_render_views batch with every output and the checked views as
single tmpt_render_outputs frames, and save both, the ray counts and the kernel that ran as <out_dir>/<case>.npz.

    python tests/views_probe.py <out_dir> <scene>:<w>:<h>:<spp>:<views>:<kind>[:<checked views, dash-separated>] ...

kind: orbit (views around the scene), dup (two orbit cameras, each twice), lens (orbit views with growing lens radii), far (orbit
views with the far camera of test_gpu_render_edges.py B among them).  Without a list every view is checked.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import toymeshpathtracer_b200 as tm  # noqa: E402
from conftest import load_scene, sponza_scene  # noqa: E402


def scene_data(name):
    if name == "sponza":
        t, mn, mx = sponza_scene()
        return {"tris": t, "bounds_min": mn, "bounds_max": mx}
    return load_scene(name)


def orbit_cameras(sc, w, h, n, apertures=None):
    """n cameras on a circle around the scene's centre, 0.3 rad above it, looking at the centre."""
    mn, mx = sc["bounds_min"].astype(np.float64), sc["bounds_max"].astype(np.float64)
    centre, r = (mn + mx) / 2, float(np.linalg.norm(mx - mn)) / 2
    cams = []
    for v in range(n):
        a = 2 * np.pi * v / n
        frm = centre + 2.5 * r * np.array([np.sin(a) * np.cos(0.3), np.sin(0.3), np.cos(a) * np.cos(0.3)])
        ap = 0.0 if apertures is None else apertures[v]
        cams.append(tm.camera_make(frm, centre, [0, 1, 0], 45.0, w / h, ap, float(np.linalg.norm(frm - centre))))
    return np.stack(cams)


def far_camera(w, h):
    """test_gpu_render_edges.py B's camera: suzanne seen from 10^5 scene sizes away, 0.0012-degree field of view."""
    sc = load_scene("suzanne")
    mn, mx = sc["bounds_min"].astype(np.float64), sc["bounds_max"].astype(np.float64)
    centre, size = (mn + mx) / 2, float(np.abs(np.concatenate([mn, mx])).max())
    frm = centre + np.array([0.3, 0.5, 1.0]) / np.linalg.norm([0.3, 0.5, 1.0]) * 1.0e5 * size
    return tm.camera_make(frm, centre, [0, 1, 0], 0.0012, w / h, 0.03, float(np.linalg.norm(frm - centre)))


def cameras(kind, sc, w, h, n):
    if kind == "orbit":
        return orbit_cameras(sc, w, h, n)
    if kind == "dup":
        two = orbit_cameras(sc, w, h, 2)
        return np.stack([two[v % 2] for v in range(n)])
    if kind == "lens":
        r = float(np.linalg.norm(sc["bounds_max"] - sc["bounds_min"]))
        return orbit_cameras(sc, w, h, n, apertures=[0.4 * r * v / max(n - 1, 1) for v in range(n)])
    if kind == "far":
        cams = orbit_cameras(sc, w, h, n)
        cams[1::2] = far_camera(w, h)
        return cams
    raise ValueError(kind)


def case_file(case):
    return case.replace(":", "_") + ".npz"


if __name__ == "__main__":
    out_dir = sys.argv[1]
    scenes = {}
    for case in sys.argv[2:]:
        parts = case.split(":")
        name, kind = parts[0], parts[5]
        w, h, spp, n = map(int, parts[1:5])
        checked = [int(v) for v in parts[6].split("-")] if len(parts) > 6 else list(range(n))
        if name not in scenes:
            sc = scene_data(name)
            scenes[name] = (sc, tm.Scene(sc["tris"]))
        sc, s = scenes[name]
        cams = cameras(kind, sc, w, h, n)
        batch, rays, _ = s.render_views(cams, w, h, spp)
        kernel, _ = s.render_kernel_choice()
        out = {"rays": np.int64(rays), "kernel": np.int64(kernel), "checked": np.array(checked, np.int64)}
        single_rays = 0
        singles = {k: [] for k in batch}
        for v in checked:
            one, r, _ = s.render_outputs(cams[v], w, h, spp)
            single_rays += r
            for k in batch:
                singles[k].append(one[k])
        out["single_rays"] = np.int64(single_rays)
        for k in batch:
            out["batch_" + k] = batch[k][checked]
            out["single_" + k] = np.stack(singles[k])
        del batch
        np.savez(os.path.join(out_dir, case_file(case)), **out)
    for _, s in scenes.values():
        s.close()
