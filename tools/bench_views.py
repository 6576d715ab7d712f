#!/usr/bin/env python
"""What a batch of views saves: N views of one scene rendered on one GPU as

    loop_rgba   N tmpt_render_outputs calls (rgba only), each into its slice of a view-major device buffer
    batch_rgba  one tmpt_render_views call (rgba only) into the same buffer
    loop_all    N tmpt_render_outputs calls with rgba, radiance, normal, depth and triangle
    batch_all   one tmpt_render_views call with every output

-- all into device buffers (torch tensors), timed the way tools/bench_outputs.py times a frame: CUDA events around each
repetition (the N calls, or the one call), a 256 MB write between repetitions to flush the 126 MB L2 (outside the events),
warm-up repetitions first, then the variants alternated repetition by repetition in one process.  After the timed repetitions
the loop's and the batch's buffers are compared byte for byte.  Prints one JSON line (GPU name and power limit included);
--out also writes it to a file.

    python tools/bench_views.py [--steps 10] [--warmup 2] [--workloads a,b] [--out FILE]

The workloads: many small views (orbits for datasets), the six faces of a cube map, and a control whose single view already
fills the GPU."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.bench_outputs import gpu_identity  # noqa: E402

VARIANTS = ("loop_rgba", "batch_rgba", "loop_all", "batch_all")
# name: (scene, views, width, height, spp, camera set)
WORKLOADS = {
    "teapot_64x256x256_16spp": ("teapot", 64, 256, 256, 16, "orbit"),
    "sponza_cubemap_6x512x512_16spp": ("sponza", 6, 512, 512, 16, "cubemap"),
    "suzanne_256x64x64_64spp": ("suzanne", 256, 64, 64, 64, "orbit"),
    "cube_8x640x360_4spp": ("cube", 8, 640, 360, 4, "orbit"),
}
PIXEL_BYTES = {"rgba": 4, "radiance": 16, "normal": 16, "depth": 4, "triangle": 4}


def orbit(tm, np, mn, mx, n, w, h):
    """n cameras on a circle around the scene's centre, 0.3 rad above it."""
    mn, mx = np.asarray(mn, np.float64), np.asarray(mx, np.float64)
    centre, r = (mn + mx) / 2, float(np.linalg.norm(mx - mn)) / 2
    cams = []
    for v in range(n):
        a = 2 * np.pi * v / n
        frm = centre + 2.5 * r * np.array([np.sin(a) * np.cos(0.3), np.sin(0.3), np.cos(a) * np.cos(0.3)])
        cams.append(tm.camera_make(frm, centre, [0, 1, 0], 45.0, w / h, 0.0, float(np.linalg.norm(frm - centre))))
    return np.stack(cams)


def cubemap(tm, np, eye):
    """The six 90-degree faces seen from `eye`: +x, -x, +y, -y, +z, -z."""
    faces = [([1, 0, 0], [0, 1, 0]), ([-1, 0, 0], [0, 1, 0]), ([0, 1, 0], [0, 0, -1]), ([0, -1, 0], [0, 0, 1]), ([0, 0, 1], [0, 1, 0]),
             ([0, 0, -1], [0, 1, 0])]
    eye = np.asarray(eye, np.float64)
    return np.stack([tm.camera_make(eye, eye + np.array(d, np.float64), up, 90.0, 1.0, 0.0, 1.0) for d, up in faces])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed repetitions per variant and workload")
    ap.add_argument("--warmup", type=int, default=2, help="untimed repetitions per variant and workload")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import numpy as np
    import torch

    import toymeshpathtracer_b200 as tm
    from bench import scene_label, scene_obj_path

    if not torch.cuda.is_available() or tm.device_count() == 0:
        raise SystemExit("bench_views.py: no CUDA device")
    names = [x for x in args.workloads.split(",") if x]
    if set(names) - set(WORKLOADS):
        raise SystemExit(f"bench_views.py: unknown workloads {sorted(set(names) - set(WORKLOADS))}")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    results = []
    for wl in names:
        scene, n, w, h, spp, kind = WORKLOADS[wl]
        path = scene_obj_path(scene)
        tris, mn, mx = tm.load_scene(path)
        if kind == "cubemap":  # the eye of the scene's own camera (main.cpp's placement)
            cams = cubemap(tm, np, tm.camera_for_scene(path, mn, mx, w, h)[:3])
        else:
            cams = orbit(tm, np, mn, mx, n, w, h)
        s = tm.Scene(tris)
        shapes = {"rgba": ((4,), torch.uint8), "radiance": ((4,), torch.float32), "normal": ((4,), torch.float32), "depth": ((), torch.float32),
                  "triangle": ((), torch.int32)}
        bufs = {f"{v}_{k}": torch.empty((n, h, w) + sh, dtype=dt, device=dev) for v in ("loop", "batch") for k, (sh, dt) in shapes.items()}

        def ptrs(side, outputs, view=None):
            off = 0 if view is None else view * w * h
            return {f"{k}_ptr": bufs[f"{side}_{k}"].data_ptr() + off * PIXEL_BYTES[k] for k in outputs}

        def rep(v):
            side, which = v.split("_")
            outputs = ("rgba",) if which == "rgba" else tm.OUTPUTS
            if side == "batch":
                return s.render_views_device(cams, w, h, spp, **ptrs("batch", outputs), stream=stream.cuda_stream)[0]
            return sum(s.render_outputs_device(cams[i], w, h, spp, **ptrs("loop", outputs, i), stream=stream.cuda_stream)[0] for i in range(n))

        variants = list(VARIANTS)
        ms = {v: [] for v in variants}
        rays = {}
        for i in range(args.warmup + args.steps):
            for v in variants:  # alternated repetition by repetition
                with torch.cuda.stream(stream):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    rays[v] = rep(v)
                    e1.record(stream)
                stream.synchronize()
                if i >= args.warmup:
                    ms[v].append(e0.elapsed_time(e1))
        identical = all(torch.equal(bufs[f"loop_{k}"].view(torch.uint8), bufs[f"batch_{k}"].view(torch.uint8)) for k in tm.OUTPUTS)
        kernel, _ = s.render_kernel_choice()
        s.close()
        entry = {"workload": wl, "scene": scene_label(scene), "views": n, "width": w, "height": h, "spp": spp, "cameras": kind,
                 "render_kernel": {0: "k_render", 1: "k_render_paths"}.get(kernel, "?"), "rays": rays, "loop_equals_batch": identical}
        for v in variants:
            a = np.array(ms[v])
            entry[v] = {"ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                        "spread_pct": float(100.0 * (a.max() - a.min()) / np.median(a)), "mrays_s": rays[v] / (float(np.median(a)) * 1e3)}
        for which in ("rgba", "all"):
            entry[f"speedup_{which}"] = entry[f"loop_{which}"]["ms_median"] / entry[f"batch_{which}"]["ms_median"]
        results.append(entry)
        del bufs
    line = {"tool": "bench_views", **gpu_identity(), "steps": args.steps, "warmup": args.warmup, "l2": "flushed between repetitions (256 MB write)",
            "buffers": "device (torch tensors), view-major [N, H, W, ...]", "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
            "results": results}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
