#!/usr/bin/env python
"""What tmpt_denoise costs and buys, per bench.py scene at its workload resolution on one GPU:

    cost       device seconds of tmpt_denoise at the default parameters (5 iterations, sigmaLuminance 4, sigmaDepth 1,
               normalPowerLog2 7): TMPT_DEVICE (torch buffers) and TMPT_HOST (numpy buffers: the copies are inside the window),
               each warmed up, then the median over --steps calls, once with a 256 MB write between calls (flushes the 126 MB L2)
               and once without; beside it the tmpt_render time of the bench.py workload frame (same size, bench.py's spp)
    quality    RMSE of RGB in 8-bit codes against a 4096-spp uniform progressive session, for the noisy and the denoised frame of
               tmpt_render_outputs at 4 / 16 / 64 spp (guides from the same frame), and for an adaptive session (tolerance 1,
               minChunks 4, passes of 4 chunks until no pixel is active or 64 chunks) denoised with guides from an 8-spp frame:
               its rays against the uniform 64-spp frame's

Prints one JSON line per scene and a final one with the GPU name and power limit read in the same run; --out also writes it.

    python tools/bench_denoise.py [--scenes sponza,teapot,suzanne,cube] [--steps 20] [--warmup 3] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import toymeshpathtracer_b200 as tm  # noqa: E402
from bench_adaptive import error, scene_data, uniform_to  # noqa: E402
from bench_outputs import gpu_identity  # noqa: E402

WORKLOADS = {"sponza": (1920, 1080, 64), "teapot": (1280, 720, 16), "suzanne": (640, 360, 4), "cube": (640, 360, 4)}  # bench.py's
QUALITY_SPP = (4, 16, 64)


def median_ms(fn, steps, warmup, flush=None):
    import torch
    times = []
    for i in range(warmup + steps):
        if flush is not None:
            flush.zero_()
        torch.cuda.synchronize()
        sec = fn()
        if i >= warmup:
            times.append(sec * 1e3)
    return {"ms_median": float(np.median(times)), "ms_min": float(np.min(times)), "ms_max": float(np.max(times))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    if tm.device_count() < 1:
        raise SystemExit("bench_denoise: no CUDA device")
    import torch
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    results = []
    for name in args.scenes.split(","):
        w, h, wspp = WORKLOADS[name]
        sc = scene_data(name)
        cam = tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)
        row = {"scene": name, "width": w, "height": h}
        with tm.Scene(sc["tris"]) as s:
            # ---- cost
            frame = torch.zeros((h, w, 4), dtype=torch.uint8, device=dev)
            row["render"] = {"spp": wspp, **median_ms(lambda: s.render_device(cam, w, h, wspp, frame.data_ptr())[1], 5, 2, flush)}
            f, _, _ = s.render_outputs(cam, w, h, wspp, outputs=("radiance", "normal", "depth"))
            t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in f.items()}
            rgba = torch.zeros((h, w, 4), dtype=torch.uint8, device=dev)
            rad = torch.zeros((h, w, 4), dtype=torch.float32, device=dev)
            torch.cuda.synchronize()

            def on_device():
                return s.denoise_device(w, h, t["radiance"].data_ptr(), t["normal"].data_ptr(), t["depth"].data_ptr(), rgba.data_ptr(),
                                        rad.data_ptr())

            def on_host():
                return s.denoise(f["radiance"], f["normal"], f["depth"])[1]

            row["denoise"] = {"device_l2_flushed": median_ms(on_device, args.steps, args.warmup, flush),
                              "device_l2_warm": median_ms(on_device, args.steps, args.warmup),
                              "host_l2_flushed": median_ms(on_host, args.steps, args.warmup, flush),
                              "host_l2_warm": median_ms(on_host, args.steps, args.warmup)}
            row["denoise_vs_render_pct"] = 100.0 * row["denoise"]["device_l2_flushed"]["ms_median"] / row["render"]["ms_median"]
            # ---- quality
            ref = uniform_to(s, cam, w, h, [512])[512][2]
            row["quality"] = []
            for spp in QUALITY_SPP:
                q, rays, _ = s.render_outputs(cam, w, h, spp, outputs=("rgba", "radiance", "normal", "depth"))
                d, _ = s.denoise(q["radiance"], q["normal"], q["depth"])
                row["quality"].append({"spp": spp, "rays": rays, "noisy": error(q["rgba"], ref), "denoised": error(d["rgba"], ref)})
            g, grays, _ = s.render_outputs(cam, w, h, 8, outputs=("normal", "depth"))
            s.progressive_begin(w, h)
            arays, passes, active = 0, 0, -1
            while active != 0 and 4 * (passes + 1) <= 64:
                outs, r, _, active = s.progressive_pass_adaptive(cam, 4, 1.0, 4)
                arays, passes = arays + r, passes + 1
            d, _ = s.denoise(outs["radiance"], g["normal"], g["depth"])
            u64 = next(x for x in row["quality"] if x["spp"] == 64)
            row["adaptive"] = {"tolerance": 1.0, "min_chunks": 4, "passes": passes, "active_left": active, "rays": arays, "guide_rays": grays,
                               "mean_spp": float(outs["samples"].mean()), "rays_vs_uniform64": (arays + grays) / u64["rays"],
                               "noisy": error(outs["rgba"], ref), "denoised": error(d["rgba"], ref)}
            row["render_kernel"] = ["k_render", "k_render_paths"][s.render_kernel_choice()[0]]
        results.append(row)
        print(json.dumps({"scene": name, "denoise_ms": row["denoise"]["device_l2_flushed"]["ms_median"], "render_ms": row["render"]["ms_median"],
                          "rmse": {q["spp"]: (round(q["noisy"]["rmse_codes"], 3), round(q["denoised"]["rmse_codes"], 3)) for q in row["quality"]}}),
              flush=True)
    out = {"tool": "bench_denoise", **gpu_identity(), "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
           "params": {"iterations": 5, "sigmaLuminance": 4.0, "sigmaDepth": 1.0, "normalPowerLog2": 7},
           "reference": "uniform progressive session to 4096 spp", "ms": "device seconds reported by the call (events around kernels and copies)",
           "steps": args.steps, "warmup": args.warmup, "results": results}
    text = json.dumps(out)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
