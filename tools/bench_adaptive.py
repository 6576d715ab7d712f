#!/usr/bin/env python
"""What adaptive progressive passes (tmpt_progressive_pass_adaptive) buy and cost, per bench.py scene at its workload resolution on
one GPU:

    reference   a uniform progressive session to 4096 spp
    uniform     one uniform session, snapshots at 64 / 128 / 256 / 512 spp: rays, ms, RMSE against the reference in 8-bit codes
                (RGB), share of pixels more than 1 code off in some channel
    adaptive    tolerance 2 / 1 / 0.5 codes, minChunks 4, passes of 4 chunks until no pixel is active or a pixel has 512 spp:
                the same metrics plus the mean spp
    headline    the cheapest adaptive session whose RMSE is at most uniform-256's: its rays and ms against uniform-256's
    overhead    a tolerance-0 adaptive pass against tmpt_progressive_pass (4 chunks each, same frame), alternated pass by pass with
                a 256 MB write between passes to flush the 126 MB L2: what select, compaction and the LIST kernels cost

ms = the passes' own `seconds` (device time including the copies to host memory).  Prints one JSON line with the GPU name and
power limit read in the same run; --out also writes it to a file.

    python tools/bench_adaptive.py [--scenes sponza,teapot,suzanne,cube] [--overhead-steps 5] [--out FILE]"""
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
from bench_outputs import aov_kernel_resources, gpu_identity  # noqa: E402

SCENES = {"sponza": (1920, 1080), "teapot": (1280, 720), "suzanne": (640, 360), "cube": (640, 360)}  # bench.py's workload sizes
UNIFORM_SPP = (64, 128, 256, 512)
TOLERANCES = (2.0, 1.0, 0.5)


def scene_data(name):
    from conftest import load_scene, sponza_scene
    if name == "sponza":
        t, mn, mx = sponza_scene()
        return {"tris": t, "bounds_min": mn, "bounds_max": mx}
    return load_scene(name)


def error(img, ref):
    d = img[..., :3].astype(np.float64) - ref[..., :3].astype(np.float64)
    return {"rmse_codes": float(np.sqrt((d * d).mean())), "share_off_by_more_than_1": float((np.abs(d) > 1).any(-1).mean())}


def uniform_to(s, cam, w, h, stops):
    """One uniform session; (rays, ms, rgba) at each chunk count in `stops`."""
    s.progressive_begin(w, h)
    done, rays, sec, out = 0, 0, 0.0, {}
    for stop in stops:
        while done < stop:
            k = min(128, stop - done)
            img, r, t, _ = s.progressive_pass(cam, k)
            done, rays, sec = done + k, rays + r, sec + t
        out[stop] = (rays, sec * 1e3, img)
    return out


def adaptive_rgba_only(s, cam, w, h):
    """A tolerance-0 adaptive pass of 4 chunks with rgba only and no samples buffer: the same copies as tmpt_progressive_pass."""
    import ctypes as C
    rgba = np.zeros((h, w, 4), np.uint8)
    out = tm.Outputs(rgba=rgba.ctypes.data)
    camf = np.ascontiguousarray(cam, np.float32)
    rays, sec = C.c_uint64(0), C.c_double(0.0)
    st = tm.lib().tmpt_progressive_pass_adaptive(s._h, camf.ctypes.data, 4, C.byref(tm.Adaptive(0.0, 2)), tm.HOST, C.byref(out), None,
                                                 C.byref(rays), C.byref(sec), None, None)
    assert st == tm.TMPT_OK, st
    return rays.value, sec.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", default=",".join(SCENES))
    ap.add_argument("--overhead-steps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    if tm.device_count() < 1:
        raise SystemExit("bench_adaptive: no CUDA device")
    import torch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")  # > 126 MB L2
    results = []
    for name in args.scenes.split(","):
        w, h = SCENES[name]
        sc = scene_data(name)
        cam = tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)
        row = {"scene": name, "width": w, "height": h}
        with tm.Scene(sc["tris"]) as s, tm.Scene(sc["tris"]) as s2:
            ref = uniform_to(s, cam, w, h, [512])[512][2]
            uni = uniform_to(s, cam, w, h, [spp // 8 for spp in UNIFORM_SPP])
            row["uniform"] = [{"spp": 8 * c, "rays": r, "ms": ms, **error(img, ref)} for c, (r, ms, img) in uni.items()]
            row["adaptive"] = []
            for tol in TOLERANCES:
                s.progressive_begin(w, h)
                rays, ms, passes, active = 0, 0.0, 0, -1
                while active != 0 and 4 * (passes + 1) <= 64:
                    outs, r, t, active = s.progressive_pass_adaptive(cam, 4, tol, 4, radiance=False)
                    rays, ms, passes = rays + r, ms + t * 1e3, passes + 1
                row["adaptive"].append({"tolerance": tol, "min_chunks": 4, "passes": passes, "active_left": active, "rays": rays, "ms": ms,
                                        "mean_spp": float(outs["samples"].mean()), "max_spp": int(outs["samples"].max()),
                                        **error(outs["rgba"], ref)})
            u256 = next(u for u in row["uniform"] if u["spp"] == 256)
            match = [a for a in row["adaptive"] if a["rmse_codes"] <= u256["rmse_codes"]]
            best = min(match, key=lambda a: a["rays"]) if match else None
            row["headline"] = ({"tolerance": best["tolerance"], "rays": best["rays"], "ms": best["ms"], "uniform256_rays": u256["rays"],
                                "uniform256_ms": u256["ms"], "rays_vs_uniform256": best["rays"] / u256["rays"],
                                "ms_vs_uniform256": best["ms"] / u256["ms"]} if best else "no adaptive session reached uniform-256's RMSE")
            # overhead: tolerance 0 (every pixel traced) against the uniform pass, alternated
            s.progressive_begin(w, h)
            s2.progressive_begin(w, h)
            t_uni, t_ad = [], []
            for i in range(args.overhead_steps + 1):
                flush.zero_()
                torch.cuda.synchronize()
                _, ru, tu, _ = s.progressive_pass(cam, 4)
                flush.zero_()
                torch.cuda.synchronize()
                ra, ta = adaptive_rgba_only(s2, cam, w, h)
                assert ra == ru
                if i:  # (the first pair is the warm-up)
                    t_uni.append(tu * 1e3)
                    t_ad.append(ta * 1e3)
            row["overhead"] = {"chunks_per_pass": 4, "uniform_ms_median": float(np.median(t_uni)), "adaptive_tol0_ms_median": float(np.median(t_ad)),
                               "overhead_pct": 100.0 * (np.median(t_ad) / np.median(t_uni) - 1.0), "uniform_ms": t_uni, "adaptive_tol0_ms": t_ad}
            row["render_kernel"] = ["k_render", "k_render_paths"][s.render_kernel_choice()[0]]
        results.append(row)
        print(json.dumps({"scene": name, "headline": row["headline"], "overhead_pct": row["overhead"]["overhead_pct"]}), flush=True)
    out = {"tool": "bench_adaptive", **gpu_identity(), "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
           "reference": "uniform progressive session to 4096 spp", "ms": "sum of the passes' device seconds, copies to host included",
           "results": results, "kernels": aov_kernel_resources(os.path.join(ROOT, "toymeshpathtracer_b200"))}
    text = json.dumps(out)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
