#!/usr/bin/env python
"""What the outputs of tmpt_render_outputs cost: every bench.py workload rendered three ways on one GPU --

    render        tmpt_render into a device frame (what bench.py's single-GPU frame does through tmpt_render_stripes)
    outputs_rgba  tmpt_render_outputs with the rgba pointer only
    outputs_all   tmpt_render_outputs with rgba, radiance, normal, depth and triangle

-- all into device buffers (torch tensors), timed the way bench.py times a frame: CUDA events around each frame, a 256 MB write
between frames to flush the 126 MB L2 (outside the events), warm-up frames first, then the variants alternated frame by frame
in one process.  Prints one JSON line (GPU name and power limit included); --out also writes it to a file.

    python tools/bench_outputs.py [--steps 10] [--warmup 2] [--variants render,outputs_rgba,outputs_all] [--root DIR] [--out FILE]

--root DIR times the package of another checkout (e.g. the parent commit, whose library has only `render`)."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = ("render", "outputs_rgba", "outputs_all")


def gpu_identity():
    """Name, power limit and maximum SM clock of GPU 0, read in the same run as the measurement."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown", "power_limit": "unknown", "error": str(e)}


def aov_kernel_resources(pkg_dir):
    """Registers and spill bytes of the render kernels, from the -Xptxas -v log the build leaves (build/ptxas.log)."""
    path = os.path.join(pkg_dir, "build", "ptxas.log")
    if not os.path.exists(path):
        return "not available (no build/ptxas.log)"
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1) if ("k_render" in m.group(1) or "k_resolve" in m.group(1)) else None
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and "spill_stores" not in out.get(cur, {}):
            out.setdefault(cur, {}).update(spill_stores=int(m.group(1)), spill_loads=int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out.setdefault(cur, {})["registers"] = int(m.group(1))
    names = subprocess.run(["c++filt"], input="\n".join(out), capture_output=True, text=True).stdout.split("\n")
    return {n: v for n, v in zip(names, out.values())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed frames per variant and workload")
    ap.add_argument("--warmup", type=int, default=2, help="untimed frames per variant and workload")
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--root", default=ROOT, help="checkout whose toymeshpathtracer_b200 is timed")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    root = os.path.abspath(args.root)
    sys.path.insert(0, root)
    sys.path.insert(1, ROOT)
    import numpy as np
    import torch

    import toymeshpathtracer_b200 as tm
    from bench import WORKLOADS, scene_label, scene_obj_path

    if not torch.cuda.is_available() or tm.device_count() == 0:
        raise SystemExit("bench_outputs.py: no CUDA device")
    variants = [v for v in args.variants.split(",") if v]
    if set(variants) - set(VARIANTS):
        raise SystemExit(f"bench_outputs.py: unknown variants {sorted(set(variants) - set(VARIANTS))}")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    results = []
    for wl in WORKLOADS:
        scene, w, h, spp = WORKLOADS[wl]
        path = scene_obj_path(scene)
        tris, mn, mx = tm.load_scene(path)
        cam = tm.camera_for_scene(path, mn, mx, w, h)
        s = tm.Scene(tris)
        bufs = {"rgba": torch.empty((h, w, 4), dtype=torch.uint8, device=dev), "radiance": torch.empty((h, w, 4), dtype=torch.float32, device=dev),
                "normal": torch.empty((h, w, 4), dtype=torch.float32, device=dev), "depth": torch.empty((h, w), dtype=torch.float32, device=dev),
                "triangle": torch.empty((h, w), dtype=torch.int32, device=dev)}
        ptrs = {f"{k}_ptr": v.data_ptr() for k, v in bufs.items()}

        def frame(v):
            if v == "render":
                return s.render_device(cam, w, h, spp, ptrs["rgba_ptr"], stream=stream.cuda_stream)[0]
            if v == "outputs_rgba":
                return s.render_outputs_device(cam, w, h, spp, rgba_ptr=ptrs["rgba_ptr"], stream=stream.cuda_stream)[0]
            return s.render_outputs_device(cam, w, h, spp, **ptrs, stream=stream.cuda_stream)[0]

        ms = {v: [] for v in variants}
        rays = {}
        for i in range(args.warmup + args.steps):
            for v in variants:  # alternated frame by frame
                with torch.cuda.stream(stream):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    rays[v] = frame(v)
                    e1.record(stream)
                stream.synchronize()
                if i >= args.warmup:
                    ms[v].append(e0.elapsed_time(e1))
        kernel, esc = s.render_kernel_choice()
        s.close()
        entry = {"workload": wl, "scene": scene_label(scene), "width": w, "height": h, "spp": spp,
                 "render_kernel": {0: "k_render", 1: "k_render_paths"}.get(kernel, "?"), "rays_per_frame": rays}
        for v in variants:
            a = np.array(ms[v])
            entry[v] = {"ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                        "spread_pct": float(100.0 * (a.max() - a.min()) / np.median(a)), "mrays_s": rays[v] / (float(np.median(a)) * 1e3)}
        for v in variants:
            if v != "render" and "render" in variants:
                entry[f"{v}_vs_render_pct"] = 100.0 * (entry[v]["ms_median"] / entry["render"]["ms_median"] - 1.0)
        results.append(entry)
        del bufs
    line = {"tool": "bench_outputs", "root": os.path.relpath(root, ROOT) if root != ROOT else ".", **gpu_identity(),
            "steps": args.steps, "warmup": args.warmup, "l2": "flushed between frames (256 MB write)", "buffers": "device (torch tensors)",
            "time": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), "results": results,
            "kernels": aov_kernel_resources(os.path.join(root, "toymeshpathtracer_b200"))}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
