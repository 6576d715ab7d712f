#!/usr/bin/env python
"""bench.py -- Mrays/s of the Trace() hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME]

One "step" = one frame of the workload: sponza stand-in (66 452 triangles, tools/gen_sponza.py;
the reference's own data/sponza.obj is absent from this environment) at 1920x1080, 64 spp --
the configuration BASELINE.json's metric is quoted on.  A ray is one HitScene-equivalent query
(primary + bounce + shadow), counted exactly like main.cpp:57, 91.

  value        whole-job Mrays/s, frame left in HBM on rank 0 (device time, max over ranks)
  e2e          the same through the C-ABI call a user makes (tmpt_render, HOST buffers): the
               frame's device->host copy is inside the timed region
  roofline     FP32-issue roofline of the path-tracing kernel (SURVEY.md 8(d): the path is
               L2-resident tree traversal, neither HBM- nor tensor-bound), with the measured
               box/triangle tests per ray from an instrumented pass, plus HBM context
  cpu_baseline the reference's own CPU program (oracle/_ref/TrimeshTracer), all host threads,
               on a bounded sample of the same workload

`--impl reference` times only the reference's CPU implementation and prints the same line.
Under torchrun (N > 1) there is one rank per GPU; rows are dealt out in stripes (multigpu.py).
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene, width, height, spp)
    "sponza_1080p_64spp": ("sponza", 1920, 1080, 64),
    "sponza_640x360_4spp": ("sponza", 640, 360, 4),
    "teapot_720p_16spp": ("teapot", 1280, 720, 16),
    "suzanne_640x360_4spp": ("suzanne", 640, 360, 4),
    "cube_640x360_4spp": ("cube", 640, 360, 4),
}
# bounded CPU samples (about 10-30 s of CPU work on the box's host cores): same scene and camera, fewer pixels / samples
CPU_SAMPLE = {"sponza": (640, 360, 8), "teapot": (640, 360, 8), "suzanne": (640, 360, 16), "cube": (640, 360, 64)}
CPU_SAMPLE_1T = {"sponza": (160, 90, 8), "teapot": (160, 90, 8), "suzanne": (320, 180, 8), "cube": (640, 360, 8)}  # one thread: a few seconds
# BASELINE.json configs 1-4 (config 5 is the headline line itself): reported in the line's "configs" array
EXTRA_CONFIGS = [("config1", "cube_640x360_4spp"), ("config2", "suzanne_640x360_4spp"), ("config3", "teapot_720p_16spp"),
                 ("config4", "sponza_640x360_4spp")]
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "TrimeshTracer")


# ------------------------------------------------------------------------------------------
# workload files
# ------------------------------------------------------------------------------------------
def scene_obj_path(scene: str) -> str:
    """An .obj file for `scene` in a scratch directory (the CLI and the reference binary take files)."""
    if scene == "sponza" and _real_sponza():
        return _real_sponza()  # the reference's own data/sponza.obj, when the caller has it: takes precedence over the stand-in
    d = os.path.join(tempfile.gettempdir(), "tmpt_bench_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"{scene}.obj")
    if os.path.exists(path):
        return path
    if scene == "sponza":
        from tools.gen_sponza import write_obj
        write_obj(path)
        return path
    z = np.load(os.path.join(ROOT, "tests", "golden", "scenes", f"{scene}.npz"))
    tris = z["tris"][:-2]  # LoadScene adds the floor itself
    tmp = path + ".tmp%d" % os.getpid()
    with open(tmp, "w") as f:
        f.writelines("v %.9g %.9g %.9g\n" % tuple(float(x) for x in v) for v in tris.reshape(-1, 3))
        f.writelines("f %d %d %d\n" % (3 * i + 1, 3 * i + 2, 3 * i + 3) for i in range(tris.shape[0]))
    os.replace(tmp, path)
    return path


def _real_sponza():
    real = os.environ.get("TMPT_SPONZA_OBJ")
    return real if real and os.path.exists(real) else None


def scene_label(scene: str) -> str:
    if scene == "sponza":
        return "sponza.obj (real)" if _real_sponza() else "sponza stand-in (tools/gen_sponza.py, 66452 tris)"
    return f"{scene}.obj"


# ------------------------------------------------------------------------------------------
# the reference's CPU program on a bounded sample
# ------------------------------------------------------------------------------------------
def run_reference_cpu(scene: str, w: int, h: int, spp: int, threads: int | None = None):
    """-> (Mrays/s, rays, seconds, kind, cores).  oracle/_ref when built, else the C restatement.  `threads`: worker threads
    of the reference's row loop (TBB_SHIM_THREADS of oracle/tbb_shim); default = every hardware thread."""
    cores = threads or os.cpu_count() or 1
    path = scene_obj_path(scene)
    if os.path.exists(REF_BIN):
        env = dict(os.environ, TBB_SHIM_THREADS=str(threads)) if threads else None
        with tempfile.TemporaryDirectory() as td:
            out = subprocess.run([REF_BIN, str(w), str(h), str(spp), path], cwd=td, capture_output=True, text=True, check=True, env=env).stdout
        m = re.search(r"in ([0-9.]+) s\n- ([0-9.]+) K Rays, ([0-9.]+) K Rays/s", out)
        sec, krays, krate = float(m.group(1)), float(m.group(2)), float(m.group(3))
        return krate / 1000.0, krays * 1000.0, sec, "reference", cores
    # fallback: the plain-C restatement (brute force over triangles -> tiny sample)
    from oracle.pyoracle import RNG_ROW, TRIG_LIBM, Oracle
    import toymeshpathtracer_b200 as tm
    tris, mn, mx = tm.load_scene(path)
    cam = tm.camera_for_scene(path, mn, mx, w, h)
    orc = Oracle()
    rows = (0, max(1, h // 16))
    t0 = time.perf_counter()
    _, rays = orc.render(tris, cam, w, h, 1, RNG_ROW, TRIG_LIBM, rows=rows, threads=threads)
    sec = time.perf_counter() - t0
    return rays / sec / 1e6, rays, sec, "port", threads or orc.threads


# ------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, throttle reasons and power of one GPU, sampled while the timed region runs: NVML from a thread every
    5 ms (an 8-GPU frame takes 60 ms: an nvidia-smi child process does not deliver a sample that fast), nvidia-smi -lms
    as the fallback when NVML is unavailable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, gpu_index: int):
        self.samples, self.proc, self.thread, self.idx = [], None, None, gpu_index
        self.stop = threading.Event()
        self.nvml = None

    def _nvml_loop(self):
        nv, h = self.nvml
        bits = []
        for name, label in (("nvmlClocksEventReasonHwSlowdown", "hw_slowdown"), ("nvmlClocksEventReasonHwThermalSlowdown", "hw_thermal_slowdown"),
                            ("nvmlClocksEventReasonSwThermalSlowdown", "sw_thermal_slowdown"), ("nvmlClocksEventReasonSwPowerCap", "sw_power_cap")):
            bit = getattr(nv, name, None) or getattr(nv, name.replace("ClocksEventReason", "ClocksThrottleReason"), None)
            bits.append((bit, label))
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while not self.stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = reasons_fn(h)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                flags = ["Active" if (bit and (r & bit)) else "Not Active" for bit, _ in bits]
                self.samples.append([str(sm), str(mx) if mx else "", *flags, "%.2f" % pw])
            except Exception:
                pass
            self.stop.wait(0.005)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nvml = (nv, nv.nvmlDeviceGetHandleByIndex(self.idx))
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        self.stop.set()
        if self.nvml and self.thread:
            self.thread.join(1.0)
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for s in self.samples if len(s) >= 6 for k in range(4) if s[2 + k].lower().startswith("active")})
        pw = [float(s[6]) for s in self.samples if len(s) > 6 and re.match(r"^[0-9.]+$", s[6])]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}



def _kernel_name(sc):
    """The render kernel the scene's last frame ran (chosen per frame by a probe: kernels.cu choose_render_kernel)."""
    k, esc = sc.render_kernel_choice()
    return {"kernel": {0: "k_render", 1: "k_render_paths"}.get(k, "?"), "probe_escape_fraction": round(esc, 4)}


def measure_extra_configs(tm, multigpu, dist, torch, sc_sponza, dev, stream, rank, world, local_rank, flush, peer_enabled):
    """BASELINE.json configs 1-4 as a `configs` array: Mrays/s and ms/frame of each small workload, timed like the headline
    (CUDA events around one frame, L2 flushed before each, 3 warm-up + 5 timed frames, max over ranks).  Configs 1-3 name one
    GPU: they are measured at N = 1 only; config 4 (sponza 640x360 4 spp, "at 1/2/4/8 GPUs") at every N."""
    out = []
    for label, wl in EXTRA_CONFIGS:
        scene, w, h, spp = WORKLOADS[wl]
        if scene != "sponza" and world > 1:
            continue
        peer = None
        if scene == "sponza":
            sc, path = sc_sponza, None
            tris = None
        else:
            path = scene_obj_path(scene)
            tris, mn, mx = tm.load_scene(path)
            sc = tm.Scene(tris, device=local_rank)
        if scene == "sponza":
            path = scene_obj_path(scene) if rank == 0 else None
            if world > 1:
                box = [path]
                dist.broadcast_object_list(box, src=0)
                path = box[0]
            _, mn, mx = tm.load_scene(path)
        cam = tm.camera_for_scene(path, mn, mx, w, h)
        if world > 1 and peer_enabled:
            peer = multigpu.PeerFrame(w, h, rank, world, local_rank)
        ms_list, rays_list = [], []
        for i in range(3 + 5):
            if world > 1:
                dist.barrier()
            with torch.cuda.stream(stream):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                _, rays = multigpu.render_frame(sc, cam, w, h, spp, rank, world, group=None, device=dev, peer=peer)
                e1.record(stream)
            stream.synchronize()
            if i >= 3:
                ms_list.append(e0.elapsed_time(e1))
                rays_list.append(int(rays.item()))
        t = torch.tensor([sum(ms_list)], dtype=torch.float64, device=dev)
        r = torch.tensor([sum(rays_list)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(r, op=dist.ReduceOp.SUM)
        out.append({"config": label, "workload": f"{scene_label(scene)} {w}x{h} {spp}spp", "n_gpus": world,
                    "value": int(r.item()) / (float(t.item()) * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": float(t.item()) / 5,
                    "rays_per_frame": int(r.item()) // 5, "frames": 5, "render_kernel": _kernel_name(sc)})
        if peer is not None:
            dist.barrier()
            peer.close()
        if scene != "sponza":
            sc.close()
    return out


def measure_hit_scene(tm, torch, sc, cam, w, h, dev):
    """Throughput of the batched HitScene entry (K2 closest hit, K3 any hit) on the rays the headline frame shoots: the camera's
    primary rays (one per pixel), the diffuse bounce rays leaving their hit points and the shadow rays towards the sun, all
    generated on the device.  Kernel time only (device pointers, CUDA events, best of 3)."""
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    camt = torch.tensor(cam, device=dev)
    ys, xs = torch.meshgrid(torch.arange(h, device=dev), torch.arange(w, device=dev), indexing="ij")
    u = ((xs + torch.rand((h, w), device=dev, generator=g)) / w).reshape(-1, 1)
    v = ((ys + torch.rand((h, w), device=dev, generator=g)) / h).reshape(-1, 1)
    origin, llc, hor, ver = camt[0:3], camt[3:6], camt[6:9], camt[9:12]
    d = llc + u * hor + v * ver - origin
    d = d / d.norm(dim=1, keepdim=True)
    rays = torch.cat([origin.expand_as(d), d], 1).contiguous().float()
    light = torch.tensor([-0.7, 1.0, 0.5], device=dev)
    light = light / light.norm()
    st = torch.cuda.Stream(dev)

    def timed(r6, mode):
        n = r6.shape[0]
        ids = torch.empty(n, dtype=torch.int32, device=dev)
        t = torch.empty(n, device=dev)
        pos = torch.empty((n, 3), device=dev)
        nrm = torch.empty((n, 3), device=dev)
        best = 1e30
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(st):
            for _ in range(4):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                sc.hit_scene_device(r6.data_ptr(), n, ids.data_ptr(), t.data_ptr(), pos.data_ptr(), nrm.data_ptr(), mode=mode, stream=st.cuda_stream)
                e1.record(st)
                st.synchronize()
                best = min(best, e0.elapsed_time(e1))
        stats = sc.hit_scene_stats(r6.data_ptr(), n, mode=mode)
        return ids, pos, nrm, {"rays": n, "ms": best, "value": n / best / 1e3, "unit": "Mrays/s", "node_visits_per_ray": stats["node_visits_per_ray"],
                               "tri_tests_per_ray": stats["tri_tests_per_ray"], "hit_rate": stats["hit_rate"]}

    out = {}
    ids, pos, nrm, out["primary_closest"] = timed(rays, tm.HIT_CLOSEST)
    hit = ids >= 0
    pos, nrm = pos[hit], nrm[hit]
    shadow = torch.cat([pos, light.expand_as(pos)], 1).contiguous()
    ids_any, _, _, out["shadow_any"] = timed(shadow, tm.HIT_ANY)
    try:  # the same shadow rays through the sun grid (what the render kernels do): must agree ray by ray
        ids_sun, _, _, out["shadow_sun_grid"] = timed(shadow, tm.HIT_SUN)
        out["shadow_sun_grid"]["agrees_with_shadow_any"] = bool(((ids_any >= 0) == (ids_sun >= 0)).all().item())
    except Exception as e:  # noqa: BLE001 -- a scene without a grid (TMPT_SUN_GRID=0)
        out["shadow_sun_grid"] = {"unavailable": repr(e)}
    r = torch.randn(pos.shape, device=dev, generator=g)
    r = r / r.norm(dim=1, keepdim=True)
    nd = nrm + r
    nd = nd / nd.norm(dim=1, keepdim=True).clamp_min(1e-20)
    bounce = torch.cat([pos, nd], 1).contiguous()
    _, _, _, out["bounce_closest"] = timed(bounce, tm.HIT_CLOSEST)
    out["ray_set"] = f"{w}x{h} camera rays (jittered, one per pixel), their diffuse bounce rays and sun shadow rays; device-generated, seed 1"
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Each array as out_dir/<name>.npy in float32 (exact for the uint8 frame) or float64 (exact for counts up to 2**53), so
    that two builds can be compared output for output on the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32))


# ------------------------------------------------------------------------------------------
def bench_reference(args, scene, w, h, spp, rank, world):
    if rank != 0:
        return 0
    cw, ch, cspp = CPU_SAMPLE[scene]
    vals, secs = [], []
    for i in range(args.warmup + args.steps):
        mr, rays, sec, kind, cores = run_reference_cpu(scene, cw, ch, cspp)
        if i >= args.warmup:
            vals.append(mr)
            secs.append(sec)
    value = statistics.mean(vals)
    sample = f"{scene_label(scene)} {cw}x{ch} {cspp}spp (same scene and camera, reduced pixels/spp), {int(rays)} rays per step"
    line = {
        "impl": "reference", "metric": "Mrays/s (primary+bounce+shadow)", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * statistics.mean(secs), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{scene_label(scene)} {w}x{h} {spp}spp", "cpu_sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)
    return 0


def bench_b200(args, scene, w, h, spp, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import toymeshpathtracer_b200 as tm
    from toymeshpathtracer_b200 import multigpu

    if not torch.cuda.is_available() or tm.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    path = scene_obj_path(scene) if rank == 0 else None
    if world > 1:
        box = [path]
        dist.broadcast_object_list(box, src=0)
        path = box[0]
    tris, mn, mx = tm.load_scene(path)
    cam = tm.camera_for_scene(path, mn, mx, w, h)
    # the scene is built twice: the first build of a process pays for loading the CUDA module and every build kernel (and, on some
    # boxes, for hundreds of ms of one-off driver work); both times are reported, `bvh.build_ms` / `scene_build_wall_ms` are the second
    t0 = time.perf_counter()
    first = tm.Scene(tris, device=local_rank)
    first_build = {"build_ms": first.info()["build_ms"], "wall_ms": (time.perf_counter() - t0) * 1e3}
    first.close()
    t0 = time.perf_counter()
    sc = tm.Scene(tris, device=local_rank)
    build_wall_ms = (time.perf_counter() - t0) * 1e3
    info = sc.info()

    stream = torch.cuda.Stream(dev)
    peer = None
    if world > 1 and args.gather == "peer":
        # every rank must agree: fall back to the NCCL gather if the IPC mapping fails anywhere
        try:
            peer = multigpu.PeerFrame(w, h, rank, world, local_rank)
            ok = torch.ones(1, dtype=torch.int32, device=dev)
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"[rank {rank}] peer frame unavailable ({e}); using the NCCL gather\n")
            ok = torch.zeros(1, dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0 and peer is not None:
            peer.close()
            peer = None
        elif int(ok.item()) == 0:
            peer = None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    launches0 = tm.launch_count()
    step_ms, step_rays = [], []
    clocks = ClockSampler(local_rank)
    frame = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step():
        nonlocal frame
        with torch.cuda.stream(stream):
            flush.zero_()  # L2 flush between timed iterations (outside the event pair)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            frame, rays = multigpu.render_frame(sc, cam, w, h, spp, rank, world, group=None, device=dev, peer=peer)
            e1.record(stream)
        stream.synchronize()
        return e0.elapsed_time(e1), int(rays.item())

    for _ in range(args.warmup):
        one_step()
    barrier()
    launches1 = tm.launch_count()
    with clocks:
        for _ in range(args.steps):
            ms, rays = one_step()
            step_ms.append(ms)
            step_rays.append(rays)
    barrier()
    launches2 = tm.launch_count()
    if args.dump_outputs:
        # what render_frame handed back in the last timed step: rank 0's frame and the ray count of the whole job
        last_rays = torch.tensor([step_rays[-1]], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(last_rays, op=dist.ReduceOp.SUM)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"frame": frame, "rays": last_rays})
        barrier()

    tot_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    tot_rays = torch.tensor([sum(step_rays)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_rays, op=dist.ReduceOp.SUM)
    tot_ms, tot_rays = float(tot_ms.item()), int(tot_rays.item())
    value = tot_rays / (tot_ms * 1e-3) / 1e6

    # e2e: the user-facing C-ABI call with HOST buffers (single-GPU form; N>1: stripes + gather + D2H of the frame)
    e2e_ms, e2e_rays = [], []
    host_frame = torch.empty((h, w, 4), dtype=torch.uint8).pin_memory() if rank == 0 else None  # caller-owned, pinned, allocated once
    for i in range(1 + min(args.steps, 3)):
        barrier()
        t0 = time.perf_counter()
        if world == 1:
            rays, sec = sc.render_into(cam, w, h, spp, host_frame.data_ptr())  # tmpt_render(TMPT_HOST): kernels + D2H of the frame
            img = host_frame
        else:
            with torch.cuda.stream(stream):
                fr, rr = multigpu.render_frame(sc, cam, w, h, spp, rank, world, device=dev, peer=peer)
                if rank == 0:  # the frame lands in pinned host memory (allocated once, outside the timed region)
                    host_frame.copy_(fr.reshape(host_frame.shape), non_blocking=True)
                    img = host_frame
            stream.synchronize()
            rays = int(rr.item())
        dt = (time.perf_counter() - t0) * 1e3  # this rank's work is done: kernels, the frame's all-reduce and (rank 0) the copy to host memory
        barrier()                               # (the frame time of the job is the MAX over ranks, taken below)
        if i > 0:
            e2e_ms.append(dt)
            e2e_rays.append(rays)
    e2e_t = torch.tensor([sum(e2e_ms)], dtype=torch.float64, device=dev)
    e2e_r = torch.tensor([sum(e2e_rays)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_r, op=dist.ReduceOp.SUM)
    e2e_value = int(e2e_r.item()) / (float(e2e_t.item()) * 1e-3) / 1e6

    # BASELINE configs 1-4 and the HitScene kernels (reported beside the headline; not part of its timed region)
    extra_configs, hit_scene = [], None
    if args.workload == "sponza_1080p_64spp" and not args.no_extras:
        extra_configs = measure_extra_configs(tm, multigpu, dist, torch, sc, dev, stream, rank, world, local_rank, flush, peer is not None)
        if world == 1:
            hit_scene = measure_hit_scene(tm, torch, sc, cam, w, h, dev)

    line = None
    if rank == 0:
        clk = clocks.summary()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_mhz = clk["sm_mhz"] or peaks.get("sm_max_mhz", 1965.0)
        fp32_peak = sm_count * 128 * 2 * sm_mhz * 1e6 / 1e12  # nominal TFLOP/s at the clock seen under load
        peak_source = f"{sm_count} SM x 128 lanes x 2 x {sm_mhz:.0f} MHz (median SM clock sampled during the timed region)"
        try:  # the FFMA rate actually measured on this pool's B200 (tools/microbench/peaks.cu), scaled to the clock seen
            pk = json.load(open(os.path.join(ROOT, "profiles", "r1_peaks.json")))
            fp32_peak = pk["ffma_tflops"] * sm_mhz / pk["at_sm_mhz"]
            peak_source = f"measured FFMA rate {pk['ffma_tflops']} TFLOP/s at {pk['at_sm_mhz']} MHz (profiles/r1_microbench_peaks.txt), scaled to {sm_mhz:.0f} MHz"
        except (OSError, KeyError, ValueError):
            pass
        stats = sc.traversal_stats(cam, w, h, spp) if hasattr(sc, "traversal_stats") else None
        flops_per_ray = (stats["box_tests_per_ray"] * 18 + stats["tri_tests_per_ray"] * 46) if stats else None
        kernel_ms = statistics.mean(step_ms)
        traffic, traffic_source = None, None
        try:  # dram__bytes_read + dram__bytes_write of this kernel on this workload: NOT measured in this run (ncu cannot run inside a
            # timed bench), read from the committed ncu --set full capture of the same instantiation and labelled as such
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2g_traffic.json")))["k_render"]
            if args.workload == "sponza_1080p_64spp" and world == 1:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                traffic_source = "from file profiles/r2g_traffic.json (" + tj["source"] + "), not measured in this run"
        except (OSError, KeyError, ValueError):
            pass
        achieved = (value / world) * 1e6 * flops_per_ray / 1e12 if flops_per_ray else None
        roofline = {
            "bound": "fp32_issue (L2-resident traversal; neither hbm nor tensor, SURVEY.md 8(d))",
            "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": (achieved / fp32_peak) if achieved else None,
            "traffic": traffic, "traffic_source": traffic_source, "per_ray": stats, "flops_per_ray": flops_per_ray,
            "peak_source": peak_source,
            "hbm_context": {"algorithmic_bytes_per_frame": int(tris.size * 4 + w * h * 4), "hbm_peak_gbs_measured": peaks.get("hbm_gbs"),
                            "hbm_frac": (tris.size * 4 + w * h * 4) / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None},
            "kernel": "k_render", "kernel_ms": kernel_ms,
            "limiter": "L1 data stage (l1tex__data_pipe_lsu_wavefronts 88 % of peak) and issue slots (65 %), profiles/r2g_k_render_ncu_summary.txt",
        }
        if stats:
            # the limiter in the kernel's own units: 16-byte rows gathered per clock and SM (7 per node step, 3 per triangle test), against
            # the rate a divergent 128-bit gather reaches when every row hits L1 (tools/microbench/gather2.cu, profiles/r1_microbench_peaks.txt)
            rows_per_ray = 7.0 * stats["node_visits_per_ray"] + 3.0 * stats["tri_tests_per_ray"]
            rows_rate = (value / world) * 1e6 * rows_per_ray / (sm_count * sm_mhz * 1e6)
            roofline["l1_gather"] = {"rows_per_ray": rows_per_ray, "rows_per_clk_per_sm": rows_rate, "peak_rows_per_clk_per_sm_all_l1_hits": 2.9,
                                     "frac": rows_rate / 2.9, "l1_hit_rate_ncu": 0.64,
                                     "note": "rows of node steps and triangle tests (the sun grid's list entries, ~1 row per shadow ray, not counted); misses cost about "
                                             "twice a hit in the data stage (1.3-1.5 rows/clk): ncu puts the stage at 88 % of its wavefront peak"}
        cw, ch, cspp = CPU_SAMPLE[scene]
        try:
            mr, crays, csec, kind, cores = run_reference_cpu(scene, cw, ch, cspp)
            cpu = {"value": mr, "unit": "Mrays/s", "cores": cores, "kind": kind,
                   "sample": f"{scene_label(scene)} {cw}x{ch} {cspp}spp (same scene and camera, reduced pixels/spp), {int(crays)} rays in {csec:.2f} s"}
            ow, oh, ospp = CPU_SAMPLE_1T[scene]
            mr1, crays1, csec1, _, _ = run_reference_cpu(scene, ow, oh, ospp, threads=1)
            cpu["one_thread"] = {"value": mr1, "unit": "Mrays/s", "cores": 1,
                                 "sample": f"{scene_label(scene)} {ow}x{oh} {ospp}spp, {int(crays1)} rays in {csec1:.2f} s"}
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": "Mrays/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}
        line = {
            "metric": "Mrays/s (primary+bounce+shadow)", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": tot_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{scene_label(scene)} {w}x{h} {spp}spp", "rays_per_frame": step_rays[-1] if world == 1 else tot_rays // args.steps,
                       "parallelism": "single GPU" if world == 1 else (f"8x4-pixel tiles interleaved ((tx + ty) % {world}) over {world} GPUs" if multigpu.DEFAULT_STRIPE_ROWS == 0 else
                                                                        f"row stripes of {multigpu.DEFAULT_STRIPE_ROWS} over {world} GPUs") + ", BVH replica per GPU, " + (
                           "pixels stored straight into rank 0's frame over NVLink (CUDA IPC peer memory)" if peer else "frame gathered to rank 0 (NCCL)"),
                       "work_unit": "8x4 pixel tile x chunk of spp/32 (1..8) samples per warp, dynamic fetch",
                       "render_kernel": _kernel_name(sc),
                       "l2": "flushed between timed iterations (256 MB write)", "bvh": {k: info[k] for k in ("node_count", "leaf_count", "max_depth", "sah_cost", "build_ms", "device_bytes")},
                       "scene_build_wall_ms": build_wall_ms, "first_build_in_process": first_build},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": 88, "d2h_bytes_per_step": w * h * 4 + 8,
                    "ms_per_step": float(e2e_t.item()) / len(e2e_ms)},
            "gpu_launches": launches2 - launches1,
            "clocks": clk, "roofline": roofline, "cpu_baseline": cpu,
            "configs": extra_configs, "hit_scene": hit_scene,
        }
        _emit(line)
    sc.close()
    if world > 1:
        dist.barrier()
        if peer:
            peer.close()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sponza_1080p_64spp", choices=sorted(WORKLOADS))
    ap.add_argument("--gather", default="peer", choices=["nccl", "peer"], help="N>1: how the frame reaches rank 0")
    ap.add_argument("--no-extras", action="store_true", help="skip the `configs` (BASELINE configs 1-4) and `hit_scene` sections")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's frame and ray count as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference's CPU program keeps no frame)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one rank per GPU
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    scene, w, h, spp = WORKLOADS[args.workload]
    # stdout carries ONE line, the JSON: whatever libraries print while the bench runs (NCCL's version banner, for one) goes to
    # stderr -- file descriptor 1 points at stderr until the line is printed
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    try:
        if args.impl == "reference":
            return bench_reference(args, scene, w, h, spp, rank, world)
        return bench_b200(args, scene, w, h, spp, rank, world, local_rank)
    finally:
        _restore_stdout()


_STDOUT_FD = None


def _restore_stdout():
    global _STDOUT_FD
    if _STDOUT_FD is not None:
        sys.stdout.flush()
        os.dup2(_STDOUT_FD, 1)
        os.close(_STDOUT_FD)
        _STDOUT_FD = None


def _emit(line):
    _restore_stdout()
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    sys.exit(main())
