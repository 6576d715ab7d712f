#!/usr/bin/env python
"""Generate tests/golden/ from the UNMODIFIED reference compiled in this container.

Test infrastructure.  Run here (needs /root/reference); the outputs are committed
because /root/reference does not exist on the GPU box.

    python oracle/gen_golden.py            # everything
    python oracle/gen_golden.py --fast     # skip the high-spp reference images

What is written (all produced by oracle/_ref/libref.so or oracle/_ref/TrimeshTracer,
i.e. by the reference's own code -- never by oracle.c or by the CUDA path):

  scenes/<name>.npz     triangle array exactly as LoadScene builds it (model + 2 floor
                        triangles, main.cpp:135-162), model bounds, the main() camera
  rays/<name>.npz       rays a reference render shoots (primary / bounce / shadow) with
                        the octree HitScene answer (flag, t, pos, normal) and the
                        ID-carrying brute-force answer (SURVEY.md 8(c))
  kat.json              RNG / sampler / camera known answers; sha256 + ray counts of the
                        reference binary's 640x360x4 renders
  images/<name>_*.png   high-spp reference renders for the statistical image gate
  rays/sponza.npz       the same ray record on the Sponza stand-in (tools/gen_sponza.py; the
                        reference's data/sponza.obj is absent), written by --sponza
  images/sponza_160x90_1024spp_{a,b}.png
                        TWO independent 1024-spp renders of the stand-in by the reference's own
                        row functor (b = the upper half of a 160x180 frame whose camera maps rows
                        90..179 onto the same view: other row seeds, main.cpp:204); their distance
                        is what the GPU image's MAE / PSNR gates are derived from (kat.json)
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.pyoracle import REF_BIN, REF_ROOT, Ref  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SCENES = ["triangle", "cube", "suzanne", "teapot"]
RAY_STRIDE = {"triangle": 16, "cube": 8, "suzanne": 8, "teapot": 8}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fast", action="store_true")
    ap.add_argument("--sponza", action="store_true", help="only (re)generate the Sponza stand-in goldens; kat.json is updated in place")
    ap.add_argument("--cli", nargs="?", const=REF_BIN, metavar="BINARY",
                    help="only (re)generate cli_args.json from BINARY (default: the reference binary)")
    args = ap.parse_args()
    if args.sponza:
        return sponza_goldens()
    if args.cli:
        return cli_goldens(args.cli)
    from PIL import Image

    R = Ref()
    for d in ("scenes", "rays", "images"):
        os.makedirs(os.path.join(GOLD, d), exist_ok=True)
    kat = {"generator": "oracle/gen_golden.py", "reference_build": "g++ 13.3 -O2 -ffp-contract=off -DNDEBUG + tbb_shim"}

    # --- RNG / samplers (maths.cpp:5-38) ---
    kat["rng"] = {}
    for seed in (1, 9782, 0xDEADBEEF, 2463534242):
        st, fl = R.rng_states(seed, 16)
        kat["rng"][str(seed)] = {"states": st.tolist(), "float_bits": bits(fl).tolist()}
    disk, s_end = R.random_in_unit_disk(12345, 64)
    kat["disk"] = {"seed": 12345, "bits": bits(disk).ravel().tolist(), "end_state": int(s_end)}
    unit, s_end = R.random_unit_vectors(4321, 64)
    kat["unit_vector"] = {"seed": 4321, "bits": bits(unit).ravel().tolist(), "end_state": int(s_end)}
    kat["light_dir_bits"] = bits(R.light_dir()).tolist()
    cam = R.camera_make([1.5, 2.0, -3.0], [0.1, -0.2, 0.3], [0, 1, 0], 60.0, 16 / 9, 0.03, 4.2)
    kat["camera_make"] = {"args": [[1.5, 2.0, -3.0], [0.1, -0.2, 0.3], [0, 1, 0], 60.0, 16 / 9, 0.03, 4.2],
                          "bits": bits(cam).tolist()}
    st2 = np.stack([np.linspace(0, 1, 32, dtype=np.float32), np.linspace(1, 0, 32, dtype=np.float32)], 1)
    rays, s_end = R.camera_get_rays(cam, st2, 777)
    kat["camera_get_rays"] = {"seed": 777, "st_bits": bits(st2).ravel().tolist(), "ray_bits": bits(rays).ravel().tolist(),
                              "end_state": int(s_end)}

    # --- scenes, ray sets, binary renders ---
    kat["renders_640x360x4"] = {}
    for name in SCENES:
        path = os.path.join(REF_ROOT, "data", f"{name}.obj")
        h, tris, mn, mx = R.scene_load(path)
        cam = R.camera_for_scene(h, path, 640, 360)
        np.savez_compressed(os.path.join(GOLD, "scenes", f"{name}.npz"), tris=tris, bounds_min=mn, bounds_max=mx,
                            camera_640x360=cam)
        rays, kind = R.record_path_rays(h, cam, 640, 360, RAY_STRIDE[name], 200000)
        flag, t, pos, nrm = R.hit_scene(h, rays)
        bid, bt, bpos, bnrm = R.hit_brute(h, rays)
        same = ((flag == 1) == (bid >= 0)).all() and (bits(t) == bits(bt)).all() and (bits(pos) == bits(bpos)).all() \
            and (bits(nrm) == bits(bnrm)).all()
        print(f"{name}: {tris.shape[0]} tris, {rays.shape[0]} rays, hits {(bid >= 0).sum()}, octree==brute: {same}")
        assert same, "reference octree HitScene and ID-carrying brute force disagree"
        np.savez_compressed(os.path.join(GOLD, "rays", f"{name}.npz"), rays=rays, kind=kind.astype(np.int8), flag=flag.astype(np.int8),
                            id=bid, t=t, pos=pos, normal=nrm)
        # the reference BINARY, unmodified main(): output.png + its own report lines
        with tempfile.TemporaryDirectory() as td:
            out = subprocess.run([REF_BIN, "640", "360", "4", path], cwd=td, check=True, capture_output=True, text=True).stdout
            img = np.array(Image.open(os.path.join(td, "output.png")).convert("RGBA"))
        krays = float(out.split("- ")[1].split(" K Rays")[0])
        rimg, rc = R.render(h, cam, 640, 360, 4)
        assert (rimg[::-1] == img).all(), "harness render != binary render"
        kat["renders_640x360x4"][name] = {"sha256_rgba_png_order": hashlib.sha256(img.tobytes()).hexdigest(), "ray_count": int(rc),
                                          "reported_krays": krays, "mean_rgb": img[..., :3].reshape(-1, 3).mean(0).tolist()}
        if not args.fast and name in ("cube", "suzanne"):
            w, hgt, spp = 320, 180, (1024 if name == "cube" else 256)
            cam_s = R.camera_for_scene(h, path, w, hgt)
            big, rc = R.render(h, cam_s, w, hgt, spp)
            Image.fromarray(big[::-1, :, :3].copy()).save(os.path.join(GOLD, "images", f"{name}_{w}x{hgt}_{spp}spp.png"), optimize=True)
            print(f"  reference image {w}x{hgt}x{spp}: {rc} rays")
        R.scene_free(h)

    with open(os.path.join(GOLD, "kat.json"), "w") as f:
        json.dump(kat, f, indent=1)
    print("wrote", GOLD)


def image_distance(a, b):
    """MAE / PSNR over pixels that are not NaN-black in either image (SURVEY.md 0.7) -- the metric of the GPU test."""
    a, b = a[..., :3].astype(np.float64), b[..., :3].astype(np.float64)
    bad = ((a.sum(-1) == 0) & (b.sum(-1) > 120)) | ((b.sum(-1) == 0) & (a.sum(-1) > 120))
    d = (a - b)[~bad]
    return float(np.abs(d).mean()), float(10 * np.log10(255.0 ** 2 / (d ** 2).mean())), int(bad.sum())


def sponza_goldens():
    """Sponza stand-in: hit-ID ray set and the converged-image pair, all from the unmodified reference (libref.so)."""
    from PIL import Image
    from tools.gen_sponza import write_obj
    R = Ref()
    with open(os.path.join(GOLD, "kat.json")) as f:
        kat = json.load(f)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "sponza.obj")  # the name triggers the hard-coded eye (main.cpp:300-301)
        write_obj(path)
        h, tris, mn, mx = R.scene_load(path)
    assert tris.shape[0] == 66452
    cam = R.camera_for_scene(h, "sponza.obj", 640, 360)
    # the scene itself is not stored (2.4 MB, regenerated by tools/gen_sponza.py): its hash pins it
    kat["sponza"] = {"tri_count": int(tris.shape[0]), "tris_sha256": hashlib.sha256(tris.tobytes()).hexdigest(),
                     "bounds_min_bits": bits(mn).tolist(), "bounds_max_bits": bits(mx).tolist(), "camera_640x360_bits": bits(cam).tolist()}
    rays, kind = R.record_path_rays(h, cam, 640, 360, 5, 200000)
    flag, t, pos, nrm = R.hit_scene(h, rays)
    bid, bt, bpos, bnrm = R.hit_brute(h, rays)
    # Flag and t bits of the octree walk and of the ID-carrying scan must agree on every ray.  The payload may differ on
    # TIES: the stand-in has a few coplanar overlapping faces, two triangles then give bit-equal t, the octree keeps the
    # first one in ITS order (scene.cpp:34), the scan the lowest input index -- the stated tie rule of this repository.
    hit = bid >= 0
    assert ((flag == 1) == hit).all() and (bits(t)[hit] == bits(bt)[hit]).all(), "reference octree HitScene and brute force disagree on flag / t"
    tie = hit & ((bits(pos) != bits(bpos)).any(1) | (bits(nrm) != bits(bnrm)).any(1))
    print(f"sponza: {tris.shape[0]} tris, {rays.shape[0]} rays ({(kind == 0).sum()} primary, {(kind == 1).sum()} bounce, "
          f"{(kind == 2).sum()} shadow), hits {hit.sum()}, octree==brute on flag and t; {tie.sum()} ties where the octree's payload comes from "
          f"another triangle with bit-equal t")
    assert tie.sum() <= 20
    ti = np.nonzero(tie)[0].astype(np.int32)
    np.savez_compressed(os.path.join(GOLD, "rays", "sponza.npz"), rays=rays, kind=kind.astype(np.int8), flag=flag.astype(np.int8),
                        id=bid, t=bt, pos=bpos, normal=bnrm, tie_rays=ti, tie_octree_pos=pos[ti], tie_octree_normal=nrm[ti])
    # converged image pair, 160x90x1024
    w, hgt, spp = 160, 90, 1024
    cam_a = R.camera_for_scene(h, "sponza.obj", w, hgt)
    img_a, rc_a = R.render(h, cam_a, w, hgt, spp)
    cam_b = cam_a.copy()          # 22 floats: origin, lowerLeftCorner, horizontal, vertical, u, v, w, lensRadius (maths.h:106-111)
    cam_b[3:6] = cam_a[3:6] - cam_a[9:12]   # lowerLeftCorner - vertical
    cam_b[9:12] = 2.0 * cam_a[9:12]         # rows 90..179 of a 160x180 frame = the same view, row seeds 90..179
    img_b2, rc_b = R.render(h, cam_b, w, 2 * hgt, spp)
    img_b = img_b2[hgt:]
    mae, psnr, bad = image_distance(img_a, img_b)
    print(f"  reference pair {w}x{hgt}x{spp}: rays {rc_a}, MAE {mae:.3f} PSNR {psnr:.2f} dB, {bad} masked")
    Image.fromarray(img_a[::-1, :, :3].copy()).save(os.path.join(GOLD, "images", f"sponza_{w}x{hgt}_{spp}spp_a.png"), optimize=True)
    Image.fromarray(img_b[::-1, :, :3].copy()).save(os.path.join(GOLD, "images", f"sponza_{w}x{hgt}_{spp}spp_b.png"), optimize=True)
    kat["sponza"]["image_pair_160x90_1024spp"] = {"mae": mae, "psnr": psnr, "masked": bad, "ray_count_a": int(rc_a),
                                                  "mean_rgb_a": img_a[..., :3].reshape(-1, 3).mean(0).tolist(),
                                                  "mean_rgb_b": img_b[..., :3].reshape(-1, 3).mean(0).tolist()}
    R.scene_free(h)
    with open(os.path.join(GOLD, "kat.json"), "w") as f:
        json.dump(kat, f, indent=1)
    print("updated", os.path.join(GOLD, "kat.json"))


CLI_STOPS = ("Usage: ", "ERROR: invalid ", "ERROR: failed to load .obj file")  # main.cpp:258-291: every exit before the render


def cli_goldens(binary):
    """Random argument lists (atoi corner cases, out-of-range values, a missing .obj) and what `binary` prints for each one on
    which it stops before rendering: exit code and stdout.  "{obj}" stands for a valid one-triangle .obj file."""
    binary = os.path.abspath(binary)
    toks = ["0", "1", "-1", "10000", "10001", "1024", "1025", "abc", "12abc", " 7", "+3", "1e3", "99999999999", "", "2.9"]
    rng = np.random.default_rng(1)
    cases = [[], ["1"], ["1", "2"], ["1", "2", "3"]]
    cases += [[toks[rng.integers(0, 15)], toks[rng.integers(0, 15)], toks[rng.integers(0, 15)], "{obj}" if rng.random() < 0.8 else "/nonexistent.obj"]
              for _ in range(120)]
    out = []
    with tempfile.TemporaryDirectory() as td:
        obj = os.path.join(td, "t.obj")
        with open(obj, "w") as f:
            f.write("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
        for args in cases:
            r = subprocess.run([binary, *(obj if a == "{obj}" else a for a in args)], cwd=td, capture_output=True, text=True)
            if r.stdout.startswith(CLI_STOPS):
                out.append({"args": args, "returncode": r.returncode, "stdout": r.stdout})
    with open(os.path.join(GOLD, "cli_args.json"), "w") as f:
        json.dump({"generator": "oracle/gen_golden.py --cli", "recorded_from": os.path.relpath(binary, ROOT), "cases": out}, f, indent=1)
    print(f"cli_args.json: {len(out)} of {len(cases)} argument lists stop before the render")


if __name__ == "__main__":
    main()
