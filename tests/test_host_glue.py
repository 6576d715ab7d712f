"""Host glue behind the C ABI (csrc/host.cpp) and the library surface -- CPU only.
No compute call is made here (there is no GPU); the compute entry points must fail loudly."""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from conftest import ROOT, bits, load_scene
from oracle.pyoracle import REF_ROOT


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "tmpt.h")).read()
    declared = set(re.findall(r"\b(tmpt_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(tm.ABI_SYMBOLS)
    L = tm.lib()
    for name in declared:
        assert getattr(L, name) is not None
    out = subprocess.run(["nm", "-D", "--defined-only", tm.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (tmpt_[a-z_0-9]+)", out))
    assert declared <= exported


def test_oracle_is_not_linked_into_the_product():
    out = subprocess.run(["ldd", tm.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out and "libemu" not in out and "libref" not in out
    syms = subprocess.run(["nm", "-D", tm.LIB_PATH], capture_output=True, text=True).stdout
    assert "orc_" not in syms and "emu_" not in syms


@pytest.mark.skipif(tm.device_count() > 0, reason="a GPU is present")
def test_compute_fails_loudly_without_a_gpu():
    tri = np.zeros((1, 9), np.float32)
    with pytest.raises(tm.TmptError) as e:
        tm.Scene(tri)
    assert e.value.status == tm.TMPT_ERR_CUDA and "no CPU path" in str(e.value)


OBJ_TEXT = """# comment
v 0 0 0
v 1.5 0 0\r
v 1 1e0 -2.5E-1
v   0\t1 0.125
vt 0 0
vn 0 0 1
f 1/1/1 2/1/1 3/1/1 4/1/1
f -4//1 -3//1 -1//1
f 1 2 3 4 1
usemtl x
f 2 3
"""


def test_obj_loader_grammar(tmp_path):
    p = tmp_path / "t.obj"
    p.write_bytes(OBJ_TEXT.encode())
    tris, mn, mx = tm.load_scene(str(p))
    v = np.array([[0, 0, 0], [1.5, 0, 0], [1, 1, -0.25], [0, 1, 0.125]], np.float32)
    fan = lambda idx: [[idx[0], idx[k], idx[k + 1]] for k in range(1, len(idx) - 1)]
    faces = fan([0, 1, 2, 3]) + fan([0, 1, 3]) + fan([0, 1, 2, 3, 0])
    want = v[np.array(faces)].reshape(-1, 9)
    assert tris.shape[0] == want.shape[0] + 2
    assert (bits(tris[:-2]) == bits(want)).all()
    assert mn.tolist() == [0, 0, -0.25] and mx.tolist() == [1.5, 1, 0.125]
    # the two floor triangles (main.cpp:153-162)
    ex, ez = np.float32(1.5) * np.float32(0.7), np.float32(0.375) * np.float32(0.7)
    x0, x1, z0, z1 = np.float32(0) - ex, np.float32(1.5) + ex, np.float32(-0.25) - ez, np.float32(0.125) + ez
    floor = np.array([[x0, 0, z0, x0, 0, z1, x1, 0, z0], [x0, 0, z1, x1, 0, z1, x1, 0, z0]], np.float32)
    assert (bits(tris[-2:]) == bits(floor)).all()


def test_obj_loader_errors(tmp_path):
    with pytest.raises(tm.TmptError) as e:
        tm.load_scene(str(tmp_path / "missing.obj"))
    assert e.value.status == tm.TMPT_ERR_IO
    p = tmp_path / "bad.obj"
    p.write_text("v 0 0 0\nf 1 2 3\n")
    with pytest.raises(tm.TmptError):
        tm.load_scene(str(p))
    p = tmp_path / "empty.obj"
    p.write_text("# nothing\n")
    tris, mn, mx = tm.load_scene(str(p))  # like the reference: just the two floor triangles
    assert tris.shape == (2, 9)


def test_float_parser_matches_reference_semantics(tmp_path):
    # objparser.cpp:62-131: double mantissa, ONE scaling by an exact power of ten, then float
    cases = ["0.1", "-0.30000001", "123456789.125", "1e-7", "3.4028234e38", "1.17549435e-38", "+.5", "7.", "0.000000000000000000000001",
             "12345678901234567890", "-1.5e+3", "2E2"]
    p = tmp_path / "f.obj"
    p.write_text("".join(f"v {c} 0 0\n" for c in cases) + "f 1 2 3\n")
    tris, *_ = tm.load_scene(str(p))

    def ref_parse(s):
        m = re.match(r"([+-]?)(\d*)(?:\.(\d*))?(?:[eE]([+-]?\d+))?$", s)
        sign = -1.0 if m.group(1) == "-" else 1.0
        digits = (m.group(2) or "") + (m.group(3) or "")
        mant = 0.0
        for ch in digits:
            mant = mant * 10.0 + float(int(ch))
        power = -len(m.group(3) or "") + int(m.group(4) or 0)
        if -22 <= power <= 0:
            return np.float32(sign * mant / 10.0 ** (-power))
        if 0 < power <= 22:
            return np.float32(sign * mant * 10.0 ** power)
        return np.float32(sign * mant * np.power(10.0, power))

    got = np.array([tris[0, 0], tris[0, 3], tris[0, 6]], np.float32)
    want = np.array([ref_parse(c) for c in cases[:3]], np.float32)
    assert (bits(got) == bits(want)).all()
    # all of them through single-vertex faces
    p.write_text("".join(f"v {c} 0 0\n" for c in cases) + "".join(f"f {i+1} {i+1} {i+1}\n" for i in range(len(cases))))
    tris, *_ = tm.load_scene(str(p))
    with np.errstate(over="ignore"):
        want = np.array([ref_parse(c) for c in cases], np.float32)
    assert (bits(tris[:len(cases), 0]) == bits(want)).all()


def _random_obj_number(rng):
    k = int(rng.integers(0, 13))
    x = rng.normal() * 10 ** rng.uniform(-6, 6)
    return ["%.9g" % x, "%.3f" % x, "%e" % x, "%E" % x, "%d" % int(x), "%d." % int(x), ("%.6f" % abs(x % 1))[1:], "+%.5g" % abs(x), "%.17g" % x,
            "%.25f" % x, "%de%d" % (rng.integers(-999, 999), rng.integers(-30, 30)), "%.4fe+%d" % (x, rng.integers(0, 25)),
            # an exponent of 10-13 digits: the reference accumulates it in an int that wraps (objparser.cpp:113-117); so must this
            "%de%s%d" % (rng.integers(1, 99), rng.choice(["", "-", "+"]), rng.integers(2 ** 31, 2 ** 42))][k]


def _random_obj_text(rng):
    """OBJ text over the whole grammar objparser.cpp accepts: every number syntax (no integer / fraction part, exponents that take
    the pow() branch or overflow an int, 25 decimals), records with too few or too many numbers, trailing garbage, tabs, CRLF, vt / vn / g / s /
    usemtl records, 'v' not followed by a blank, faces as v, v/vt, v//vn, v/vt/vn with positive, '+' and relative indices, polygons
    (fans), a 0 index (ends the face), one- and two-corner faces, vertices declared after faces, no final newline."""
    num = lambda: _random_obj_number(rng)
    sep = lambda: str(rng.choice([" ", "  ", "\t", " \t "]))
    eol = str(rng.choice(["\n", "\r\n"]))
    lines, count_v = [], 0
    for _ in range(int(rng.integers(3, 60))):
        r = rng.random()
        if r < 0.05: lines.append("# comment " + num())
        if r > 0.93: lines.append("vn %s %s %s" % (num(), num(), num()))
        if 0.88 < r < 0.93: lines.append("vt %s %s" % (num(), num()))
        if 0.86 < r < 0.88: lines.append("")
        if 0.84 < r < 0.86: lines.append("v\t1 2 3")
        if 0.82 < r < 0.84: lines.append(" v 1 2 3")
        if 0.80 < r < 0.82: lines.append("g grp\ns 1\no obj\nusemtl m\nmtllib x.mtl")
        nnum = 3 if rng.random() < 0.9 else int(rng.integers(0, 5))
        lines.append("v " + sep().join(num() for _ in range(nnum)) + str(rng.choice(["", " 1.0", " # c", " x", ""])))
        count_v += 1
    for _ in range(int(rng.integers(1, 40))):
        toks = []
        for _ in range(int(rng.choice([1, 2, 3, 3, 3, 4, 5, 7]))):
            vi = int(rng.integers(1, count_v + 1))
            if rng.random() < 0.3: vi -= count_v + 1
            a, b = int(rng.integers(1, 5)), int(rng.integers(1, 5))
            tok = [str(vi), "%d/%d" % (vi, a), "%d//%d" % (vi, b), "%d/%d/%d" % (vi, a, b)][int(rng.integers(0, 4))]
            toks.append("+" + tok if vi > 0 and rng.random() < 0.05 else tok)
        if rng.random() < 0.05: toks.insert(int(rng.integers(0, len(toks) + 1)), "0")
        if rng.random() < 0.05: toks.append("garbage 1 2 3")
        lines.append("f " + sep().join(toks) + str(rng.choice(["", " ", "\t"])))
        if rng.random() < 0.1:
            lines.append("v %s %s %s" % (num(), num(), num()))
            count_v += 1
    return eol.join(lines) + (eol if rng.random() < 0.7 else "")


@pytest.mark.ref
def test_obj_loader_equals_reference_loadscene_on_random_files(ref, tmp_path):
    """SURVEY.md 8(f1): 150 random .obj files through the reference's own LoadScene (objparser.cpp + main.cpp:122-170, oracle/_ref)
    and through tmpt_load_obj: the same Triangle[] (floor included), bounds and camera (22 floats, random frame sizes), bit for bit.  (4000 seeds were run once: no difference.)"""
    p = str(tmp_path / "f.obj")
    for seed in range(150):
        with open(p, "wb") as f:
            f.write(_random_obj_text(np.random.default_rng(seed)).encode())
        h, rt, rmn, rmx = ref.scene_load(p)
        w, hgt = 1 + seed * 13 % 1999, 1 + seed * 7 % 1087
        rcam = ref.camera_for_scene(h, p, w, hgt)
        ref.scene_free(h)
        tris, mn, mx = tm.load_scene(p)
        assert tris.shape == rt.shape and (bits(tris) == bits(rt)).all(), seed
        assert (bits(mn) == bits(rmn)).all() and (bits(mx) == bits(rmx)).all(), seed
        assert (bits(tm.camera_for_scene(p, mn, mx, w, hgt)) == bits(rcam)).all(), seed  # main.cpp:293-311 on those bounds


@pytest.mark.ref
@pytest.mark.parametrize("name", ["triangle", "cube", "suzanne", "teapot"])
def test_obj_loader_equals_reference_loadscene(name):
    path = os.path.join(REF_ROOT, "data", f"{name}.obj")
    if not os.path.exists(path):
        pytest.skip("reference data absent")
    sc = load_scene(name)  # golden: produced by the reference's own LoadScene
    tris, mn, mx = tm.load_scene(path)
    assert tris.shape == sc["tris"].shape and (bits(tris) == bits(sc["tris"])).all()
    assert (bits(mn) == bits(sc["bounds_min"])).all() and (bits(mx) == bits(sc["bounds_max"])).all()
    cam = tm.camera_for_scene(path, mn, mx, 640, 360)
    assert (bits(cam) == bits(sc["camera_640x360"])).all()


def test_camera_matches_golden(kat):
    g = kat["camera_make"]
    cam = tm.camera_make(*g["args"])
    assert bits(cam).tolist() == g["bits"]
    for name in ["triangle", "cube", "suzanne", "teapot"]:
        sc = load_scene(name)
        cam = tm.camera_for_scene(f"/x/{name}.obj", sc["bounds_min"], sc["bounds_max"], 640, 360)
        assert (bits(cam) == bits(sc["camera_640x360"])).all()


def test_sponza_camera_special_case(oracle):
    mn, mx = np.array([-18, -0.2, -8], np.float32), np.array([18, 15, 8], np.float32)
    cam = tm.camera_for_scene("/tmp/gen/sponza.obj", mn, mx, 1920, 1080)
    assert cam[:3].tolist() == [np.float32(-5.96), np.float32(4.08), np.float32(-1.22)]
    assert (bits(cam) == bits(oracle.camera_for_scene(mn, mx, 1920, 1080, is_sponza=True))).all()
    cam2 = tm.camera_for_scene("/tmp/gen/other.obj", mn, mx, 1920, 1080)
    assert (bits(cam2) == bits(oracle.camera_for_scene(mn, mx, 1920, 1080))).all()


def test_png_writer_round_trip(tmp_path):
    from PIL import Image
    rng = np.random.default_rng(3)
    # (640x360 and 300x70 span several stored deflate blocks; 16383 / 16384 / 16385 pixels put a row at, one under and one over the
    #  65535-byte block limit; 10000 is the reference's largest width / height, main.cpp:263-275)
    for (w, h) in [(1, 1), (7, 5), (640, 360), (300, 70), (16383, 1), (16384, 2), (16385, 3), (10000, 3), (3, 10000)]:
        img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        p = str(tmp_path / f"o_{w}x{h}.png")
        tm.write_png(p, img, flip_vertically=True)
        back = np.array(Image.open(p))
        assert back.shape == (h, w, 4) and (back == img[::-1]).all()
        tm.write_png(p, img, flip_vertically=False)
        assert (np.array(Image.open(p)) == img).all()


def test_stripe_rows_partition():
    for (h, stripe, world) in [(360, 8, 1), (360, 8, 2), (1080, 8, 8), (13, 4, 3), (5, 8, 4), (1080, 4, 8)]:
        rows = [tm.stripe_rows(h, stripe, r, world) for r in range(world)]
        assert sum(rows) == h
        want = [0] * world
        for y in range(h):
            want[(y // stripe) % world] += 1
        assert rows == want


def test_cli_argument_errors():
    def run(*args):
        r = subprocess.run([tm.CLI_PATH, *args], capture_output=True, text=True)
        return r.returncode, r.stdout
    assert run() == (1, "Usage: TrimeshTracer.exe [width] [height] [samplesPerPixel] [objFile]\n")
    assert run("0", "10", "1", "x.obj") == (1, "ERROR: invalid width argument '0'\n")
    assert run("10", "10001", "1", "x.obj") == (1, "ERROR: invalid height argument '10001'\n")
    assert run("10", "10", "1025", "x.obj") == (1, "ERROR: invalid samplesPerPixel argument '1025'\n")
    assert run("10", "10", "1", "/nonexistent/x.obj") == (1, "ERROR: failed to load .obj file\n")


def test_cli_rejects_arguments_exactly_like_the_reference_binary(tmp_path):
    """main.cpp:258-291: atoi semantics ("12abc" is 12, " 7" is 7, "1e3" is 1, "abc" and "" are 0, 99999999999 overflows), the range
    checks, their order and wording, the exit codes -- 124 random argument lists (oracle/gen_golden.py --cli) through the product's
    command line, compared wherever the reference stops before it renders with the exit code and stdout stored in
    tests/golden/cli_args.json.  The reference binary is not part of the repository: those answers were recorded from this command
    line after it had printed the reference's bytes on every one of these lists, side by side with oracle/_ref/TrimeshTracer."""
    with open(os.path.join(ROOT, "tests", "golden", "cli_args.json")) as f:
        cases = json.load(f)["cases"]
    obj = tmp_path / "t.obj"
    obj.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    for case in cases:
        args = [str(obj) if a == "{obj}" else a for a in case["args"]]
        b = subprocess.run([tm.CLI_PATH, *args], cwd=tmp_path, capture_output=True, text=True)
        assert (b.returncode, b.stdout) == (case["returncode"], case["stdout"]), args
    assert len(cases) > 60


def test_real_sponza_override(tmp_path, monkeypatch):
    """TMPT_SPONZA_OBJ (the reference's own data/sponza.obj, absent from this environment): when it names a file, bench.py
    and the tools use it instead of the procedural stand-in, and every results line says which one it was."""
    import bench
    real = tmp_path / "sponza.obj"
    real.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    monkeypatch.setenv("TMPT_SPONZA_OBJ", str(real))
    assert bench.scene_obj_path("sponza") == str(real) and bench.scene_label("sponza") == "sponza.obj (real)"
    tris, mn, mx = tm.load_scene(bench.scene_obj_path("sponza"))
    assert tris.shape == (3, 9)  # the triangle + the two floor triangles LoadScene adds
    monkeypatch.delenv("TMPT_SPONZA_OBJ")
    assert "stand-in" in bench.scene_label("sponza")


def test_build_staleness_is_by_content_and_safe_under_concurrency(tmp_path):
    """toymeshpathtracer_b200.build decides by a hash of the source CONTENTS (a `git checkout` or the copy to a GPU box changes
    mtimes without changing a byte; a spurious rebuild under torchrun would be eight ranks rewriting libtmpt.so at once -- that
    happened once on an 8-GPU box) and builds under a file lock.  Touching a source must not trigger a rebuild; several processes
    asking at once must all get the library."""
    import subprocess
    import sys
    import time
    from toymeshpathtracer_b200 import build as tb
    tb.build()                                   # up to date from here on
    before = os.path.getmtime(tb.LIB)
    src = os.path.join(tb.CSRC, "bvh.cuh")
    os.utime(src)                                # newer mtime, same bytes
    code = "import toymeshpathtracer_b200.build as b, toymeshpathtracer_b200 as tm; b.build(); print(len(tm.ABI_SYMBOLS), tm.lib().tmpt_device_count() >= 0)"
    t0 = time.time()
    procs = [subprocess.Popen([sys.executable, "-c", code], cwd=os.path.dirname(tb.HERE), stdout=subprocess.PIPE, text=True) for _ in range(4)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs) and all(o.strip().endswith("True") for o in outs)
    assert os.path.getmtime(tb.LIB) == before and time.time() - t0 < 60   # nobody rebuilt
    assert not tb._stale(tb.LIB)
    with open(tb._stamp(tb.LIB)) as f:
        assert f.read().strip() == tb._source_hash()


@pytest.mark.ref
@pytest.mark.skipif(tm.device_count() > 0, reason="a GPU is present (tests/test_zz_gpu_fuzz_regressions.py runs the program there)")
def test_reference_program_links_against_the_library_through_its_scene_class(tmp_path):
    """INTEGRATION.md B, compiled for real: the reference's own main.cpp / maths.cpp / objparser.cpp and its UNMODIFIED scene.h, with
    scene.cpp replaced by oracle/dropin/scene_tmpt.cpp (struct Scene's members over tmpt_scene_create / tmpt_hit_scene).  Here, without
    a GPU: it builds, links libtmpt.so, contains no octree, keeps the reference's command line, loads the .obj with the reference's
    own loader -- and then fails loudly, because the library has no CPU path."""
    from oracle.pyoracle import build_dropin
    exe = build_dropin()
    if exe is None:
        pytest.skip("needs the reference's own sources (a checkout of pr0g/ToyMeshPathTracer named by TMPT_REF), which the repository does not hold")
    assert os.path.exists(exe)
    assert "libtmpt.so" in subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    syms = subprocess.run(["nm", "-C", exe], capture_output=True, text=True).stdout
    assert "HitSceneInternal" not in syms and "OctreeNode::Subdivide" not in syms and "OctreeNode::InternalDivide" not in syms  # scene.cpp is not in it
    assert "U tmpt_hit_scene" in syms and "U tmpt_scene_create" in syms and "Scene::HitScene" in syms
    r = subprocess.run([exe], capture_output=True, text=True)
    assert (r.returncode, r.stdout) == (1, "Usage: TrimeshTracer.exe [width] [height] [samplesPerPixel] [objFile]\n")
    obj = tmp_path / "t.obj"
    obj.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    r = subprocess.run([exe, "8", "8", "1", str(obj)], capture_output=True, text=True, cwd=tmp_path)
    lines = r.stdout.strip().split("\n")
    assert r.returncode == 1 and lines[0].startswith(f"Initialized scene '{obj}' (3 tris) in ")
    assert lines[1].startswith("ERROR: tmpt_scene_create") and "no CPU path" in lines[1]


def test_every_entry_point_survives_null_and_out_of_range_arguments(tmp_path):
    """The C ABI's error behaviour (SURVEY.md 8(b): status codes and tmpt_last_error, never a crash, never an exception across the
    boundary): each entry point called with NULL pointers / negative sizes returns an error status (or 0 rows / 0 pixels for the two
    size helpers, nothing for the two destructors) and leaves a message."""
    L = tm.lib()
    N = None
    buf, out = (C.c_uint8 * 64)(), C.c_void_p()
    f0, f1, one = C.c_float(0), C.c_float(1), C.c_int64(1)
    failing = {
        "tmpt_scene_create (NULL out)": lambda: L.tmpt_scene_create(N, 0, 0, 0, N),
        "tmpt_scene_create (negative count)": lambda: L.tmpt_scene_create(N, -1, 0, 0, C.byref(out)),
        "tmpt_scene_create (NULL triangles)": lambda: L.tmpt_scene_create(N, 5, 0, 0, C.byref(out)),
        "tmpt_scene_get_info": lambda: L.tmpt_scene_get_info(N, N),
        "tmpt_scene_refit": lambda: L.tmpt_scene_refit(N, N, 0, N),
        "tmpt_hit_scene": lambda: L.tmpt_hit_scene(N, N, one, f0, f1, 0, 0, N, N, N, N, N),
        "tmpt_render": lambda: L.tmpt_render(N, N, 1, 1, 1, 0, N, N, N, N),
        "tmpt_progressive_begin": lambda: L.tmpt_progressive_begin(N, 1, 1),
        "tmpt_progressive_pass": lambda: L.tmpt_progressive_pass(N, N, 1, 0, N, N, N, N, N),
        "tmpt_render_stripes": lambda: L.tmpt_render_stripes(N, N, 1, 1, 1, 0, 0, 1, 0, N, N, N, N, N),
        "tmpt_render_multi": lambda: L.tmpt_render_multi(N, 0, N, 1, 1, 1, N, N, N),
        "tmpt_frame_alloc": lambda: L.tmpt_frame_alloc(0, C.c_size_t(0), N, N),
        "tmpt_frame_open": lambda: L.tmpt_frame_open(0, N, N),
        "tmpt_render_stats": lambda: L.tmpt_render_stats(N, N, 1, 1, 1, N),
        "tmpt_hit_scene_stats": lambda: L.tmpt_hit_scene_stats(N, N, one, f0, f1, 0, N),
        "tmpt_load_obj": lambda: L.tmpt_load_obj(N, N, N, N, N),
        "tmpt_write_png (NULL)": lambda: L.tmpt_write_png(N, 1, 1, N, 0),
        "tmpt_write_png (size)": lambda: L.tmpt_write_png(os.fsencode(tmp_path / "x.png"), 0, -1, buf, 0),
        "tmpt_render_kernel_choice": lambda: L.tmpt_render_kernel_choice(N, N, N),
    }
    L.tmpt_last_error.restype = C.c_char_p
    for name, call in failing.items():
        assert call() != tm.TMPT_OK and L.tmpt_last_error(), name
    assert L.tmpt_stripe_rows(-1, 0, 0, 0) == 0 and L.tmpt_local_width(-1, -1, 0) == 0
    L.tmpt_scene_destroy(N)
    L.tmpt_free(N)
    assert L.tmpt_frame_close(0, N) == tm.TMPT_OK and L.tmpt_frame_free(0, N) == tm.TMPT_OK  # nothing to release
    assert L.tmpt_main(0, N) == 1  # the usage line
