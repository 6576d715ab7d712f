"""The render path's work decomposition at the shapes the other GPU tests do not reach, bit for bit against the oracle's restatement:
ragged last chunks under both render kernels (A), a camera beyond the far limit with outputs, progressive and adaptive passes (B),
every forced launch configuration in every output mode (C), partitioned frames split into accumulation bands (D), stream indices
past 2^32 (E), the instrumented passes (F) and the device form of tmpt_hit_scene (G).

Comparisons: rgba and ray count against oracle.render, radiance against its linear mean, normal / depth / triangle against
AovOracle.render_aov, adaptive passes against AdaptiveOracle.pass_; float buffers with the NaN rule of test_gpu_outputs.same_bits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import toymeshpathtracer_b200 as tm
from adaptive_binding import AdaptiveOracle, State
from aov_binding import AovOracle
from conftest import ROOT, bits, load_rays, load_scene, sponza_scene

pytestmark = pytest.mark.gpu
KERNELS = ("0", "1")  # TMPT_RENDER_PATHS: k_render, k_render_paths
CFGS = ("1", "2", "3")  # TMPT_RENDER_CFG: 256 x 4, 512 x 2, 1024 x 1 threads
BUDGET = 4 << 30       # the accumulation buffer's budget (kernels.cu: prepare_accum)


def same_bits(a, b):
    """Float buffers equal bit for bit; NaN where the other has NaN (IEEE 754 fixes no NaN payload, and the GPU's is canonical)."""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    nan = np.isnan(a)
    return (nan == np.isnan(b)).all() and (a.view(np.uint32)[~nan] == b.view(np.uint32)[~nan]).all()


def chunk_len(spp):
    return min(max(spp // 32, 1), 8)  # integ::chunk_len


def band_units(units, unit_width, chunks, planes, granule=4):
    """Rows (or list entries) per accumulation band: the formula of kernels.cu prepare_accum."""
    return min(units, max(granule, (BUDGET // (unit_width * chunks * planes * 16)) & ~(granule - 1)))


def owned_row_to_global(r, stripe, rank, world):
    ls = r // stripe
    return (ls * world + rank) * stripe + (r - ls * stripe)


def scene_data(name):
    if name == "sponza":
        t, mn, mx = sponza_scene()
        return {"tris": t, "bounds_min": mn, "bounds_max": mx}
    return load_scene(name)


def camera(name, w, h):
    sc = scene_data(name)
    return tm.camera_for_scene(f"{name}.obj", sc["bounds_min"], sc["bounds_max"], w, h)


_ORACLE_CACHE = {}


def check_outputs(oracle, aov_oracle, tris, cam, w, h, spp, outs, rays, rows=None, tag=None):
    """rgba, rays, radiance against oracle.render; normal, depth, triangle against the AOV oracle (rows: only those rows)."""
    r0, r1 = rows or (0, h)
    key = (tris.tobytes(), np.asarray(cam, np.float32).tobytes(), w, h, spp, rows)
    if key not in _ORACLE_CACHE:  # (the forced-configuration tests compare three runs with one oracle frame)
        _ORACLE_CACHE[key] = (oracle.render(tris, cam, w, h, spp, rows=rows, linear=True), aov_oracle.render_aov(tris, cam, w, h, spp, rows=rows)[0])
    (oimg, orays, lin), want = _ORACLE_CACHE[key]
    if rows is None:
        assert rays == orays, tag
    assert (outs["rgba"][r0:r1] == oimg[r0:r1]).all(), tag
    assert same_bits(outs["radiance"][r0:r1, :, :3], lin[r0:r1]) and (outs["radiance"][r0:r1, :, 3] == 1.0).all(), tag
    assert (outs["triangle"][r0:r1] == want["triangle"][r0:r1]).all(), tag
    assert same_bits(outs["normal"][r0:r1], want["normal"][r0:r1]), tag
    assert same_bits(outs["depth"][r0:r1], want["depth"][r0:r1]), tag


def run_probe(script, args, env_set, env_pop=(), timeout=1800):
    env = dict(os.environ, **env_set)
    for k in env_pop:
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", script), *args], env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]


@pytest.fixture(scope="module")
def aov_oracle():
    return AovOracle()


@pytest.fixture(scope="module")
def ad_oracle():
    return AdaptiveOracle()


@pytest.fixture(scope="module")
def scenes():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = tm.Scene(scene_data(name)["tris"])
        return cache[name]
    yield get
    for s in cache.values():
        s.close()


# ---- A: ragged last chunks ------------------------------------------------------------------------------------------------------
# spp 65, 100, 191, 255, 257, 1023: chunks of 2, 3, 5, 7, 8, 8 samples whose last chunk holds 1, 1, 1, 3, 1, 7
RAGGED = [("cube", 48, 27, 65), ("suzanne", 32, 18, 100), ("teapot", 16, 9, 191), ("cube", 7, 3, 255), ("suzanne", 16, 9, 257),
          ("teapot", 12, 8, 100), ("cube", 24, 16, 1023), ("triangle", 7, 3, 1023)]
RAGGED_LAST = {65: 1, 100: 1, 191: 1, 255: 3, 257: 1, 1023: 7}


def probe_outputs(tmp_path_factory, tag, env_set, env_pop, cases):
    d = tmp_path_factory.mktemp(tag)
    run_probe("outputs_probe.py", [str(d), *[":".join(map(str, c)) for c in cases]], env_set, env_pop)
    return {c: dict(np.load(d / "{}_{}x{}x{}.npz".format(*c))) for c in cases}


@pytest.fixture(scope="module")
def ragged_runs(tmp_path_factory):
    """Every ragged case through tmpt_render and tmpt_render_outputs, once per forced render kernel (one process each)."""
    return {k: probe_outputs(tmp_path_factory, f"ragged{k}", {"TMPT_RENDER_PATHS": k}, ("TMPT_RENDER_CFG",), RAGGED) for k in KERNELS}


@pytest.mark.parametrize("case", RAGGED, ids=lambda c: "%s_%dx%dx%d" % c)
def test_a_ragged_last_chunk_equals_the_oracle(ragged_runs, oracle, aov_oracle, case):
    """A pixel's last chunk shorter than the others (integ::chunk_start clamps it to spp; k_render_paths counts it down in the low
    byte of its item word): the GPU tests' other spp values are all multiples of their chunk length.  tmpt_render's frame and ray
    count and every output of tmpt_render_outputs equal the oracle's, through k_render and k_render_paths."""
    name, w, h, spp = case
    n = chunk_len(spp)
    assert spp - (spp - 1) // n * n == RAGGED_LAST[spp] < n  # the last chunk is ragged
    tris = scene_data(name)["tris"]
    cam = camera(name, w, h)
    for k in KERNELS:
        z = ragged_runs[k][case]
        assert int(z["kernel"]) == int(k)
        assert int(z["render_rays"]) == int(z["rays"]) and (z["render_rgba"] == z["rgba"]).all(), k
        check_outputs(oracle, aov_oracle, tris, cam, w, h, spp, z, int(z["rays"]), tag=k)


# ---- B: a camera beyond the far limit -------------------------------------------------------------------------------------------
FAR_SIZES, FAR_VFOV = 1.0e5, 0.0012


def far_camera(w, h):
    """suzanne seen from 10^5 scene sizes away, framed by a 0.0012-degree field of view.  Beyond the far limit (16 scene sizes) the
    render kernels' FAR instantiations answer camera rays with the exact scan; out to about 10^4 sizes the padded boxes still give
    the scan's answers for these rays, at 10^5 they do not, so only the FAR instantiations produce the oracle's frame here."""
    sc = load_scene("suzanne")
    mn, mx = sc["bounds_min"].astype(np.float64), sc["bounds_max"].astype(np.float64)
    centre, size = (mn + mx) / 2, float(np.abs(np.concatenate([mn, mx])).max())
    frm = centre + np.array([0.3, 0.5, 1.0]) / np.linalg.norm([0.3, 0.5, 1.0]) * FAR_SIZES * size
    return tm.camera_make(frm, centre, [0, 1, 0], FAR_VFOV, w / h, 0.03, float(np.linalg.norm(frm - centre)))


@pytest.mark.parametrize("spp", [3, 100])
def test_b_far_camera_outputs_equal_the_oracle(scenes, oracle, aov_oracle, spp):
    """tmpt_render_outputs with every output from a camera 10^5 scene sizes away (k_render<..., FAR, Aov>), at one-sample chunks
    and at a ragged spp (100: chunks of 3, the last of 1); rgba and rays are tmpt_render's (FAR, Frame)."""
    w, h = 64, 36
    cam = far_camera(w, h)
    s = scenes("suzanne")
    img, rays, _ = s.render(cam, w, h, spp)
    outs, orays, _ = s.render_outputs(cam, w, h, spp)
    assert orays == rays and (outs["rgba"] == img).all()
    check_outputs(oracle, aov_oracle, load_scene("suzanne")["tris"], cam, w, h, spp, outs, rays)
    assert img[..., :3].std() > 5 and (outs["triangle"] >= 0).mean() > 0.2  # the model fills part of the frame


def test_b_far_camera_progressive_passes(scenes, oracle):
    """Uniform progressive passes from the far camera (34 chunks in passes of 1, 3, 12, 1, 17) equal tmpt_render_outputs at
    272 spp, which equals the oracle: the FAR instantiation with chunk0 > 0 and the running sums."""
    w, h = 32, 18
    cam = far_camera(w, h)
    s = scenes("suzanne")
    want, want_rays, _ = s.render_outputs(cam, w, h, 272, outputs=("rgba", "radiance"))
    oimg, orays, lin = oracle.render(load_scene("suzanne")["tris"], cam, w, h, 272, linear=True)
    assert want_rays == orays and (want["rgba"] == oimg).all() and same_bits(want["radiance"][..., :3], lin)
    s.progressive_begin(w, h)
    total = 0
    for n in (1, 3, 12, 1, 17):
        got, rays, _, spp = s.progressive_pass_outputs(cam, n)
        total += rays
    assert spp == 272 and total == want_rays
    assert (got["rgba"] == want["rgba"]).all() and same_bits(got["radiance"], want["radiance"])
    assert oimg[..., :3].std() > 5


def test_b_far_camera_adaptive_passes(scenes, ad_oracle):
    """An adaptive session from the far camera (k_render<..., FAR, List>) with nonzero tolerances: every pass's rgba, radiance,
    samples, rays and active count equal the adaptive oracle's."""
    w, h = 40, 24
    cam = far_camera(w, h)
    s = scenes("suzanne")
    tris = load_scene("suzanne")["tris"]
    state = State(w, h)
    s.progressive_begin(w, h)
    actives = []
    for n, tol, mn in ((2, 0.0, 2), (2, 1.0, 4), (3, 0.5, 4), (2, 0.25, 5)):
        got, rays, _, active = s.progressive_pass_adaptive(cam, n, tol, mn)
        want, orays, oactive = ad_oracle.pass_(tris, cam, state, n, tol, mn)
        assert (rays, active) == (orays, oactive), (n, tol)
        assert (got["rgba"] == want["rgba"]).all() and same_bits(got["radiance"], want["radiance"]), (n, tol)
        assert (got["samples"] == want["samples"]).all(), (n, tol)
        actives.append(active)
    assert actives[0] == w * h > actives[-1] and len(set(actives)) > 2  # the tolerances stop some pixels


# ---- C: forced launch configurations in every output mode ------------------------------------------------------------------------
CFG_CASES = [("suzanne", 128, 72, 3), ("cube", 7, 3, 33), ("cube", 1, 1, 1), ("teapot", 24, 16, 100), ("cube", 160, 90, 4)]
CFG_STEPS = [["begin"], ["a", 2, 0.0, 2], ["a", 2, 1.0, 4], ["a", 3, 0.5, 4]]
CFG_SESSIONS = [("cube", 64, 36), ("cube", 7, 3)]
CFG_PROG = ("suzanne", 101, 57, 20, ("2", "1", "3"))


@pytest.fixture(scope="module")
def cfg_runs(tmp_path_factory):
    """Per forced configuration, in fresh processes: the outputs cases, the adaptive sessions and a progressive session; and the
    progressive session unforced."""
    spec = tmp_path_factory.mktemp("cfgspec") / "sessions.json"
    spec.write_text(json.dumps([{"name": f"{n}_{w}x{h}", "scene": n, "w": w, "h": h, "steps": CFG_STEPS} for n, w, h in CFG_SESSIONS]))
    name, w, h, spp, passes = CFG_PROG
    runs = {}
    for cfg in CFGS + (None,):
        env, pop = ({"TMPT_RENDER_CFG": cfg}, ()) if cfg else ({}, ("TMPT_RENDER_CFG",))
        d = tmp_path_factory.mktemp(f"cfg{cfg}")
        run_probe("render_probe.py", [name, str(w), str(h), str(spp), str(d / "prog.npz"), *passes], env, pop)
        res = {"prog": dict(np.load(d / "prog.npz"))}
        if cfg:
            res["outputs"] = probe_outputs(tmp_path_factory, f"cfgout{cfg}", env, pop, CFG_CASES)
            run_probe("adaptive_probe.py", [str(d), str(spec)], env, pop)
            res["adaptive"] = {(n, sw, sh): dict(np.load(d / f"{n}_{sw}x{sh}.npz")) for n, sw, sh in CFG_SESSIONS}
        runs[cfg] = res
    return runs


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("case", CFG_CASES, ids=lambda c: "%s_%dx%dx%d" % c)
def test_c_forced_configuration_outputs_equal_the_oracle(cfg_runs, oracle, aov_oracle, cfg, case):
    """TMPT_RENDER_CFG = 1, 2, 3 forces k_render<256, 4>, <512, 2> or <1024, 1> whatever the frame size, so the AOV
    instantiations of the 512-thread configuration run, and the 1024-thread one on frames (7x3, 1x1) with fewer work items than
    one CTA has warps.  rgba, rays and every output equal the oracle's, also at a ragged spp (100)."""
    name, w, h, spp = case
    z = cfg_runs[cfg]["outputs"][case]
    assert int(z["kernel"]) == 0  # a forced configuration runs k_render
    assert int(z["render_rays"]) == int(z["rays"]) and (z["render_rgba"] == z["rgba"]).all()
    check_outputs(oracle, aov_oracle, scene_data(name)["tris"], camera(name, w, h), w, h, spp, z, int(z["rays"]), tag=cfg)


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("name,w,h", CFG_SESSIONS)
def test_c_forced_configuration_adaptive_passes(cfg_runs, ad_oracle, cfg, name, w, h):
    """The List instantiations of each forced configuration (a 7x3 frame is one list tile): every adaptive pass equals the
    adaptive oracle's."""
    res = cfg_runs[cfg]["adaptive"][(name, w, h)]
    tris = load_scene(name)["tris"]
    cam = camera(name, w, h)
    state = State(w, h)
    for i, step in enumerate(CFG_STEPS):
        if step[0] == "begin":
            continue
        want, rays, active = ad_oracle.pass_(tris, cam, state, step[1], step[2], step[3])
        assert (int(res[f"{i}_rays"]), int(res[f"{i}_active"])) == (rays, active), i
        assert (res[f"{i}_rgba"] == want["rgba"]).all() and same_bits(res[f"{i}_radiance"], want["radiance"]), i
        assert (res[f"{i}_samples"] == want["samples"]).all(), i


@pytest.mark.parametrize("cfg", CFGS)
def test_c_forced_configuration_progressive_passes(cfg_runs, cfg):
    """Progressive passes (chunk0 > 0, running sums) under each forced configuration give the unforced session's bytes and rays."""
    got, want = cfg_runs[cfg]["prog"], cfg_runs[None]["prog"]
    assert int(got["kernel"]) == 0
    assert int(got["rays"]) == int(want["rays"]) and (got["img"] == want["img"]).all()


# ---- D: partitioned frames split into bands -------------------------------------------------------------------------------------
BW, BH, BSPP = 10000, 500, 1023  # 128 chunks of 8 samples, the last of 7
PARTITIONS = [(100, 2), (7, 2), (0, 2)]  # (stripe rows, world); 0 = tile interleave


def band_boundaries(units, band):
    return list(range(band, units, band))


@pytest.fixture(scope="module")
def banded(scenes):
    cam = camera("cube", BW, BH)
    s = scenes("cube")
    img, rays, _ = s.render(cam, BW, BH, BSPP)
    outs, orays, _ = s.render_outputs(cam, BW, BH, BSPP)
    return cam, img, rays, outs, orays


def test_d_single_gpu_band_rows_equal_the_oracle(banded, oracle):
    """cube 10000 x 500 at 1023 spp: 128 chunk planes of a 10000-pixel row make bands of 208 rows.  Rows 0 and 499 and the rows
    either side of every band boundary equal the oracle's."""
    cam, img, rays, _, _ = banded
    chunks = -(-BSPP // chunk_len(BSPP))
    band = band_units(BH, BW, chunks, 1)
    assert (chunks, band) == (128, 208)
    tris = load_scene("cube")["tris"]
    for r0, r1 in [(0, 1), (BH - 1, BH)] + [(b - 1, b + 1) for b in band_boundaries(BH, band)]:
        oimg, _ = oracle.render(tris, cam, BW, BH, BSPP, rows=(r0, r1))
        assert (img[r0:r1] == oimg[r0:r1]).all(), (r0, r1)


def test_d_outputs_band_rows_equal_the_oracle(banded, oracle, aov_oracle):
    """The same frame with every output: two plane sets per chunk halve the bands to 104 rows.  Rows 0 and 499 and either side of
    every band boundary equal the oracle's in every output; rgba and rays are tmpt_render's."""
    cam, img, rays, outs, orays = banded
    assert orays == rays and (outs["rgba"] == img).all()
    band = band_units(BH, BW, 128, 2)
    assert band == 104
    tris = load_scene("cube")["tris"]
    for rows in [(0, 1), (BH - 1, BH)] + [(b - 1, b + 1) for b in band_boundaries(BH, band)]:
        check_outputs(oracle, aov_oracle, tris, cam, BW, BH, BSPP, outs, rays, rows=rows, tag=rows)


@pytest.mark.parametrize("stripe,world", PARTITIONS)
def test_d_banded_partitions_compose_to_the_single_gpu_frame(banded, scenes, stripe, world):
    """Each rank's owned rows are banded like a frame's: rank 0 of 100-row stripes owns 300 rows, bands of 208, so a band
    boundary falls at frame row 408, inside a stripe; 7-row stripes cut bands inside stripes too; the tile interleave's local width
    5000 gives bands of 416 rows.  Packed stripes + tmpt_unpack_stripes and the peer-frame form give the single-GPU frame byte for
    byte, with its ray count."""
    import torch
    from toymeshpathtracer_b200 import multigpu
    cam, full, full_rays, _, _ = banded
    s = scenes("cube")
    lw = multigpu.local_width(BW, stripe, world)
    crossings = []
    for r in range(world):
        owned = tm.stripe_rows(BH, stripe, r, world)
        band = band_units(owned, lw, 128, 1)
        crossings += [b if stripe == 0 else owned_row_to_global(b, stripe, r, world) for b in band_boundaries(owned, band)]
    assert crossings  # rank 0 renders more than one band
    if stripe == 100:
        assert 408 in crossings
    if stripe == 0:
        assert lw == 5000 and band_units(BH, lw, 128, 1) == 416
    if stripe > 0:
        assert any(c % stripe for c in crossings)  # a band boundary inside a stripe
    rows, max_rows = multigpu.stripe_plan(BH, stripe, world)
    gathered = torch.zeros((world, max_rows, lw, 4), dtype=torch.uint8, device="cuda")
    rays = torch.zeros(world, dtype=torch.int64, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for r in range(world):
            s.render_stripes(cam, BW, BH, BSPP, stripe, r, world, gathered[r].data_ptr(), rays[r:].data_ptr(), stream=st.cuda_stream)
        frame = torch.empty((BH, BW, 4), dtype=torch.uint8, device="cuda")
        tm._check(tm.lib().tmpt_unpack_stripes(gathered.data_ptr(), BW, BH, stripe, world, 0, frame.data_ptr(), st.cuda_stream))
    st.synchronize()
    assert int(rays.sum()) == full_rays and (frame.cpu().numpy() == full).all()
    frame2 = torch.zeros((BH, BW, 4), dtype=torch.uint8, device="cuda")
    rays.zero_()
    with torch.cuda.stream(st):
        for r in range(world):
            s.render_stripes(cam, BW, BH, BSPP, stripe, r, world, 0, rays[r:].data_ptr(), peer_frame_ptr=frame2.data_ptr(), stream=st.cuda_stream)
    st.synchronize()
    assert int(rays.sum()) == full_rays and (frame2.cpu().numpy() == full).all()


# ---- E: stream indices past 2^32 ------------------------------------------------------------------------------------------------
def test_e_stream_index_past_2_pow_32(scenes, oracle):
    """cube 10000 x 10000 at 350 spp: 44 chunks of 8 samples (the last of 6).  ex::chunk_seed's index chunk * 10^8 + pixel passes
    2^32 inside chunk 42, at pixel 94 967 296 (row 9496, x = 7296), and lies above it for every pixel of chunk 43, so the high word
    of the index seeds those streams.  Bands are 608 rows.  Rows at the frame's edges, either side of the first band boundary and
    around row 9496 equal the oracle's."""
    w = h = 10000
    spp = 350
    chunks = -(-spp // chunk_len(spp))
    assert chunks == 44 and band_units(h, w, chunks, 1) == 608
    assert 42 * w * h < 2 ** 32 <= 42 * w * h + 9496 * w + 7296 and 2 ** 32 - 42 * w * h - 1 == 9496 * w + 7295
    cam = camera("cube", w, h)
    img, rays, sec = scenes("cube").render(cam, w, h, spp)
    print(f"10000x10000x350: {rays} rays in {sec:.2f} s = {rays / sec / 1e6:.0f} Mrays/s")
    assert rays > 2 ** 32
    tris = load_scene("cube")["tris"]
    for row in (0, 607, 608, 9495, 9496, 9497, 9999):
        oimg, _ = oracle.render(tris, cam, w, h, spp, rows=(row, row + 1))
        assert (img[row] == oimg[row]).all(), row


# ---- F: instrumented passes -----------------------------------------------------------------------------------------------------
def render_stats(s, cam, w, h, spp):
    st = np.zeros(tm.STATS_COUNT, np.uint64)
    tm._check(tm.lib().tmpt_render_stats(s.handle, np.ascontiguousarray(cam, np.float32).ctypes.data, w, h, spp, st.ctypes.data))
    return [int(x) for x in st]


STATS_CASES = [("suzanne", 64, 36, 4), ("sponza", 64, 36, 2), ("suzanne", 48, 28, 100), ("far", 64, 36, 3)]


@pytest.mark.parametrize("name,w,h,spp", STATS_CASES)
def test_f_render_stats_count_the_frame_s_rays(scenes, name, w, h, spp):
    """tmpt_render_stats is tmpt_render compiled with work counters: its ray count is the frame's, for an open scene, the closed
    hall, a ragged spp and the camera 10^5 scene sizes away (the instrumented pass must answer far camera rays like the frame, with
    the exact scan).  The counters are consistent (stack-depth histogram monotone, overflows <= rays, lane iterations <= 32 x warp
    iterations), and a frame after the pass has its old bytes."""
    s = scenes("suzanne" if name == "far" else name)
    cam = far_camera(w, h) if name == "far" else camera(name, w, h)
    img, rays, _ = s.render(cam, w, h, spp)
    v = render_stats(s, cam, w, h, spp)
    assert v[0] == rays, (v[0], rays)
    assert all(v[11 + i] >= v[12 + i] for i in range(4)), v[11:16]
    assert v[10] <= v[0] and v[4] <= 32 * v[9] and v[1] > 0
    after, rays2, _ = s.render(cam, w, h, spp)
    assert rays2 == rays and (after == img).all()


@pytest.mark.parametrize("name", ["suzanne", "sponza"])
def test_f_hit_scene_stats_count_rays_and_hits(scenes, name):
    """tmpt_hit_scene_stats on the golden rays, in the CLOSEST, ANY and SUN modes: [0] counts every ray, [3] the hits HitScene
    reports for the same rays."""
    import torch
    rays = np.ascontiguousarray(load_rays(name)["rays"], np.float32)
    s = scenes(name)
    dev = torch.from_numpy(rays).cuda()
    torch.cuda.synchronize()
    for mode in (tm.HIT_CLOSEST, tm.HIT_ANY, tm.HIT_SUN):
        ids = s.HitScene(rays, mode=mode)[0]
        st = np.zeros(tm.STATS_COUNT, np.uint64)
        tm._check(tm.lib().tmpt_hit_scene_stats(s.handle, dev.data_ptr(), len(rays), tm.K_MIN_T, tm.K_MAX_T, mode, st.ctypes.data))
        assert int(st[0]) == len(rays), mode
        assert int(st[3]) == int((ids >= 0).sum()) > 0, mode


# ---- G: tmpt_hit_scene on device buffers ----------------------------------------------------------------------------------------
SUBSETS = [("ids",), ("ids", "t"), ("ids", "pos", "nrm"), ("ids", "t", "pos", "nrm")]
SENTINEL = np.uint32(0xDEADBEEF)


@pytest.mark.parametrize("name", ["suzanne", "sponza"])
def test_g_hit_scene_device_form(scenes, name):
    """TMPT_DEVICE: the golden rays in device memory, the query asynchronous on a non-default stream, each output subset and every
    mode.  ids equal the host form's, t / pos / normal of hits equal its bits, and every slot the query does not answer (rays that
    miss; all of t / pos / normal in the ANY and SUN modes, which report ids only) keeps its pre-filled contents."""
    import torch
    rays = np.ascontiguousarray(load_rays(name)["rays"], np.float32)
    n = len(rays)
    s = scenes(name)
    d_rays = torch.from_numpy(rays).cuda()
    st = torch.cuda.Stream()
    shapes = {"t": (n,), "pos": (n, 3), "nrm": (n, 3)}
    for mode in (tm.HIT_CLOSEST, tm.HIT_ANY, tm.HIT_BRUTE, tm.HIT_SUN):
        hid, ht, hpos, hnrm = s.HitScene(rays, mode=mode)
        host = {"t": ht, "pos": hpos, "nrm": hnrm}
        hit = hid >= 0
        assert hit.any() and (~hit).any(), mode
        for subset in SUBSETS:
            fill = {k: np.full(shapes[k], SENTINEL, np.uint32) for k in subset if k != "ids"}
            dev = {k: torch.from_numpy(v.view(np.int32)).cuda() for k, v in fill.items()}
            dev["ids"] = torch.full((n,), 12345, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            with torch.cuda.stream(st):
                s.hit_scene_device(d_rays.data_ptr(), n, dev["ids"].data_ptr(), *(dev[k].data_ptr() if k in dev else 0 for k in ("t", "pos", "nrm")),
                                   mode=mode, stream=st.cuda_stream)
            st.synchronize()
            assert (dev["ids"].cpu().numpy() == hid).all(), (mode, subset)
            payload = mode in (tm.HIT_CLOSEST, tm.HIT_BRUTE)
            for k in fill:
                got = dev[k].cpu().numpy().view(np.uint32)
                answered = hit if payload else np.zeros(n, bool)
                assert (got[~answered] == SENTINEL).all(), (mode, subset, k)
                if payload:
                    assert (got[answered] == bits(host[k])[answered]).all(), (mode, subset, k)
