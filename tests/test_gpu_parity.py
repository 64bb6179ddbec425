"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): pyramid pixels, keypoint sets, octaves, responses and descriptors bit-exact; angles
within 1e-4 rad; uRight / depth within 1e-3 px.  Descriptor bit flips may only come from last-ulp libm differences
(CUDA vs glibc atan2/sin/cos) landing on a rounding tie; they are counted and bounded.
"""
import hashlib
import os

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

pytestmark = pytest.mark.gpu

ANGLE_TOL_DEG = np.degrees(1e-4)


def _camera(c):
    return api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], tuple(c["dist"]), c["depth_scale"])


def _cmp_kps(got, exp, got_desc, exp_desc, what=""):
    assert len(got) == len(exp), f"{what}: {len(got)} vs {len(exp)} keypoints"
    for f in ("x", "y", "size", "response", "octave", "class_id"):
        assert np.array_equal(got[f], exp[f]), f"{what}: field {f}"
    dang = np.abs(got["angle"] - exp["angle"])
    dang = np.minimum(dang, 360.0 - dang)
    assert dang.max(initial=0.0) <= ANGLE_TOL_DEG, f"{what}: max angle error {dang.max()} deg"
    flips = int(np.unpackbits(got_desc ^ exp_desc).sum())
    # a flip needs a 1-ulp libm difference to cross a float rounding boundary or a .5 tie: expect none, tolerate a trace
    assert flips <= 2, f"{what}: {flips} descriptor bit flips"
    return flips, int((got["angle"] != exp["angle"]).sum())


CONFIGS = [
    ("K2000", 376, 1241, 2000, 8, 1.2, 0),
    ("K500", 376, 1241, 500, 8, 1.2, 1),
    ("K4000", 376, 1241, 4000, 8, 1.2, 2),
    ("T1000", 480, 640, 1000, 8, 1.2, 3),
    ("H5000", 1080, 1920, 5000, 12, 1.2, 4),
    ("S300x5", 240, 320, 300, 5, 1.3, 5),
    ("odd", 333, 517, 700, 6, 1.25, 6),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_extract_matches_oracle(oracle, cfg):
    name, h, w, nf, nl, sc, seed = cfg
    img = synth.synth_image(h, w, seed)
    ctx = api.Context(w, h, nf, nl, sc)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, nf, nl, sc)
    # pyramid and blurred pyramid: every pixel
    for blurred in (False, True):
        levels = ctx.get_pyramid(0, blurred)
        for l in range(nl):
            exp = e.pyr.blurred(l) if blurred else e.pyr.level(l)
            assert np.array_equal(levels[l], exp), f"{name} level {l} blurred={blurred}"
    for l in range(nl):
        lw, lh, sf, q = ctx.level_info(l)
        assert (lw, lh, q) == (e.pyr.w[l], e.pyr.h[l], e.pyr.quota[l]) and sf == e.pyr.sf[l]
    flips, inexact = _cmp_kps(kps, e.kps, desc, e.desc, name)
    print(f"{name}: {len(kps)} kps, {flips} bit flips, {inexact} angles differing in the last float ulp")
    ctx.close()


@pytest.mark.parametrize("kind", ["texture", "noise", "lowcontrast"])
def test_fast_and_quadtree_stages_match_oracle(oracle, kind):
    """stage-level parity: the per-level FAST corner lists (detection order, scores) and the quadtree survivors"""
    if kind == "texture":
        img = synth.synth_image(376, 1241, 7)
    elif kind == "noise":
        img = np.random.default_rng(3).integers(0, 256, (376, 1241), dtype=np.uint8)
    else:
        img = (synth.synth_image(376, 1241, 8).astype(np.float32) * 0.3 + 80).astype(np.uint8)
    ctx = api.Context(1241, 376, 2000, 8, 1.2)
    ctx.extract(img)
    e = oracle.extract(img)
    for l in range(8):
        got = ctx.level_corners(0, l)
        exp, _ = oracle.fast_cells(e.pyr.level(l))
        assert np.array_equal(got, exp), f"{kind}: FAST list of level {l}: {len(got)} vs {len(exp)}"
        w, h, _, quota = ctx.level_info(l)
        idx, _ = oracle.quadtree_select(w - 32, h - 32, exp[:, 0].astype(np.float32), exp[:, 1].astype(np.float32), exp[:, 2].astype(np.float32), quota)
        sel = ctx.level_selected(0, l)
        assert np.array_equal(sel, exp[idx] + np.array([16, 16, 0], np.int32)), f"{kind}: quadtree survivors of level {l}"
    ctx.close()


def test_random_configurations(oracle):
    """seeded sweep over image sizes (not multiples of any tile), level counts, scale factors, quotas and thresholds"""
    rng = np.random.default_rng(2024)
    done = 0
    for trial in range(60):
        w, h = int(rng.integers(80, 900)), int(rng.integers(80, 700))
        nl = int(rng.integers(1, 9))
        sc = float(np.float32(rng.uniform(1.1, 1.6)))
        nf = int(rng.integers(20, 3000))
        ini, mn = int(rng.integers(8, 40)), int(rng.integers(2, 12))
        rc, lw, lh = oracle.level_sizes(w, h, sc, nl)
        if rc != 0 or min(lw[-1], lh[-1]) < 62:
            with pytest.raises(api.ImageSizeError):
                api.Context(w, h, nf, nl, sc, ini, mn)
            continue
        img = synth.synth_image(h, w, 1000 + trial)
        if trial % 4 == 0:
            img = np.ascontiguousarray(np.pad(img, ((0, 0), (0, 13)))[:, :w + 13])[:, :w]  # non-contiguous rows (stride != width)
        ctx = api.Context(w, h, nf, nl, sc, ini, mn)
        kps, desc = ctx.extract(img)
        e = oracle.extract(img, nf, nl, sc, ini, mn)
        _cmp_kps(kps, e.kps, desc, e.desc, f"trial {trial}: {w}x{h} L{nl} s{sc:.3f} N{nf} th{ini}/{mn}")
        lv = ctx.get_pyramid(0, True)
        assert np.array_equal(lv[-1], e.pyr.blurred(nl - 1))
        ctx.close()
        done += 1
    assert done >= 30


@pytest.mark.parametrize("cfg", [(640, 480, 3, 2.0), (642, 481, 3, 2.0), (900, 600, 3, 3.0), (400, 300, 8, 1.05), (1280, 720, 4, 2.0)],
                         ids=["2x-even", "2x-odd", "3x", "1.05x", "2x-720p"])
def test_exact_decimation_and_extreme_scale_factors(oracle, cfg):
    """scale 2 on even sizes takes cv::resize's INTER_AREA re-route for level 1 (exact 2x2 means) while level 2 (4x) stays
    bilinear; odd sizes and other factors stay bilinear throughout"""
    w, h, nl, sc = cfg
    img = synth.synth_image(h, w, 77)
    ctx = api.Context(w, h, 800, nl, sc)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, 800, nl, sc)
    _cmp_kps(kps, e.kps, desc, e.desc, str(cfg))
    for l, (a, b) in enumerate(zip(ctx.get_pyramid(0), [e.pyr.level(i) for i in range(nl)])):
        assert np.array_equal(a, b), f"level {l}"
    for l, (a, b) in enumerate(zip(ctx.get_pyramid(0, True), [e.pyr.blurred(i) for i in range(nl)])):
        assert np.array_equal(a, b), f"blurred level {l}"
    ctx.close()


@pytest.mark.parametrize("no_tma", [False, True], ids=["tma-staged", "l2-gather"])
def test_resize_source_paths_agree(oracle, monkeypatch, no_tma):
    """levels 1-3 of the 1.2 pyramid take their level-0 source rectangle through a TMA box load, the others (and every level with
    ORBX_PYR_NO_TMA set, read at context creation) gather the same taps from L2: both must give the reference's pixels"""
    if no_tma:
        monkeypatch.setenv("ORBX_PYR_NO_TMA", "1")
    w, h, nl = 1241, 376, 8
    img = synth.synth_image(h, w, 31)
    strided = np.ascontiguousarray(np.pad(img, ((0, 0), (0, 7))))[:, :w]  # rows at an odd stride (1248), like a caller's ROI
    ctx = api.Context(w, h, 2000, nl, 1.2)
    ctx.extract(strided)
    e = oracle.extract(img, 2000, nl, 1.2)
    for l in range(nl):
        assert np.array_equal(ctx.get_pyramid(0)[l], e.pyr.level(l)), f"level {l}"
        assert np.array_equal(ctx.get_pyramid(0, True)[l], e.pyr.blurred(l)), f"blurred level {l}"
    ctx.close()


def test_degenerate_images(oracle):
    ctx = api.Context(320, 240, 1000, 4, 1.2)
    kps, desc = ctx.extract(np.zeros((240, 320), np.uint8))
    assert len(kps) == 0
    kps, desc = ctx.extract(np.full((240, 320), 255, np.uint8))
    assert len(kps) == 0
    # uniform noise: tens of thousands of corners per level
    img = np.random.default_rng(1).integers(0, 256, (240, 320), dtype=np.uint8)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, 1000, 4, 1.2)
    _cmp_kps(kps, e.kps, desc, e.desc, "noise")
    ctx.close()


def test_dense_level_uses_global_quadtree_path(oracle):
    """more corners on a level than the shared-memory list holds (4096) -> the global-scratch path of the quadtree"""
    img = np.random.default_rng(2).integers(0, 256, (376, 1241), dtype=np.uint8)
    ctx = api.Context(1241, 376, 2000, 8, 1.2)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, 2000, 8, 1.2)
    fc, _ = oracle.fast_cells(e.pyr.level(0))
    assert len(fc) > 4096
    _cmp_kps(kps, e.kps, desc, e.desc, "dense")
    ctx.close()


def test_starved_level_returns_zero(oracle):
    img = np.full((240, 320), 128, np.uint8)
    img[60:180, 80:240] = synth.synth_image(120, 160, 11)
    ctx = api.Context(320, 240, 3000, 3, 1.2)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, 3000, 3, 1.2)
    assert (e.level_counts == 0).any()
    _cmp_kps(kps, e.kps, desc, e.desc, "starved")
    ctx.close()


def test_fallback_threshold_cells(oracle):
    """low-contrast image: most cells only produce corners at minThFAST"""
    img = (synth.synth_image(240, 320, 21).astype(np.float32) * 0.25 + 90).astype(np.uint8)
    _, nfb = oracle.fast_cells(img)
    assert nfb > 10
    ctx = api.Context(320, 240, 500, 3, 1.2)
    kps, desc = ctx.extract(img)
    e = oracle.extract(img, 500, 3, 1.2)
    _cmp_kps(kps, e.kps, desc, e.desc, "fallback")
    ctx.close()


def test_errors():
    with pytest.raises(api.ImageSizeError):
        api.Context(100, 60, 500, 8, 1.2)
    with pytest.raises(api.ImageSizeError):
        api.Context(60, 60, 100, 1, 1.2)  # one level, but no room for a 30-px FAST cell
    with pytest.raises(api.FileNotOpenError):
        api.ORBExtractor(np.zeros((240, 320), np.uint8), 500, 4, 1.2, "/nonexistent/brief_template.txt", 20, 7)
    ctx = api.Context(320, 240, 500, 4, 1.2, max_batch=2)
    import torch

    d = torch.zeros((3, 240, 320), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):  # device-resident batches are limited by max_batch (host sequences are not)
        ctx.stereo_batch_device(3, d.data_ptr(), d.data_ptr(), 320, 320 * 240)
    ctx.close()


STEREO = [
    ("K2000_d17", synth.KITTI, 2000, 0, 17),
    ("K2000_d5", synth.KITTI, 2000, 1, 5),
    ("K1000_d63", synth.KITTI, 1000, 2, 63),
    ("K500_d42", synth.KITTI, 500, 5, 42),    # BASELINE.json configs[3]: 500/1000/2000/4000 features
    ("K4000_d17", synth.KITTI, 4000, 6, 17),
    ("T1000_d17", synth.TUM, 1000, 3, 17),
    ("H5000_d42", synth.HD, 5000, 4, 42),
]


@pytest.mark.parametrize("cfg", STEREO, ids=[c[0] for c in STEREO])
def test_stereo_matches_oracle(oracle, cfg):
    name, c, nf, seed, disp = cfg
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])  # zero distortion
    left, right = synth.synth_stereo_pair(c["height"], c["width"], seed, disp)
    ctx = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam)
    r = ctx.stereo_frame(left, right)
    el = oracle.extract(left, nf, c["n_levels"], c["scale_factor"])
    er = oracle.extract(right, nf, c["n_levels"], c["scale_factor"])
    _cmp_kps(r.kps_left, el.kps, r.desc_left, el.desc, name + " left")
    _cmp_kps(r.kps_right, er.kps, r.desc_right, er.desc, name + " right")
    nm, ur, dp, _ = oracle.search_by_stereo(el, er, np.float32(c["fx"]), cam.bf)
    assert r.n_matches == nm and nm > 0.3 * len(el.kps)
    assert np.array_equal(r.u_right >= 0, ur >= 0)
    assert np.abs(r.u_right - ur).max() <= 1e-3 and np.abs(r.depth - dp).max() <= 1e-3 * np.abs(dp).max()
    print(f"{name}: {nm} matches, exact uRight {np.array_equal(r.u_right, ur)}, exact depth {np.array_equal(r.depth, dp)}")
    # right pyramid is retrievable too (Frame::getRightPyramid)
    assert np.array_equal(ctx.get_pyramid(1)[1], er.pyr.level(1))
    ctx.close()


# the reference's outputs for the two pairs below: kitti_stereo_seed0_d17 comes from libref.so (scripts/make_golden.py),
# tum_stereo_seed3_d17 from the restatement, which tests/test_oracle_vs_ref.py::test_stereo_identical held identical to it
REF_FIXTURES = {"K2000_d17": "kitti_stereo_seed0_d17.npz", "T1000_d17": "tum_stereo_seed3_d17.npz"}


@pytest.mark.parametrize("cfg", [STEREO[0], STEREO[5]], ids=["K2000_d17", "T1000_d17"])
def test_stereo_matches_the_compiled_reference(oracle, have_ref, template_path, cfg):
    """the CUDA path against the reference's own outputs, not through the restatement: oracle/_ref/libref.so directly where
    it is built (the reference's ORBExtractor.cc / ORBMatcher.cc translation units), the stored fixture otherwise"""
    name, c, nf, seed, disp = cfg
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    left, right = synth.synth_stereo_pair(c["height"], c["width"], seed, disp)
    if have_ref:
        oracle.ref_reset()
        bf = oracle.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)
        ref = oracle.ref_stereo(left, right, template_path, nf, c["n_levels"], c["scale_factor"])
        assert ref["status"] == 0 and float(cam.bf) == float(bf)
    else:
        ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", REF_FIXTURES[name]))
        assert (int(ref["seed"]), int(ref["disparity"])) == (seed, disp)
        assert [hashlib.sha256(a.tobytes()).hexdigest() for a in (left, right)] == [str(ref["left_sha"]), str(ref["right_sha"])]
    ctx = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam)
    r = ctx.stereo_frame(left, right)
    _cmp_kps(r.kps_left, ref["kl"], r.desc_left, ref["dl"], name + " left vs reference")
    _cmp_kps(r.kps_right, ref["kr"], r.desc_right, ref["dr"], name + " right vs reference")
    assert r.n_matches == int(ref["n_matches"])
    assert np.abs(r.u_right - ref["u_right"]).max() <= 1e-3 and np.abs(r.depth - ref["depth"]).max() <= 1e-3 * np.abs(ref["depth"]).max()
    ctx.close()


def test_stereo_with_distortion_uses_undistorted_left(oracle):
    """Frame.cc:106 undistorts the left keypoints before searchByStereo; mild distortion keeps SAD windows inside"""
    c = synth.KITTI
    dist = (0.02, -0.01, 0.0005, -0.0003, 0.0)
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], dist)
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 8, 17)
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam)
    r = ctx.stereo_frame(left, right)
    el, er = oracle.extract(left, 1000), oracle.extract(right, 1000)
    kl_u = el.kps.copy()
    xy = oracle.undistort_points(np.stack([el.kps["x"], el.kps["y"]], 1), c["fx"], c["fy"], c["cx"], c["cy"], np.array(dist[:4], np.float32))
    kl_u["x"], kl_u["y"] = xy[:, 0], xy[:, 1]
    assert np.abs(r.kps_left["x"] - kl_u["x"]).max() <= 1e-3 and np.abs(r.kps_left["y"] - kl_u["y"]).max() <= 1e-3
    # feed the oracle the device's undistorted coordinates so the comparison isolates the matcher
    nm, ur, dp, _ = oracle.search_by_stereo(el, er, np.float32(c["fx"]), cam.bf, kps_left_undist=r.kps_left)
    assert r.n_matches == nm
    assert np.abs(r.u_right - ur).max() <= 1e-3
    ctx.close()


@pytest.mark.parametrize("use_dist", [False, True], ids=["nodist", "tumdist"])
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
def test_rgbd_matches_oracle(oracle, use_dist, dtype):
    c = synth.TUM
    dist = tuple(c["dist"]) if use_dist else (0.0,) * 5
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], dist, c["depth_scale"])
    gray = synth.synth_image(c["height"], c["width"], 12)
    depth = synth.synth_depth_u16(c["height"], c["width"], 12, c["depth_scale"])
    if dtype == np.float32:
        depth = depth.astype(np.float32)
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam)
    r = ctx.rgbd_frame(gray, depth)
    e = oracle.extract(gray, 1000, 8, 1.2)
    _cmp_kps(r.kps_raw, e.kps, r.desc, e.desc, "rgbd")
    ku = e.kps.copy()
    if use_dist:
        xy = oracle.undistort_points(np.stack([e.kps["x"], e.kps["y"]], 1), c["fx"], c["fy"], c["cx"], c["cy"], np.array(dist, np.float32))
        ku["x"], ku["y"] = xy[:, 0], xy[:, 1]
        assert np.abs(r.kps["x"] - e.kps["x"]).max() > 0.5  # distortion is not a no-op
    assert np.abs(r.kps["x"] - ku["x"]).max() <= 1e-3 and np.abs(r.kps["y"] - ku["y"]).max() <= 1e-3
    ur, dp = oracle.rgbd_lookup(depth, c["depth_scale"], e.kps, ku, cam.bf)
    assert np.array_equal(r.depth, dp)
    assert np.abs(r.u_right - ur).max() <= 1e-3
    assert 0.05 < (dp < 0).mean() < 0.2  # ~10 % invalid depth pixels
    ctx.close()


def test_sequence_sharded_batches_equal_oracle(oracle):
    """BASELINE.json configs[2] in miniature: a frame sequence split into per-rank blocks (shard.frame_range), each block
    run through the batch call; every frame's descriptors must equal the oracle's regardless of its position in a batch"""
    from orb_slam2_ros2_b200 import shard

    c = synth.KITTI
    F, R, B = 11, 2, 4
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], F, seed0=70)
    ctx = api.Context(c["width"], c["height"], 500, 8, 1.2, camera=_camera(c), max_batch=B)
    got_desc = np.zeros((F, 500, 32), np.uint8)
    got_n = np.zeros(F, np.int32)
    got_nm = np.zeros(F, np.int32)
    for rank in range(R):
        frames = list(shard.frame_range(F, rank, R))
        for i in range(0, len(frames), B):
            blk = frames[i : i + B]
            ob = ctx.stereo_batch(lefts[blk[0] : blk[-1] + 1], rights[blk[0] : blk[-1] + 1])
            got_desc[blk] = ob.desc_left
            got_n[blk] = ob.n_left
            got_nm[blk] = ob.n_matches
    for f in (0, 5, 10):
        el, er = oracle.extract(lefts[f], 500), oracle.extract(rights[f], 500)
        assert got_n[f] == len(el.kps) and np.array_equal(got_desc[f, : got_n[f]], el.desc)
        nm, _, _, _ = oracle.search_by_stereo(el, er, np.float32(c["fx"]), _camera(c).bf)
        assert got_nm[f] == nm
    ctx.close()


def test_init_grid_matches_restatement(oracle):
    """VirtualFrame::initGrid (Frame.cc:53-69) for a stereo frame (KITTI, no distortion) and an RGB-D frame (TUM distortion)"""
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 4, 17)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=_camera(c))
    r = ctx.stereo_frame(left, right)
    rows, cols, mnu, mnv, mxu, mxv = ctx.grid_info()
    assert (rows, cols, mnu, mnv, mxu, mxv) == (8, 20, 0.0, 0.0, 1241.0, 376.0)
    got, exp = ctx.get_grid(0), oracle.init_grid(r.kps_left, mnu, mnv, mxu, mxv)
    assert sum(len(x) for row in got for x in row) == len(r.kps_left)
    for i in range(rows):
        for j in range(cols):
            assert np.array_equal(got[i][j], exp[i][j]), (i, j)
    ctx.close()

    c = synth.TUM
    cam = _camera(c)
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam)
    rg = ctx.rgbd_frame(synth.synth_image(c["height"], c["width"], 12), synth.synth_depth_u16(c["height"], c["width"], 12, c["depth_scale"]))
    rows, cols, mnu, mnv, mxu, mxv = ctx.grid_info()
    b = oracle.undistort_points(np.array([[0, 0], [c["width"], c["height"]]], np.float32), c["fx"], c["fy"], c["cx"], c["cy"], np.array(c["dist"], np.float32))
    assert np.abs(np.array([mnu, mnv, mxu, mxv]) - b.reshape(-1)).max() <= 1e-3
    got, exp = ctx.get_grid(0), oracle.init_grid(rg.kps, mnu, mnv, mxu, mxv)
    assert len(got) == len(exp) and len(got[0]) == len(exp[0])
    for i in range(rows):
        for j in range(cols):
            assert np.array_equal(got[i][j], exp[i][j]), (i, j)
    ctx.close()


def test_long_sequence_streams_through_the_slots(oracle):
    """a host sequence longer than max_batch: every frame's results equal the single-frame results"""
    c = synth.KITTI
    cam = _camera(c)
    n = 37
    base_l, base_r = synth.synth_stereo_pool(c["height"], c["width"], 5, seed0=90)
    order = np.arange(n) % 5
    lefts, rights = np.ascontiguousarray(base_l[order]), np.ascontiguousarray(base_r[order])
    ctx = api.Context(c["width"], c["height"], 800, 8, 1.2, camera=cam, max_batch=16)  # 2 slots of 8 frames
    ob = ctx.stereo_batch(lefts, rights)
    one = api.Context(c["width"], c["height"], 800, 8, 1.2, camera=cam, max_batch=1)
    ref = [one.stereo_frame(base_l[i], base_r[i]) for i in range(5)]
    for f in range(n):
        r = ref[order[f]]
        a = ob.n_left[f]
        assert (a, ob.n_right[f], ob.n_matches[f]) == (len(r.kps_left), len(r.kps_right), r.n_matches), f
        assert np.array_equal(ob.kps_left[f, :a].view(np.uint8), r.kps_left.view(np.uint8))
        assert np.array_equal(ob.desc_left[f, :a], r.desc_left) and np.array_equal(ob.desc_right[f, : ob.n_right[f]], r.desc_right)
        assert np.array_equal(ob.u_right[f, :a], r.u_right) and np.array_equal(ob.depth[f, :a], r.depth)
    ctx.close()
    one.close()


def test_batch_equals_single_frames(oracle):
    c = synth.KITTI
    cam = _camera(c)
    n = 5
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=30)
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam, max_batch=8)
    ob = ctx.stereo_batch(lefts, rights)
    one = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam, max_batch=1)
    for f in range(n):
        r = one.stereo_frame(lefts[f], rights[f])
        a, b = ob.n_left[f], ob.n_right[f]
        assert (a, b, ob.n_matches[f]) == (len(r.kps_left), len(r.kps_right), r.n_matches)
        assert np.array_equal(ob.kps_left[f, :a].view(np.uint8), r.kps_left.view(np.uint8))
        assert np.array_equal(ob.kps_right[f, :b].view(np.uint8), r.kps_right.view(np.uint8))
        assert np.array_equal(ob.desc_left[f, :a], r.desc_left) and np.array_equal(ob.desc_right[f, :b], r.desc_right)
        assert np.array_equal(ob.u_right[f, :a], r.u_right) and np.array_equal(ob.depth[f, :a], r.depth)
    # and one frame against the oracle
    el, er = oracle.extract(lefts[2], 1000), oracle.extract(rights[2], 1000)
    _cmp_kps(ob.kps_left[2, : ob.n_left[2]], el.kps, ob.desc_left[2, : ob.n_left[2]], el.desc, "batch left")
    ctx.close()
    one.close()


def test_device_batch_and_launch_count():
    import torch

    c = synth.KITTI
    n = 4
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=50)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=_camera(c), max_batch=n)
    host = ctx.stereo_batch(lefts, rights)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    before = ctx.launch_count
    res = ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    assert ctx.launch_count - before == 7  # pyramid level 0, pyramid levels >= 1 (+blur), FAST, quadtree, orientation+BRIEF, frame index (row index + grid), stereo (one chunk: n <= 8)
    nm = ctx.read_device(res.n_matches, (n,), np.int32)
    assert np.array_equal(nm, host.n_matches) and (nm > 500).all()
    desc = ctx.read_device(res.desc, (2 * n, 2000, 32), np.uint8)
    assert np.array_equal(desc[0::2], host.desc_left) and np.array_equal(desc[1::2], host.desc_right)
    ur = ctx.read_device(res.u_right, (n, 2000), np.float64)
    assert np.array_equal(ur, host.u_right)
    ctx.set_stream(None)
    ctx.close()


def test_reference_shaped_classes(oracle, template_path):
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 0, 17)
    ex = api.ORBExtractor(left, 2000, 8, 1.2, template_path, 20, 7)
    kps, desc = ex.extract()
    e = oracle.extract(left)
    _cmp_kps(kps, e.kps, desc, e.desc, "ORBExtractor")
    assert np.array_equal(ex.getScaledFactors(), e.pyr.sf)
    assert np.array_equal(ex.getPyramid()[3], e.pyr.level(3))
    f = api.Frame.createStereo(left, right, 2000, template_path, 20, 7, None, 8, 1.2, camera=_camera(c))
    assert f.mnN == int((f.mvDepths > 0).sum()) and f.mnN > 1000
