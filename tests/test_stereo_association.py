"""Stereo association (stereo_kernel, the port of ORBMatcher::searchByStereo, src/ORBMatcher.cc:18-81,841-1011) held
bit for bit, on scenes that reach every branch of the search.

CPU: a literal Python restatement (tests/stereo_restatement.py) equals oracle_search_by_stereo on every scene of
tests/stereo_scenes.py and on the constant-disparity pairs of synth.synth_stereo_pair, with and without lens
distortion; a census over the scenes shows that each branch and each tie / boundary case is reached; the oracle equals
the compiled reference where oracle/_ref/libref.so is built.
GPU: the kernel, fed its own keypoints and descriptors, equals the oracle fed the same ones: match count, uRight and
depth as float64 arrays with np.array_equal.  The oracle is compiled with -ffp-contract=off and the kernel rounds
every float / double step with an explicit _rn intrinsic, so equality is the bar.
"""
from collections import Counter

import numpy as np
import pytest

import stereo_restatement as SR
import stereo_scenes as SS
from orb_slam2_ros2_b200 import api, synth

BARREL = (-0.15, 0.0, 0.0, 0.0, 0.0)
STRONG_BARREL = (-0.3, 0.1, 0.0, 0.0, 0.0)
MILD_BARREL = (-0.05, 0.0, 0.0, 0.0, 0.0)  # undistorted keypoints stay inside the image and their windows inside the levels

# (name, camera config, features, seed, distortion of the left view, fx of the search or None for the config's)
SCENES = [
    ("K500", synth.KITTI, 500, 1, None, None),
    ("K2000", synth.KITTI, 2000, 0, None, None),
    ("K4000", synth.KITTI, 4000, 2, None, None),
    ("T2000", synth.TUM, 2000, 3, None, None),
    ("H5000", synth.HD, 5000, 4, None, None),
    ("K2000_fx60", synth.KITTI, 2000, 5, None, 60.0),  # fx below the scene's largest disparity: minU rejects true matches
    ("K2000_barrel", synth.KITTI, 2000, 6, BARREL, None),
    ("T2000_barrel", synth.TUM, 2000, 7, STRONG_BARREL, None),
    ("K4000_barrel", synth.KITTI, 4000, 9, STRONG_BARREL, None),
    ("K2000_mild", synth.KITTI, 2000, 8, MILD_BARREL, None),
]

# the constant-disparity pairs the rest of the suite uses (tests/test_gpu_parity.py::STEREO)
PAIRS = [
    ("K2000_d17", synth.KITTI, 2000, 0, 17),
    ("K2000_d5", synth.KITTI, 2000, 1, 5),
    ("K1000_d63", synth.KITTI, 1000, 2, 63),
    ("K500_d42", synth.KITTI, 500, 5, 42),
    ("K4000_d17", synth.KITTI, 4000, 6, 17),
    ("T1000_d17", synth.TUM, 1000, 3, 17),
    ("H5000_d42", synth.HD, 5000, 4, 42),
]


def _camera(c, dist=None, fx=None):
    return api.Camera(fx or c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], tuple(dist or (0.0,) * 5))


_scene_cache = {}


def scene_images(cfg):
    name, c, nf, seed, dist, fx = cfg
    if name not in _scene_cache:
        left, right, _ = SS.render(SS.make_scene(name, c["height"], c["width"], seed), c, dist)
        _scene_cache[name] = (left, right)
    return _scene_cache[name]


def _undistorted(oracle, kps, c, dist):
    if dist is None:
        return kps
    ku = kps.copy()
    xy = oracle.undistort_points(np.stack([kps["x"], kps["y"]], 1), c["fx"], c["fy"], c["cx"], c["cy"], np.array(dist, np.float32))
    ku["x"], ku["y"] = xy[:, 0], xy[:, 1]
    return ku


def _restate(el, er, kl, c, fx, bf):
    nl = c["n_levels"]
    return SR.search_by_stereo([el.pyr.level(l) for l in range(nl)], [er.pyr.level(l) for l in range(nl)], el.pyr.sf, kl, el.desc, er.kps, er.desc,
                               fx, bf, c["width"], c["height"])


def _same(r, nm, ur, dp, mi=None):
    return (r["n_matches"] == nm and np.array_equal(r["u_right"], ur) and np.array_equal(r["depth"], dp)
            and (mi is None or np.array_equal(r["match_idx"], mi)))


# ---- CPU ------------------------------------------------------------------------------------------------------------
_census = {}


@pytest.mark.parametrize("cfg", SCENES, ids=[s[0] for s in SCENES])
def test_restatement_equals_oracle_on_scenes(oracle, cfg):
    name, c, nf, seed, dist, fx = cfg
    left, right = scene_images(cfg)
    el = oracle.extract(left, nf, c["n_levels"], c["scale_factor"])
    er = oracle.extract(right, nf, c["n_levels"], c["scale_factor"])
    cam = _camera(c, dist, fx)
    kl = _undistorted(oracle, el.kps, c, dist)
    nm, ur, dp, mi = oracle.search_by_stereo(el, er, np.float32(cam.fx), cam.bf, kps_left_undist=kl)
    r = _restate(el, er, kl, c, np.float32(cam.fx), cam.bf)
    assert _same(r, nm, ur, dp, mi), name
    assert nm > 0.25 * len(kl)
    _census[name] = r["census"]


@pytest.mark.parametrize("dist", [None, BARREL], ids=["nodist", "barrel"])
@pytest.mark.parametrize("cfg", PAIRS, ids=[p[0] for p in PAIRS])
def test_restatement_equals_oracle_on_constant_disparity_pairs(oracle, cfg, dist):
    """the images are undistorted here; distorting the left keypoints still moves them, and their windows, outside"""
    name, c, nf, seed, disp = cfg
    left, right = synth.synth_stereo_pair(c["height"], c["width"], seed, disp)
    el = oracle.extract(left, nf, c["n_levels"], c["scale_factor"])
    er = oracle.extract(right, nf, c["n_levels"], c["scale_factor"])
    cam = _camera(c, dist)
    kl = _undistorted(oracle, el.kps, c, dist)
    nm, ur, dp, mi = oracle.search_by_stereo(el, er, np.float32(cam.fx), cam.bf, kps_left_undist=kl)
    r = _restate(el, er, kl, c, np.float32(cam.fx), cam.bf)
    assert _same(r, nm, ur, dp, mi), name


# Measured over SCENES: row_outside 60, no_candidate 1395, dist_gt_75 11404, octave_mismatch 2037, window_outside 50,
# sad_edge 1640, parabola 8649, fallback 265, hamming_tie 2060, sad_tie 578, minU_excluded_better 1676, dist_eq_75 387,
# x_eq_maxU 2848.  The minimums sit at a quarter to a third of that, so that other seeds or a retuned layer still pass.
CENSUS_MIN = {
    "row_outside": 15, "no_candidate": 400, "dist_gt_75": 3500, "octave_mismatch": 600, "window_outside": 12, "sad_edge": 500,
    "parabola": 2800, "fallback": 70, "hamming_tie": 600, "sad_tie": 150, "minU_excluded_better": 500, "dist_eq_75": 100, "x_eq_maxU": 800,
}


def test_census_reaches_every_branch(oracle):
    """every outcome the search can reach, and both sides of its two strict comparisons, on the scene set; the constant-
    disparity pairs alone do not reach them"""
    for cfg in SCENES:
        if cfg[0] not in _census:
            test_restatement_equals_oracle_on_scenes(oracle, cfg)
    total = sum((_census[s[0]] for s in SCENES), Counter())
    print("census over the scenes:", dict(total))
    for k, lo in CENSUS_MIN.items():
        assert total[k] >= lo, f"{k}: {total[k]} < {lo}"
    assert set(CENSUS_MIN) == set(SR.OUTCOMES + SR.COUNTERS)
    pairs = Counter()
    for p in PAIRS:
        left, right = synth.synth_stereo_pair(p[1]["height"], p[1]["width"], p[3], p[4])
        el = oracle.extract(left, p[2], p[1]["n_levels"], p[1]["scale_factor"])
        er = oracle.extract(right, p[2], p[1]["n_levels"], p[1]["scale_factor"])
        cam = _camera(p[1])
        pairs += _restate(el, er, el.kps, p[1], np.float32(cam.fx), cam.bf)["census"]
    assert pairs["fallback"] == 0 and pairs["window_outside"] == 0 and pairs["row_outside"] == 0, dict(pairs)


MILD = SCENES[-1]


def test_oracle_equals_the_compiled_reference_on_scenes(oracle, have_ref, template_path):
    """oracle_search_by_stereo, after its own extraction, against the reference's Frame::createStereo; one camera with a
    mild distortion, under which the reference must not throw (no row leaves the image and no window its level there)"""
    if not have_ref:
        pytest.skip("oracle/_ref/libref.so not built (needs the reference sources)")
    for cfg in [s for s in SCENES if s[4] is None] + [MILD]:
        name, c, nf, seed, dist, fx = cfg
        left, right = scene_images(cfg)
        cam = _camera(c, dist, fx)
        oracle.ref_reset()
        bf = oracle.ref_set_camera(cam.fx, c["fy"], c["cx"], c["cy"], c["bl"], None if dist is None else np.array(dist, np.float32))
        ref = oracle.ref_stereo(left, right, template_path, nf, c["n_levels"], c["scale_factor"])
        assert ref["status"] == 0, f"{name}: the reference threw"
        assert np.float32(bf) == cam.bf
        el = oracle.extract(left, nf, c["n_levels"], c["scale_factor"])
        er = oracle.extract(right, nf, c["n_levels"], c["scale_factor"])
        kl = _undistorted(oracle, el.kps, c, dist)
        nm, ur, dp, _ = oracle.search_by_stereo(el, er, np.float32(cam.fx), cam.bf, kps_left_undist=kl)
        assert np.array_equal(ref["kl"].view(np.uint8), kl.view(np.uint8)) and np.array_equal(ref["dl"], el.desc), name
        assert nm == ref["n_matches"] and np.array_equal(ur, ref["u_right"]) and np.array_equal(dp, ref["depth"]), name
        if dist is not None:
            census = _restate(el, er, kl, c, np.float32(cam.fx), cam.bf)["census"]
            assert census["window_outside"] == 0 and census["row_outside"] == 0
    oracle.ref_reset()
    oracle.ref_set_camera(synth.KITTI["fx"], synth.KITTI["fy"], synth.KITTI["cx"], synth.KITTI["cy"], synth.KITTI["bl"], None)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _isolated(oracle, el, er, kps_left, desc_left, kps_right, desc_right, cam):
    """the oracle's search on the device's keypoints and descriptors, over the oracle's pyramids"""
    L = oracle.Extracted(kps_left, desc_left, None, None, el.pyr)
    R = oracle.Extracted(kps_right, desc_right, None, None, er.pyr)
    return oracle.search_by_stereo(L, R, np.float32(cam.fx), cam.bf, kps_left_undist=kps_left)


def _assert_pyramids(ctx, el, er, n_levels, what):
    for side, e in ((0, el), (1, er)):
        got = ctx.get_pyramid(side)
        for l in range(n_levels):
            assert np.array_equal(got[l], e.pyr.level(l)), f"{what}: pyramid {side} level {l}"


def _assert_isolated(oracle, ctx, r, left, right, c, nf, cam, what):
    el = oracle.extract(left, nf, c["n_levels"], c["scale_factor"])
    er = oracle.extract(right, nf, c["n_levels"], c["scale_factor"])
    _assert_pyramids(ctx, el, er, c["n_levels"], what)
    nm, ur, dp, _ = _isolated(oracle, el, er, r.kps_left, r.desc_left, r.kps_right, r.desc_right, cam)
    assert r.n_matches == nm, f"{what}: {r.n_matches} vs {nm} matches"
    assert np.array_equal(r.u_right, ur), f"{what}: uRight differs at {np.nonzero(r.u_right != ur)[0][:8]}"
    assert np.array_equal(r.depth, dp), f"{what}: depth differs at {np.nonzero(r.depth != dp)[0][:8]}"
    return nm


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", SCENES, ids=[s[0] for s in SCENES])
def test_isolated_matcher_exact_on_scenes(oracle, cfg):
    name, c, nf, seed, dist, fx = cfg
    left, right = scene_images(cfg)
    cam = _camera(c, dist, fx)
    ctx = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam)
    r = ctx.stereo_frame(left, right)
    nm = _assert_isolated(oracle, ctx, r, left, right, c, nf, cam, name)
    assert nm > 0.25 * len(r.kps_left)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", PAIRS, ids=[p[0] for p in PAIRS])
def test_isolated_matcher_exact_on_constant_disparity_pairs(oracle, cfg):
    name, c, nf, seed, disp = cfg
    left, right = synth.synth_stereo_pair(c["height"], c["width"], seed, disp)
    cam = _camera(c)
    ctx = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam)
    r = ctx.stereo_frame(left, right)
    _assert_isolated(oracle, ctx, r, left, right, c, nf, cam, name)
    ctx.close()


@pytest.mark.gpu
def test_device_batch_equals_single_frames_and_oracle(oracle):
    """three barrel-distorted scenes and two degenerate frames (uniform right view: no right keypoints; uniform left view:
    no left keypoints) in one device batch: per frame the same bytes as stereo_frame and the oracle's search on the
    batch's own keypoints"""
    import torch

    c, nf = synth.KITTI, 2000
    cam = _camera(c, BARREL)
    lefts, rights = [], []
    for seed in (6, 11, 12):
        l, r, _ = SS.render(SS.make_scene(f"batch{seed}", c["height"], c["width"], seed), c, BARREL)
        lefts.append(l)
        rights.append(r)
    flat = np.full((c["height"], c["width"]), 128, np.uint8)
    lefts += [lefts[0], flat]
    rights += [flat, rights[0]]
    n = len(lefts)
    L, R = np.stack(lefts), np.stack(rights)
    ctx = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam, max_batch=n)
    dl, dr = torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()
    torch.cuda.synchronize()
    res = ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    nk = ctx.read_device(res.n_kps, (2 * n,), np.int32)
    kps_und = ctx.read_device(res.kps_und, (2 * n, nf), api.KP_DTYPE)
    kps = ctx.read_device(res.kps, (2 * n, nf), api.KP_DTYPE)
    desc = ctx.read_device(res.desc, (2 * n, nf, 32), np.uint8)
    ur, dp = ctx.read_device(res.u_right, (n, nf), np.float64), ctx.read_device(res.depth, (n, nf), np.float64)
    nm = ctx.read_device(res.n_matches, (n,), np.int32)
    assert nk[2 * 3 + 1] == 0 and nk[2 * 4] == 0 and nk[2 * 3] > 0 and nk[2 * 4 + 1] > 0
    for f in range(n):
        a, b = nk[2 * f], nk[2 * f + 1]
        one = ctx.stereo_frame(lefts[f], rights[f])
        assert (a, b, nm[f]) == (len(one.kps_left), len(one.kps_right), one.n_matches), f
        assert ur[f, :a].tobytes() == one.u_right.tobytes() and dp[f, :a].tobytes() == one.depth.tobytes(), f
        el = oracle.extract(lefts[f], nf, c["n_levels"], c["scale_factor"])
        er = oracle.extract(rights[f], nf, c["n_levels"], c["scale_factor"])
        _assert_pyramids(ctx, el, er, c["n_levels"], f"frame {f}")
        e_nm, e_ur, e_dp, _ = _isolated(oracle, el, er, kps_und[2 * f, :a], desc[2 * f, :a], kps[2 * f + 1, :b], desc[2 * f + 1, :b], cam)
        assert nm[f] == e_nm and np.array_equal(ur[f, :a], e_ur) and np.array_equal(dp[f, :a], e_dp), f
    assert nm[3] == 0 and nm[4] == 0 and (nm[:3] > 500).all()
    ctx.close()
