"""The plain-C restatement (oracle/orb_oracle.c) against the reference's OWN code compiled unmodified
(oracle/_ref/libref.so = the reference's src/ORB_SLAM2/src/{ORBExtractor,Camera}.cc + the searchByStereo line ranges
of ORBMatcher.cc built against oracle/stub).  Everything must be identical to the last bit.

The reference sources are not part of this repository, so every case also checks the restatement against the SHA-256
digests in tests/golden/oracle_vs_ref_sha256.json: the outputs on which the restatement and the compiled reference
agreed bit for bit (recorded from the restatement, which this module held identical to libref.so on these inputs).
Where libref.so is present the cases compare against it directly as well.  To re-record the digests after a deliberate
change of the inputs, run this module with ORBX_RECORD_DIGESTS=<file> and check the new file against libref.so."""
import hashlib
import json
import os

import numpy as np
import pytest

from orb_slam2_ros2_b200 import synth

DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref_sha256.json")
_RECORD = os.environ.get("ORBX_RECORD_DIGESTS")
_recorded = {}


@pytest.fixture(scope="module")
def R(oracle):
    return oracle


@pytest.fixture(scope="module")
def digests():
    if _RECORD:
        yield None
        with open(_RECORD, "w") as f:
            json.dump(_recorded, f, indent=1, sort_keys=True)
    else:
        with open(DIGESTS) as f:
            yield json.load(f)


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _check(digests, key, *arrays):
    if digests is None:
        _recorded[key] = _sha(*arrays)
    else:
        assert _sha(*arrays) == digests[key], f"{key}: the restatement's outputs differ from the ones the reference produced"


def _same_kps(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _bf(c):
    return np.float32(c["fx"]) * np.float32(c["bl"])  # Camera.cc: mbf = mb * fx, in float


CONFIGS = [
    ("K2000", 376, 1241, 2000, 8, 1.2, 0),
    ("K500", 376, 1241, 500, 8, 1.2, 1),
    ("K4000", 376, 1241, 4000, 8, 1.2, 2),
    ("T1000", 480, 640, 1000, 8, 1.2, 3),
    ("H5000", 1080, 1920, 5000, 12, 1.2, 4),
    ("S300x5", 240, 320, 300, 5, 1.3, 5),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_extract_identical(R, have_ref, digests, template_path, cfg):
    name, h, w, nf, nl, sc, seed = cfg
    img = synth.synth_image(h, w, seed)
    e = R.extract(img, nf, nl, sc)
    assert len(e.kps) > 0
    _check(digests, "extract/" + name, e.kps, e.desc, e.pyr.sf, *[e.pyr.level(l) for l in range(nl)], *[e.pyr.blurred(l) for l in range(nl)])
    if not have_ref:
        return
    R.ref_reset()
    n, kps, desc, info = R.ref_extract(img, template_path, nf, nl, sc, want_pyramid=True)
    assert n == len(e.kps)
    assert _same_kps(kps, e.kps)
    assert np.array_equal(desc, e.desc)
    assert np.array_equal(info["sf"], e.pyr.sf)
    for l in range(nl):
        assert np.array_equal(info["levels"][l], e.pyr.level(l))
    blurred = R.ref_blurred(img, template_path, nf, nl, sc, info["lw"], info["lh"])
    for l in range(nl):
        assert np.array_equal(blurred[l], e.pyr.blurred(l))


def test_extract_degenerate_images(R, have_ref, digests, template_path):
    for img in (np.zeros((376, 1241), np.uint8), np.full((200, 300), 255, np.uint8)):
        e = R.extract(img, 1000, 4, 1.2)
        assert len(e.kps) == 0
        if have_ref:
            R.ref_reset()
            n, kps, desc, _ = R.ref_extract(img, template_path, 1000, 4, 1.2)
            assert n == 0
    # uniform noise: tens of thousands of corners per level, quotas still met
    img = np.random.default_rng(1).integers(0, 256, (240, 320), dtype=np.uint8)
    e = R.extract(img, 1000, 4, 1.2)
    _check(digests, "extract_noise", e.kps, e.desc)
    if have_ref:
        n, kps, desc, _ = R.ref_extract(img, template_path, 1000, 4, 1.2)
        assert n == len(e.kps) and _same_kps(kps, e.kps) and np.array_equal(desc, e.desc)


def test_starved_level_returns_zero(R, have_ref, digests, template_path):
    """a level with fewer usable corners than its quota drains the multimap and yields 0 keypoints (ORBExtractor.cc:151)"""
    img = np.full((240, 320), 128, np.uint8)
    img[60:180, 80:240] = synth.synth_image(120, 160, 11)  # corners only in the centre
    e = R.extract(img, 3000, 3, 1.2)
    assert (e.level_counts == 0).any()
    _check(digests, "starved_level", e.kps, e.desc, e.level_counts)
    if have_ref:
        R.ref_reset()
        n, kps, desc, _ = R.ref_extract(img, template_path, 3000, 3, 1.2)
        assert n == len(e.kps) and _same_kps(kps, e.kps) and np.array_equal(desc, e.desc)


def test_errors(R, have_ref, template_path):
    """the compiled reference's own error paths; there is nothing to compare them with when it is absent"""
    if not have_ref:
        pytest.skip("oracle/_ref/libref.so not built (needs the reference sources)")
    R.ref_reset()
    img = synth.synth_image(60, 100, 0)
    n, *_ = R.ref_extract(img, template_path, 500, 8, 1.2)
    assert n == -1  # ImageSizeError
    R.ref_reset()
    n, *_ = R.ref_extract(synth.synth_image(240, 320, 0), "/nonexistent/brief_template.txt", 500, 4, 1.2)
    assert n == -2  # FileNotOpenError
    R.ref_reset()


def test_quadtree_identical(R, have_ref, digests):
    rng = np.random.default_rng(7)
    cases = []
    for it in range(60):
        w, h = int(rng.integers(40, 1300)), int(rng.integers(40, 400))
        n = int(rng.integers(0, 3000))
        xs = rng.integers(3, max(4, w - 3), n).astype(np.float32)
        ys = rng.integers(3, max(4, h - 3), n).astype(np.float32)
        if it % 5 == 0 and n:  # corners exactly on root / first split lines
            xs[: n // 4] = np.float32(w / max(1, round(w / h)) / 2)
            ys[n // 4 : n // 2] = np.float32(h // 2) if h % 2 == 0 else ys[n // 4 : n // 2]
        resp = rng.integers(6, 120, n).astype(np.float32)
        for need in sorted({0, 1, 2, int(rng.integers(3, 600)), n + 5}):
            a, _ = R.quadtree_select(w, h, xs, ys, resp, need)
            if have_ref and not (n == 0 and need == 1):  # the reference reads kps[0] out of bounds there
                assert np.array_equal(a, R.ref_quadtree(w, h, xs, ys, resp, need)), (w, h, n, need)
            cases.append(a)
    assert len(cases) > 200
    _check(digests, "quadtree", *cases)


def test_quadtree_portrait_and_wide(R, have_ref, digests):
    rng = np.random.default_rng(3)
    cases = []
    for w, h in [(100, 400), (100, 260), (3000, 100), (64, 64)]:
        n = 800
        xs = rng.integers(3, w - 3, n).astype(np.float32)
        ys = rng.integers(3, h - 3, n).astype(np.float32)
        resp = rng.integers(6, 120, n).astype(np.float32)
        for need in (5, 50, 300):
            a, _ = R.quadtree_select(w, h, xs, ys, resp, need)
            if have_ref:
                assert np.array_equal(a, R.ref_quadtree(w, h, xs, ys, resp, need)), (w, h, need)
            cases.append(a)
    _check(digests, "quadtree_portrait_and_wide", *cases)


STEREO = [
    ("K2000_d17", synth.KITTI, 2000, 0, 17),
    ("K2000_d5", synth.KITTI, 2000, 1, 5),
    ("K1000_d63", synth.KITTI, 1000, 2, 63),
    ("T1000_d17", synth.TUM, 1000, 3, 17),
    ("H5000_d42", synth.HD, 5000, 4, 42),
]


@pytest.mark.parametrize("cfg", STEREO, ids=[c[0] for c in STEREO])
def test_stereo_identical(R, have_ref, digests, template_path, cfg):
    name, c, nf, seed, disp = cfg
    left, right = synth.synth_stereo_pair(c["height"], c["width"], seed, disp)
    el = R.extract(left, nf, c["n_levels"], c["scale_factor"])
    er = R.extract(right, nf, c["n_levels"], c["scale_factor"])
    nm, ur, dp, _ = R.search_by_stereo(el, er, np.float32(c["fx"]), _bf(c))
    assert nm > 0.3 * len(el.kps)
    _check(digests, "stereo/" + name, el.kps, er.kps, el.desc, er.desc, np.int64(nm), ur, dp)
    # sanity: matched disparities sit at the synthetic disparity
    m = ur >= 0
    assert np.median(el.kps["x"][m] - ur[m]) == pytest.approx(disp, abs=1.0)
    if not have_ref:
        return
    R.ref_reset()
    bf = R.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)  # zero distortion
    assert np.float32(bf) == _bf(c)
    r = R.ref_stereo(left, right, template_path, nf, c["n_levels"], c["scale_factor"])
    assert r["status"] == 0
    assert _same_kps(r["kl"], el.kps) and _same_kps(r["kr"], er.kps)
    assert np.array_equal(r["dl"], el.desc) and np.array_equal(r["dr"], er.desc)
    assert nm == r["n_matches"]
    assert np.array_equal(ur, r["u_right"]) and np.array_equal(dp, r["depth"])


@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("use_dist", [True, False], ids=["tum_distortion", "no_distortion"])
def test_rgbd_ctor_identical(R, have_ref, digests, template_path, dtype, use_dist):
    """the reference's own RGB-D Frame ctor body (src/Frame.cc:130-158, compiled verbatim into oracle/_ref) against the
    restatement: extraction, undistortion, depth lookup at the RAW keypoint, uRight = x_undistorted - bf / d"""
    c = synth.TUM
    gray = synth.synth_image(c["height"], c["width"], 12)
    depth = synth.synth_depth_u16(c["height"], c["width"], 12, c["depth_scale"])
    if dtype == np.float32:
        depth = depth.astype(np.float32)
    dist = np.array(c["dist"], np.float32) if use_dist else None
    e = R.extract(gray, 1000, 8, 1.2)
    ku = e.kps.copy()
    if use_dist:
        xy = R.undistort_points(np.stack([e.kps["x"], e.kps["y"]], 1), c["fx"], c["fy"], c["cx"], c["cy"], dist)
        ku["x"], ku["y"] = xy[:, 0], xy[:, 1]
    our, odp = R.rgbd_lookup(depth, c["depth_scale"], e.kps, ku, _bf(c))
    assert 0.05 < (odp < 0).mean() < 0.2 and (odp > 0).sum() > 700
    _check(digests, f"rgbd/{np.dtype(dtype).name}/{'dist' if use_dist else 'nodist'}", ku, e.desc, our, odp)
    if not have_ref:
        return
    R.ref_reset()
    bf = R.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], dist)
    assert np.float32(bf) == _bf(c)
    kps, desc, ur, dp = R.ref_rgbd(gray, depth, c["depth_scale"], template_path, 1000, 8, 1.2)
    assert _same_kps(kps, ku) and np.array_equal(desc, e.desc)
    assert np.array_equal(dp, odp) and np.array_equal(ur, our)
    R.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)


def test_undistort_identical(R, have_ref, digests):
    c = synth.TUM
    rng = np.random.default_rng(5)
    pts = np.stack([rng.uniform(19, 620, 1000), rng.uniform(19, 460, 1000)], 1).astype(np.float32)
    a = R.undistort_points(pts, c["fx"], c["fy"], c["cx"], c["cy"], np.array(c["dist"], np.float32))
    _check(digests, "undistort", a)
    if not have_ref:
        return
    R.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], np.array(c["dist"], np.float32))
    assert np.array_equal(a, R.ref_undistort(pts))
    R.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)
    assert np.array_equal(R.ref_undistort(pts), pts)  # k1 == 0 -> early return (Camera.cc:31)


# ---- tracking-side matchers (SURVEY section 8(f) rank 2): Frame.cc:53-69,286-311 and ORBMatcher.cc:967-990,1013-1051 ----
def _frame(R, have_ref, template_path, h, w, nf, nl, seed):
    """the reference's keypoints of a synthetic frame; the restatement's where libref.so is absent (test_extract_identical
    holds the two identical)"""
    img = synth.synth_image(h, w, seed)
    if have_ref:
        R.ref_reset()
        n, kps, desc, info = R.ref_extract(img, template_path, nf, nl, 1.2)
        return kps, desc, info["sf"]
    e = R.extract(img, nf, nl, 1.2)
    return e.kps, e.desc, e.pyr.sf


@pytest.mark.parametrize("shape", [(376, 1241, 2000, 8), (480, 640, 1000, 8), (240, 320, 300, 4)], ids=["K", "T", "S"])
def test_init_grid_identical(R, have_ref, digests, template_path, shape):
    h, w, nf, nl = shape
    kps, _, _ = _frame(R, have_ref, template_path, h, w, nf, nl, 21)
    out = []
    for bounds in [(0.0, 0.0, float(w), float(h)), (-7.25, -3.5, w + 11.75, h + 6.5)]:
        a = R.grid_csr(kps, *bounds)
        if have_ref:
            b = R.ref_grid_csr(kps, *bounds)
            assert a[:2] == b[:2] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
        flat = [c for row in R.init_grid(kps, *bounds) for c in row]
        assert np.array_equal(np.concatenate(flat), a[3])
        out += [np.array(a[:2], np.int64), a[2], a[3]]
    _check(digests, f"init_grid/{h}x{w}", *out)


@pytest.mark.parametrize("mode", ["window", "up", "down"])
@pytest.mark.parametrize("shape", [(376, 1241, 2000, 8), (480, 640, 1000, 8)], ids=["K", "T"])
def test_search_in_area_identical(R, have_ref, digests, template_path, shape, mode):
    h, w, nf, nl = shape
    kps, desc, sf = _frame(R, have_ref, template_path, h, w, nf, nl, 22)
    bounds = (0.0, 0.0, float(w), float(h))
    out = []
    for th, seed in [(15.0, 1), (30.0, 2), (3.0, 3)]:
        q, qd, ex, _ = synth.synth_area_queries(kps, desc, 700, seed, w, h, nl, th, mode=mode)
        for e in (None, ex):
            a = R.search_in_area(kps, desc, bounds, sf, q, qd, e)
            if have_ref:
                b = R.ref_search_in_area(kps, desc, bounds, sf, q, qd, e)
                for k in a:
                    assert np.array_equal(a[k], b[k], equal_nan=True), (k, th, e is None)
            assert (a["n_cand"] > 0).sum() > 300
            out += [a[k] for k in sorted(a)]
    _check(digests, f"search_in_area/{h}x{w}/{mode}", *out)


def test_best_match_second_best_rule_and_ties(R, have_ref, digests, template_path):
    """getBestMatch keeps the FIRST minimum and its `second` ignores displaced minima: duplicated descriptors, zero
    distances (ratio 0/0 = NaN) and strictly descending distance sequences (second stays INT_MAX) must all agree."""
    kps, desc, sf = _frame(R, have_ref, template_path, 240, 320, 300, 4, 23)
    rng = np.random.default_rng(3)
    desc = desc.copy()
    desc[rng.integers(0, len(desc), 80)] = desc[rng.integers(0, len(desc), 80)]  # duplicates -> ties
    q, qd, ex, src = synth.synth_area_queries(kps, desc, 500, 4, 320, 240, 4, 60.0, flip_bits=0)  # exact copies: distance 0
    a = R.search_in_area(kps, desc, (0.0, 0.0, 320.0, 240.0), sf, q, qd, None)
    if have_ref:
        b = R.ref_search_in_area(kps, desc, (0.0, 0.0, 320.0, 240.0), sf, q, qd, None)
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert np.isnan(a["ratio"]).any() and (a["best_dist"] == 0).sum() > 100
    _check(digests, "best_match_ties", *[a[k] for k in sorted(a)])


def test_verify_angle_identical(R, have_ref, digests, template_path):
    kps, desc, sf = _frame(R, have_ref, template_path, 376, 1241, 2000, 8, 24)
    rng = np.random.default_rng(5)
    out = []
    for n, spread in [(1500, 25.0), (40, 200.0), (3, 1.0), (0, 1.0)]:
        qi = rng.integers(0, len(kps), n).astype(np.int32)
        ti = np.arange(n, dtype=np.int32)
        k2 = np.zeros(max(n, 1), R.KP_DTYPE)
        ang = kps["angle"][qi].astype(np.float64) + rng.normal(0, spread, n)
        k2["angle"][:n] = (180.0 - np.mod(180.0 - ang, 360.0)).astype(np.float32)  # back into (-180, 180] like IC angles (:449)
        k2["angle"][: n // 7] = kps["angle"][qi[: n // 7]]  # zero differences and exact wrap-arounds
        di = rng.integers(0, 50, n).astype(np.float32)
        a = R.verify_angle(qi, ti, di, kps, k2)
        if have_ref:
            assert all(np.array_equal(x, y) for x, y in zip(a, R.ref_verify_angle(qi, ti, di, kps, k2))), n
        assert len(a[0]) <= n
        out += list(a)
    _check(digests, "verify_angle", *out)
