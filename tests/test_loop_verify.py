"""Loop verification (orbx_loopver_*: searchByBow + verifyAngle + a fixed-scale Horn RANSAC per (query, candidate) pair, the
check of ORB-SLAM2's LoopClosing::ComputeSim3 under the rules of include/orbx.h).

PARITY UNPINNED: the reference's LoopClosing / Sim3Solver and ORB-SLAM2 are not vendored.  CPU: the plain-C oracle_loopver
(tests/loopver_oracle.c) equals a literal Python restatement in ORB-SLAM2's sequential shape (tests/loopver_restatement.py)
on record sets crafted to reach every rule, transform bits included; on rendered stereo loops (tests/loop_scenes.py) the
oracle's own extraction accepts the true loops near the ground-truth pose and rejects unrelated scenes.  GPU: the CUDA
verifier equals the oracle bit for bit on the crafted sets and on the device's own records of a rendered sequence; sharded
use and the error codes."""
from collections import Counter

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api

import loop_scenes as S
import loopver_restatement as R

OUT = api.LOOPVER_OUTPUTS


@pytest.fixture(scope="module")
def crafted(oracle):
    c = R.crafted(oracle.KP_DTYPE)
    c["O"] = oracle.Vocabulary(**c["voc"])
    c["sf"] = oracle.scale_factors(R.SCALE, R.N_LEVELS)
    return c


def _assert_same(got, exp, what=""):
    for k in OUT:
        g, e = np.asarray(got[k]).reshape(np.shape(exp[k])), exp[k]
        if k == "T":
            assert np.array_equal(g.view(np.uint64), e.view(np.uint64)), f"{what} T bits"
        else:
            assert np.array_equal(g, e), f"{what} {k}: {g} != {e}"


def _angle_deg(Ra, Rb) -> float:
    c = (np.trace(np.asarray(Ra).T @ np.asarray(Rb)) - 1) / 2
    return float(np.degrees(np.arccos(np.clip(c, -1, 1))))


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_oracle_equals_literal_restatement_and_reaches_every_rule(oracle, crafted):
    c = crafted
    seen = Counter()
    for prm in c["configs"]:
        exp = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], prm)
        py = R.py_verify(oracle, c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], prm, seen)
        _assert_same(exp, py, str(prm))
        # a sub-range of queries keeps its frame ids
        sub = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 5, c["table"][5:12], prm)
        _assert_same(sub, {k: v[5:12] for k, v in exp.items()}, f"sub-range {prm}")
    rules = {"matches_below_min", "matches_at_min", "corr_below_min_inliers", "corr_eq_min_inliers_one_iteration", "inliers_eq_min_not_accepted",
             "accepted_at_min_plus_one", "tied_best", "collinear_sample", "coincident_sample", "point_behind_camera", "zero_depth_dropped", "empty_slot",
             "candidate_is_query", "loop_frame_by_round", "rotation_check_drops", "refit_from_samples"}
    assert rules <= {b for b, n in seen.items() if n > 0}, dict(seen)


def test_crafted_set_reads_as_designed(crafted):
    """query 0: 19 matches stop, 20 give n_corr == min_inliers (one hypothesis, 20 inliers: not accepted), 21 are accepted at
    the first hypothesis with the true pose; a candidate that equals its query is accepted with the identity"""
    c = crafted
    r = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], R.params())
    assert r["n_matches"][0].tolist() == [19, 20, 21] and r["n_corr"][0].tolist() == [0, 20, 21]
    assert r["n_iters"][0].tolist() == [0, 1, 1] and r["accepted"][0].tolist() == [0, 0, 1] and r["n_inliers"][0].tolist() == [0, 20, 21]
    (q, cand), (Rt, tt) = next(iter(c["truth"].items()))
    assert r["loop_frame"][q] == cand
    T = r["T"][q, 2]
    assert _angle_deg(T[:9].reshape(3, 3), Rt) < 1e-4 and np.abs(T[9:] - tt).max() < 1e-5  # float32 keypoints
    self_row = [i for i in range(len(c["table"])) if c["table"][i][0] == i]
    assert self_row and r["accepted"][self_row[0], 0] == 1
    assert np.abs(r["T"][self_row[0], 0] - np.r_[np.eye(3).ravel(), np.zeros(3)]).max() < 1e-9


# Bounds on the refitted pose of a rendered loop, relative to the true motion (20 degrees and 0.42 m) so that the identity
# or t = 0 (an error of the whole rotation or of the whole translation) fails.  The inlier test measures pixel errors, which
# hardly see a depth error along the viewing ray, but Horn fits 3-D points and weighs it fully, so the stereo depth noise (a
# fraction of a pixel of disparity at bf = 240, a few cm at 3 m) tilts the fit: against 1 degree and 0.1 m the oracle's loops
# show up to 1.97 degrees (10 % of their rotation) and 0.081 m (19 % of their translation).  ORB-SLAM2 refines this pose with
# g2o on reprojection errors, which is out of scope.
ROT_TOL, T_TOL = 0.4, 0.5


def _pose_error(T, Rt, tt):
    """(rotation error / true rotation angle, translation error / true translation)"""
    return _angle_deg(T[:9].reshape(3, 3), Rt) / _angle_deg(np.eye(3), Rt), float(np.linalg.norm(T[9:] - tt) / np.linalg.norm(tt))


def test_oracle_accepts_rendered_loops_near_the_true_pose(oracle):
    seq = S.loop_sequence(oracle)
    r = R.oracle_verify(seq["O"], seq["levelsup"], seq["frames"], seq["cam"], seq["sf"], 0, seq["table"], R.params())
    for (q, sl), (Rt, tt) in seq["truth"].items():
        assert r["accepted"][q, sl] == 1, (q, sl, r["n_matches"][q, sl], r["n_corr"][q, sl], r["n_inliers"][q, sl])
        err = _pose_error(r["T"][q, sl], Rt, tt)
        assert err[0] < ROT_TOL and err[1] < T_TOL, (q, sl, err)
    for q, sl in seq["unrelated"]:
        assert r["accepted"][q, sl] == 0, (q, sl, r["n_matches"][q, sl], r["n_inliers"][q, sl])


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _crafted_ctx(**kw):
    return api.Context(320, 240, R.N_FEATURES, R.N_LEVELS, R.SCALE, camera=api.Camera(*R.CAM, 0.1), **kw)


def _device_verify(torch, LV, q_lo, table, prm):
    nq, k = table.shape
    N = LV.ctx.n_features
    tab = torch.from_numpy(np.ascontiguousarray(table, np.int32)).cuda()
    t = {n: torch.full((nq, k), 7, dtype=torch.int32, device="cuda") for n in OUT[:7]}
    t.update(T=torch.full((nq, k, 12), 7.0, dtype=torch.float64, device="cuda"), match=torch.full((nq, k, N), 7, dtype=torch.int32, device="cuda"),
             loop_frame=torch.full((nq,), 7, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    LV.verify_ptr(q_lo, nq, tab.data_ptr(), k, [t[n].data_ptr() for n in OUT], on_device=True, **prm)
    LV.ctx.synchronize()
    return {n: v.cpu().numpy() for n, v in t.items()}


@pytest.mark.gpu
def test_cuda_verifier_equals_oracle_on_crafted_sets(crafted):
    import torch

    c = crafted
    ctx = _crafted_ctx()
    assert np.array_equal(ctx.scaled_factors(), c["sf"])
    V = api.Vocabulary(ctx, **c["voc"])
    rec = R.to_records(ctx, c["frames"])
    F = len(rec)
    d_rec = torch.from_numpy(rec.view(np.uint8).reshape(F, -1).copy()).cuda()
    torch.cuda.synchronize()
    for LV in (api.LoopVerifier.build(ctx, V, rec, F, levelsup=c["levelsup"]), api.LoopVerifier.build(ctx, V, d_rec.data_ptr(), F, levelsup=c["levelsup"])):
        for prm in c["configs"]:
            exp = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], prm)
            _assert_same(LV.verify(0, c["table"], **prm), exp, f"host {prm}")
            _assert_same(_device_verify(torch, LV, 0, c["table"], prm), exp, f"device {prm}")
            _assert_same(LV.verify(5, c["table"][5:12], **prm), {k: v[5:12] for k, v in exp.items()}, f"sub-range {prm}")
        # a device table entry outside [-1, F) is an empty slot
        bad = c["table"].copy()
        bad[0, 1], bad[1, 0] = F, -5
        exp = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, np.where((bad >= 0) & (bad < F), bad, -1), R.params())
        _assert_same(_device_verify(torch, LV, 0, bad, R.params()), exp, "device table with out-of-range entries")
        LV.close()
    V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_verifier_on_the_devices_own_records_of_a_rendered_loop(oracle):
    import torch

    seq = S.loop_sequence(oracle, with_images=True)
    ctx = S.context(max_batch=4)
    F, N = len(seq["left"]), ctx.n_features
    lay = ctx.record_layout()
    d_rec = torch.zeros((F, lay.record_bytes), dtype=torch.uint8, device="cuda")
    left, right = seq["left"], seq["right"]
    res = ctx.sequence_stereo_ptr(F, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], records_ptr=d_rec.data_ptr(),
                                  record_stride=lay.record_bytes, records_on_device=True)
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=10, L=4, seed=3)
    D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=N)
    top_k, window = 4, 3
    cand = torch.zeros((F, top_k), dtype=torch.int32, device="cuda")
    D.query_ptr(0, F, top_k, window, 0.0, [cand.data_ptr()] + [0] * 6, on_device=True)
    LV = api.LoopVerifier.build(ctx, V, d_rec.data_ptr(), F, levelsup=S.LEVELSUP)
    prm = R.params(seed=9)
    got = _device_verify(torch, LV, 0, cand.cpu().numpy(), prm)
    # the oracle on the same records, vocabulary and table
    rec = d_rec.cpu().numpy().view(ctx.record_dtype()).reshape(F)
    fr = dict(kps=rec["kps_left"], desc=rec["desc_left"], depth=rec["depth"], n=rec["n_left"])
    a, i = V.arrays(), V.info()
    O = oracle.Vocabulary(i["k"], i["L"], a["parent"], a["is_leaf"], a["desc"], a["weight"])
    cam = (ctx.camera.fx, ctx.camera.fy, ctx.camera.cx, ctx.camera.cy)
    table = cand.cpu().numpy()
    exp = R.oracle_verify(O, S.LEVELSUP, fr, cam, ctx.scaled_factors(), 0, table, prm)
    _assert_same(got, exp, "device records")
    # the true loops among the database's candidates are accepted near the true pose
    n_true = 0
    for q in range(F):
        for sl in range(top_k):
            g = int(table[q, sl])
            if g >= 0 and S.is_loop(seq, q, g):
                n_true += 1
                assert got["accepted"][q, sl] == 1, (q, g)
                Rt, tt = S.relative_pose(seq, q, g)
                err = _pose_error(got["T"][q, sl], Rt, tt)
                assert err[0] < ROT_TOL and err[1] < T_TOL, (q, g, err)
    assert n_true >= 2
    for o in (LV, D, V, ctx):
        o.close()


@pytest.mark.gpu
def test_cuda_two_local_ranks_verify_their_blocks(crafted):
    c = crafted
    ranks = [_crafted_ctx() for _ in range(2)]
    rec = R.to_records(ranks[0], c["frames"])
    F = len(rec)
    parts, whole = [], None
    for r, ctx in enumerate(ranks):
        V = api.Vocabulary(ctx, **c["voc"])
        LV = api.LoopVerifier.build(ctx, V, rec, F, levelsup=c["levelsup"])
        blk = api.frame_range(F, r, 2)
        parts.append(LV.verify(blk.start, c["table"][blk.start : blk.stop], seed=4))
        if r == 0:
            whole = LV.verify(0, c["table"], seed=4)
        LV.close()
        V.close()
    for k in OUT:
        assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), k
    assert whole["accepted"].sum() > 5
    for o in ranks:
        o.close()


@pytest.mark.gpu
def test_cuda_verifier_rejects_bad_arguments(crafted):
    c = crafted
    ctx = _crafted_ctx()
    V = api.Vocabulary(ctx, **c["voc"])
    rec = R.to_records(ctx, c["frames"])
    F = len(rec)
    with pytest.raises(ValueError, match="invalid argument"):
        api.LoopVerifier.build(ctx, V, rec, F, levelsup=-1)
    with pytest.raises(ValueError, match="invalid argument"):  # record stride not a multiple of 16
        api.LoopVerifier.build(ctx, V, np.zeros((F, rec.dtype.itemsize + 8), np.uint8), F)
    import torch

    d_rec = torch.zeros(F * rec.dtype.itemsize + 16, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="invalid argument"):  # device records that are not 16-byte aligned
        api.LoopVerifier.build(ctx, V, d_rec.data_ptr() + 8, F, levelsup=c["levelsup"], record_stride=rec.dtype.itemsize)
    bad_n = rec.copy()
    bad_n["n_left"][2] = R.N_FEATURES + 1
    with pytest.raises(ValueError, match="invalid argument"):
        api.LoopVerifier.build(ctx, V, bad_n, F)
    LV = api.LoopVerifier.build(ctx, V, rec, F, levelsup=c["levelsup"])
    tab = c["table"]
    for kw in [dict(probability=0.0), dict(probability=1.0), dict(min_inliers=2), dict(max_iterations=0), dict(ratio=float("nan"))]:
        with pytest.raises(ValueError, match="invalid argument"):
            LV.verify(0, tab, **kw)
    for q_lo, t in [(1, tab), (-1, tab[:2]), (0, np.zeros((F, 0), np.int32))]:
        with pytest.raises(ValueError, match="invalid argument"):
            LV.verify(q_lo, t)
    for v in (F, -2):
        t = tab.copy()
        t[3, 1] = v
        with pytest.raises(ValueError, match="invalid argument"):
            LV.verify(0, t)
    assert LV.verify(F, tab[:0])["loop_frame"].size == 0  # no queries: nothing is enqueued
    other = _crafted_ctx()
    W = api.Vocabulary(other, **c["voc"])
    with pytest.raises(ValueError, match="another context"):
        api.LoopVerifier.build(ctx, W, rec, F, levelsup=c["levelsup"])
    E = api.LoopVerifier.build(other, W, rec, F, levelsup=c["levelsup"])
    E.ctx = ctx
    with pytest.raises(ValueError, match="another context"):
        E.verify(0, tab)
    for o in (LV, E, W, V, other, ctx):
        o.close()
