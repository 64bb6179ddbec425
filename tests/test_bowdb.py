"""Keyframe database (orbx_bowdb_*: the BoW inverted file and the first stage of ORB-SLAM2's
KeyFrameDatabase::DetectLoopCandidates / DetectRelocalizationCandidates with DBoW3's L1 score, under the rules of include/orbx.h).

PARITY UNPINNED, as the transform: DBoW3 and the reference's KeyFrameDatabase are not vendored.  CPU: the plain-C
oracle_bowdb_query (tests/bowdb_oracle.c) equals a literal Python restatement in ORB-SLAM2's shape (tests/bowdb_restatement.py)
on databases crafted to reach every rule, score bits included.  GPU: the CUDA database equals the oracle bit for bit, on those
databases and on the device's own descriptors of a sequence; the resident-frame query, sharded use and the error codes."""
from collections import Counter

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

import bowdb_restatement as R

OUT = api.BOWDB_OUTPUTS


@pytest.fixture(scope="module")
def cases(oracle):
    return {name: R.case(oracle, name) for name in R.CASES}


def _assert_same(got, exp, what=""):
    for k in OUT:
        g, e = np.asarray(got[k]).reshape(np.shape(exp[k])), exp[k]
        if k == "cand_score":
            assert np.array_equal(g.view(np.uint32), e.view(np.uint32)), f"{what} {k}"  # score bits
        else:
            assert np.array_equal(g, e), f"{what} {k}: {g} != {e}"


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_oracle_equals_literal_restatement_and_reaches_every_rule(cases):
    seen = Counter()
    for name, c in cases.items():
        db = c["db"]
        F = len(db["n"])
        bows = R.bow_dicts(db["ids"], db["vals"], db["n"])
        seen["frame_without_keypoints"] += int((c["counts"] == 0).sum())
        seen["frame_all_stopped"] += int(((c["counts"] > 0) & (db["n"] == 0)).sum())
        for window, min_score, top_k in c["configs"]:
            py = R.py_query(bows, [(q, bows[q], q) for q in range(F)], window, min_score, top_k, seen)
            _assert_same(R.oracle_query(db, db, 0, window, min_score, top_k), py, f"{name} {window} {min_score} {top_k}")
            # the same BowVectors as outside queries (the resident-frame rule: nothing excluded)
            py = R.py_query(bows, [(q, bows[q], None) for q in range(F)], -1, min_score, top_k)
            _assert_same(R.oracle_query(db, db, 0, -1, min_score, top_k), py, f"{name} unexcluded")
    rules = {"common_eq_min_common_rejected", "common_eq_whole_min_common_rejected", "min_common_whole", "min_common_truncated", "score_eq_min_score_kept",
             "window_edge_excluded", "window_edge_plus_one_listed", "frame_without_keypoints", "frame_all_stopped", "shares_only_connected", "tied_scores",
             "top_k_below_n_kept", "top_k_at_or_above_n_kept", "one_frame_database", "empty_sharing"}
    assert rules <= {b for b, n in seen.items() if n > 0}, dict(seen)


def test_crafted_loop_database_reads_as_designed(cases):
    """frame 5 of the loop database at window 1: frames 0 / 9 (10 shared words, tied), 2 and 3 (9) are scored, 1 (8 == the
    whole min_common) and 10 (3) are not, 4 and 6 are connected; frame 13 (7 shared words, min_common 5 from 5.6)
    scores 15 and 17 but not 16 (5)"""
    db = cases["loop"]["db"]
    r = R.oracle_query(db, db, 0, 1, 0.0, 18)
    assert (r["max_common"][5], r["n_scored"][5], r["n_kept"][5]) == (10, 4, 4)
    row = list(r["cand_frame"][5][:4])
    i = row.index(0)
    assert row[i + 1] == 9 and r["cand_score"][5][i] == r["cand_score"][5][i + 1]  # the tie, in frame order
    assert set(r["cand_frame"][5][:4]) == {0, 2, 3, 9} and r["n_sharing"][5] == 6
    assert (r["max_common"][13], r["n_scored"][13]) == (7, 2) and set(r["cand_frame"][13][:2]) == {15, 17}
    assert r["n_sharing"][11] == 0 and r["n_sharing"][12] == 0 and r["n_sharing"][7] == 0


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _small_ctx(**kw):
    return api.Context(320, 240, 500, 4, 1.2, camera=api.Camera(300.0, 300.0, 160.0, 120.0, 0.1), **kw)


def _device_query(torch, D, q_lo, q_hi, top_k, window, min_score):
    n = q_hi - q_lo
    t = dict(cand_frame=torch.full((n, top_k), 7, dtype=torch.int32, device="cuda"), cand_score=torch.zeros((n, top_k), dtype=torch.float32, device="cuda"),
             cand_common=torch.zeros((n, top_k), dtype=torch.int32, device="cuda"), **{k: torch.full((n,), 7, dtype=torch.int32, device="cuda") for k in OUT[3:]})
    D.query_ptr(q_lo, q_hi, top_k, window, min_score, [t[k].data_ptr() for k in OUT], on_device=True)
    D.ctx.synchronize()
    return {k: v.cpu().numpy() for k, v in t.items()}


@pytest.mark.gpu
def test_cuda_database_equals_oracle_on_crafted_cases(cases):
    import torch

    ctx = _small_ctx()
    for name, c in cases.items():
        V = api.Vocabulary(ctx, **c["voc"])
        db = c["db"]
        F = len(db["n"])
        d_desc, d_n = torch.from_numpy(c["desc"]).cuda(), torch.from_numpy(c["counts"]).cuda()
        torch.cuda.synchronize()
        for D in (api.BowDatabase.build(ctx, V, c["desc"], c["counts"]),
                  api.BowDatabase.build(ctx, V, d_desc.data_ptr(), d_n.data_ptr(), n_frames=F, stride=c["desc"].shape[1])):
            assert D.info() == dict(n_frames=F, n_words=db["n_words"], n_postings=int(db["n"].sum()))
            for window, min_score, top_k in c["configs"]:
                exp = R.oracle_query(db, db, 0, window, min_score, top_k)
                _assert_same(D.query(0, F, top_k, window, min_score), exp, f"{name} host {window} {min_score} {top_k}")
                _assert_same(_device_query(torch, D, 0, F, top_k, window, min_score), exp, f"{name} device")
                if F > 3:  # a sub-range: the queries keep their own frame ids
                    sub = D.query(2, F - 1, top_k, window, min_score)
                    _assert_same(sub, {k: v[2 : F - 1] for k, v in exp.items()}, f"{name} sub-range")
            D.close()
        V.close()
    ctx.close()


def _kitti_ctx(max_batch):
    c = synth.KITTI
    return api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=max_batch)


@pytest.fixture(scope="module")
def kitti_sequence():
    """a 256-frame KITTI-shaped sequence whose 64-pair pool repeats (frame f = pair f mod 64)"""
    c = synth.KITTI
    pool_l, pool_r = synth.synth_stereo_pool(c["height"], c["width"], 64, seed0=70, disparity=9)
    idx = np.arange(256) % 64
    return pool_l, pool_r, np.ascontiguousarray(pool_l[idx]), np.ascontiguousarray(pool_r[idx])


def _oracle_vocab(oracle, V):
    a, i = V.arrays(), V.info()
    return oracle.Vocabulary(i["k"], i["L"], a["parent"], a["is_leaf"], a["desc"], a["weight"])


@pytest.mark.gpu
def test_cuda_database_on_a_sequence_and_the_resident_frame_query(oracle, kitti_sequence):
    pool_l, pool_r, lefts, rights = kitti_sequence
    F = len(lefts)
    ctx = _kitti_ctx(8)
    N = ctx.n_features
    res = ctx.sequence_stereo_ptr(F, lefts.ctypes.data, rights.ctypes.data, lefts.strides[1], lefts.strides[0])
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=10, L=5, seed=4)
    epoch = ctx.frame_epoch
    D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=N)
    assert ctx.frame_epoch == epoch
    gd = ctx.read_device(res.gathered_desc, (F, N, 32), np.uint8)
    gn = ctx.read_device(res.gathered_n, (F,), np.int32)
    O = _oracle_vocab(oracle, V)
    db = R.bow_arrays(oracle, O, gd, gn)
    for window, top_k, min_score in [(0, 10, 0.0), (70, 3, 0.0), (2, F, 0.05)]:
        exp = R.oracle_query(db, db, 0, window, min_score, top_k)
        _assert_same(D.query(0, F, top_k, window, min_score), exp, f"window {window}")
    # every frame finds its three copies (f +- 64 k) first, all with one score
    r = D.query(0, F, 3, 0)
    for f in range(F):
        assert sorted(r["cand_frame"][f]) == [g for g in range(f % 64, F, 64) if g != f], f
        assert len(set(r["cand_score"][f].tolist())) == 1
    # relocalisation: a pool pair as the context's resident frame, its bag of words from the database's vocabulary
    j = 5
    fr = ctx.stereo_frame(pool_l[j], pool_r[j])
    bow = ctx.bow_transform(V)
    D2 = api.BowDatabase.build(ctx, V, gd, gn)  # building leaves the resident frame and its bag of words alone
    q = R.bow_arrays(oracle, O, fr.desc_left[None], np.array([len(fr.desc_left)], np.int32))
    for top_k in (4, 10):
        exp = R.oracle_query(db, q, 0, -1, 0.0, top_k)
        _assert_same(D.query_frame(0, top_k), exp, "resident frame")
        _assert_same(D2.query_frame(0, top_k), exp, "resident frame, second database")
    assert sorted(D.query_frame(0, 4)["cand_frame"][0]) == [j, j + 64, j + 128, j + 192]
    # searchByBow on the resident frame still works after the builds
    again = ctx.search_by_bow(bow, fr.desc_left)
    assert len(again["kf_idx"]) > 100 and (again["best_dist"] == 0).all()
    # the epoch moves on: the resident bag of words is gone
    ctx.stereo_frame(pool_l[j], pool_r[j])
    with pytest.raises(ValueError, match="invalid state"):
        D.query_frame(0, 4)
    # another vocabulary's bag of words is not the database's
    W = api.Vocabulary.build(ctx, gd, gn, k=10, L=3, seed=1)
    ctx.bow_transform(W)
    with pytest.raises(ValueError, match="invalid state"):
        D.query_frame(0, 4)
    for o in (D, D2, V, W, ctx):
        o.close()


@pytest.mark.gpu
def test_cuda_two_local_ranks_query_their_blocks(kitti_sequence):
    _, _, lefts, rights = kitti_sequence
    F = 96
    lefts, rights = lefts[:F], rights[:F]
    ranks = [_kitti_ctx(4) for _ in range(2)]
    comms = api.Communicator.local(ranks, F)
    results = []
    for r in range(2):
        blk = api.frame_range(F, r, 2)
        lo = lefts[blk.start : blk.stop]
        results.append(ranks[r].sequence_stereo_ptr(F, lo.ctypes.data, rights[blk.start : blk.stop].ctypes.data, lo.strides[1], lo.strides[0], comms[r]))
    parts, whole = [], None
    for r in range(2):
        ctx, res = ranks[r], results[r]
        V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=ctx.n_features, k=10, L=4, seed=2)
        D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=ctx.n_features)
        blk = api.frame_range(F, r, 2)
        parts.append(D.query(blk.start, blk.stop, 5, 1))
        if r == 0:
            whole = D.query(0, F, 5, 1)
        D.close()
        V.close()
    for k in OUT:
        assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), k
    assert (whole["n_kept"][:32] > 0).all()  # frames 0..31 have a copy 64 frames on
    for o in comms + ranks:
        o.close()


@pytest.mark.gpu
def test_cuda_database_at_the_frame_limit(oracle, cases):
    """ORBX_BOWDB_MAX_FRAMES one-word frames: the counters fill the query kernel's shared memory and the candidate lists
    (up to a third of the frames) live in global scratch; one more frame is refused"""
    c = cases["loop"]
    ctx = _small_ctx()
    V = api.Vocabulary(ctx, **c["voc"])
    _, pool, _ = R.word_descriptors(oracle, c["voc"])
    F = api.BOWDB_MAX_FRAMES
    f = np.arange(F)
    desc = np.zeros((F, 2, 32), np.uint8)
    desc[:, 0] = np.asarray(pool)[f % 3]
    desc[:, 1] = np.asarray(pool)[3 + f % 61]
    counts = np.where(f % 11 == 4, 1, 2).astype(np.int32)
    D = api.BowDatabase.build(ctx, V, desc, counts)
    db = R.bow_arrays(oracle, c["O"], desc, counts)
    for lo, hi, top_k, window in [(0, 6, 10, 1), (F - 40, F, 3, 0), (1003, 1006, F, 5)]:
        exp = R.oracle_query(db, {k: db[k][lo:hi] for k in ("ids", "vals", "n")}, lo, window, 0.0, top_k)
        _assert_same(D.query(lo, hi, top_k, window), exp, f"{lo}..{hi}")
    assert exp["n_scored"].max() > 30000  # frame 1005 holds one word: every frame sharing it is scored
    D.close()
    with pytest.raises(ValueError, match="ORBX_BOWDB_MAX_FRAMES"):
        api.BowDatabase.build(ctx, V, np.zeros((F + 1, 1, 32), np.uint8), np.ones(F + 1, np.int32))
    V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_database_rejects_bad_arguments(cases):
    c = cases["loop"]
    ctx = _small_ctx()
    V = api.Vocabulary(ctx, **c["voc"])
    desc, counts = c["desc"], c["counts"]
    F = len(counts)
    with pytest.raises(ValueError, match="invalid argument"):
        api.BowDatabase.build(ctx, V, desc[:0], counts[:0])
    bad = counts.copy()
    bad[3] = desc.shape[1] + 1
    with pytest.raises(ValueError, match="invalid argument"):
        api.BowDatabase.build(ctx, V, desc, bad)
    bad[3] = -1
    with pytest.raises(ValueError, match="invalid argument"):
        api.BowDatabase.build(ctx, V, desc, bad)
    import torch

    d_desc, d_bad = torch.from_numpy(np.ascontiguousarray(desc)).cuda(), torch.from_numpy(np.ascontiguousarray(bad, np.int32)).cuda()
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match=r"invalid argument \(keyframe database: a count lies outside 0\.\.stride"):  # the same counts in device memory
        api.BowDatabase.build(ctx, V, d_desc.data_ptr(), d_bad.data_ptr(), n_frames=F, stride=desc.shape[1])
    with pytest.raises(ValueError, match="invalid argument"):  # stride outside 1..ORBX_BOW_MAX_STRIDE
        api.BowDatabase.build(ctx, V, np.zeros((1, api.BOW_MAX_STRIDE + 1, 32), np.uint8), np.zeros(1, np.int32))
    D = api.BowDatabase.build(ctx, V, desc, counts)
    for args in [(0, F + 1, 3, 1), (-1, 2, 3, 1), (3, 2, 3, 1), (0, F, 0, 1), (0, F, F + 1, 1), (0, F, 3, -1), (0, F, 3, 1, float("nan"))]:
        with pytest.raises(ValueError, match="invalid argument"):
            D.query(*args)
    with pytest.raises(ValueError, match="invalid argument"):
        D.query_frame(-1, 3)
    with pytest.raises(ValueError, match="invalid state"):  # no resident bag of words
        D.query_frame(0, 3)
    assert D.query(4, 4, 3)["n_kept"].size == 0  # an empty range enqueues nothing
    # a vocabulary or a database of another context
    other = _small_ctx()
    W = api.Vocabulary(other, **c["voc"])
    with pytest.raises(ValueError, match="another context"):
        api.BowDatabase.build(ctx, W, desc, counts)
    E = api.BowDatabase.build(other, W, desc, counts)
    with pytest.raises(ValueError, match="another context"):
        E.ctx = ctx
        E.query(0, F, 3, 1)
    for o in (D, E, W, V, other, ctx):
        o.close()
