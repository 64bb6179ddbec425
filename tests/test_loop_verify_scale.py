"""Loop verification (orbx_loopver_*) at the benchmark's frame size and beyond one pass of the verifier's block structure.

tests/test_loop_verify.py holds the CUDA verifier to tests/loopver_oracle.c on record sets of at most 128 features, and on
tables whose pairs each get a CTA of their own.  There, every block scan of loopver_pair_kernel (the kept rows, the
correspondences) and the chunk carry of verify_angle_block run a single chunk of 256, no CTA verifies a second pair after
another, and nothing asserts where in the rounds of eight hypotheses a RANSAC stops.  Here:

  CPU  crafted_large (tests/loopver_restatement.py) reaches 0 / 255 / 256 / 257 / 512 / 513 / 2000 features per frame,
       kept rows, matches and correspondences on both sides of 256 and 512, getBestMatch over several 32-lane chunks, and
       hypotheses that stop at every position of a round of eight; a census over the oracle's outputs asserts that they do.
  GPU  the CUDA verifier equals the oracle bit for bit (T as uint64) on those sets, with host and device io; on a table of
       more than four pairs per resident CTA with the pair kinds shuffled; on bench.py's KITTI shape through the device
       pipeline (records, vocabulary, keyframe database, table); with any subset of the host-copied outputs; and for
       back-to-back calls on one stream, including one that grows the verifier's staging buffer.
"""
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

import loop_scenes as S
import loopver_restatement as R

OUT = api.LOOPVER_OUTPUTS
N_LARGE, LEVELS_LARGE = 2000, 8
# the builder's seed and the configs' RANSAC seeds, chosen by scanning seeds with oracle_loopver so that every config
# reaches every case of the census below (test_large_sets_reach_the_kernels_structure fails if the builder or the oracle
# drifts off them)
LARGE_SEED, LARGE_PARAM_SEEDS = 3, (1, 11, 21)


@pytest.fixture(scope="module")
def large(oracle):
    c = R.crafted_large(oracle.KP_DTYPE, N_LARGE, LEVELS_LARGE, seed=LARGE_SEED, param_seeds=LARGE_PARAM_SEEDS)
    c["O"] = oracle.Vocabulary(**c["voc"])
    c["sf"] = oracle.scale_factors(R.SCALE, LEVELS_LARGE)
    c["exp"] = [R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], prm) for prm in c["configs"]]
    return c


def _assert_same(got, exp, what=""):
    for k in OUT:
        g, e = np.asarray(got[k]).reshape(np.shape(exp[k])), exp[k]
        if k == "T":
            assert np.array_equal(g.view(np.uint64), e.view(np.uint64)), f"{what} T bits"
        else:
            assert np.array_equal(g, e), f"{what} {k}: {np.argwhere(g != e)[:8].tolist()}"


def _rows(exp, lo, hi):
    return {k: v[lo:hi] for k, v in exp.items()}


def census(fr, table, prm, r) -> dict:
    """how often each piece of the verifier's structure is reached by one config's oracle outputs"""
    h, it, acc = r["hypothesis"], r["n_iters"], r["accepted"] == 1
    ran = it > 0
    rej = ran & ~acc
    c = {
        "accepted_h_mod8_eq7": int((acc & (h % 8 == 7)).sum()),
        "accepted_h_mod8_eq0_h_ge8": int((acc & (h % 8 == 0) & (h >= 8)).sum()),
        "accepted_h_ge64": int((acc & (h >= 64)).sum()),
        "rejected_partial_last_round": int((rej & (it % 8 != 0) & (it > 8)).sum()),
        "rejected_at_max_iterations": int((rej & (it == prm["max_iterations"])).sum()),
        "rejected_maxima_tie_across_rounds": int((rej & (h // 8 > r["first_best"] // 8)).sum()),
        "empty_slot": int((table < 0).sum()),
        "candidate_is_query": int((table == np.arange(len(table))[:, None]).sum()),
        "empty_frame_query": int(sum(1 for q in range(len(table)) if fr["n"][q] == 0 and (table[q] >= 0).any())),
        "loop_frame_by_rounds_of_5_not_8": 0,
    }
    for q in range(len(table)):
        sl = np.flatnonzero(acc[q])
        if len(sl):
            by5 = min((int(h[q, s]) // 5, int(s)) for s in sl)[1]
            by8 = min((int(h[q, s]) // 8, int(s)) for s in sl)[1]
            assert r["loop_frame"][q] == table[q, by5]
            c["loop_frame_by_rounds_of_5_not_8"] += int(by5 != by8)
    live = table >= 0
    for k in ("n_bow", "n_matches", "n_corr"):
        v = r[k][live]
        for name, n in (("le256", (v <= 256).sum()), ("gt256", (v > 256).sum()), ("eq256", (v == 256).sum()), ("eq257", (v == 257).sum()),
                        ("gt512", (v > 512).sum())):
            c[f"{k}_{name}"] = int(n)
    return c


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_large_sets_reach_the_kernels_structure(large):
    c = large
    assert c["frames"]["kps"].shape[1] == N_LARGE and sorted(set(c["frames"]["n"].tolist()) & {0, 255, 256, 257, 512, 513, N_LARGE}) == [
        0, 255, 256, 257, 512, 513, N_LARGE]
    assert set(np.unique(c["frames"]["kps"]["octave"][c["frames"]["kps"]["size"] > 0]).tolist()) == set(range(LEVELS_LARGE))
    for prm, r in zip(c["configs"], c["exp"]):
        cen = census(c["frames"], c["table"], prm, r)
        print(prm, cen)
        assert all(n > 0 for n in cen.values()), (prm, {k: n for k, n in cen.items() if n == 0})


def test_large_rows_tie_across_chunks(oracle, large):
    """scene A's query holds five landmarks twice, far apart in their node's candidate list: their rows' two best distances
    tie (ratio 1), so ratio 0.75 drops them and ratio 1.0 keeps the first occurrence"""
    c = large
    fr, q, cf = c["frames"], 0, int(c["table"][0, 6])
    bq = oracle.bow_transform(c["O"], fr["desc"][q][: fr["n"][q]], c["levelsup"])
    bc = oracle.bow_transform(c["O"], fr["desc"][cf][: fr["n"][cf]], c["levelsup"])
    r = oracle.search_by_bow(bq, fr["desc"][q][: fr["n"][q]], bc, fr["desc"][cf][: fr["n"][cf]])
    tie = (r["ratio"] == 1.0) & (r["best_dist"] <= 50)
    assert tie.sum() == 5 and (r["best_dist"][tie] > 0).all()
    # the two features of each tie lie in different 32-lane chunks of their node's list
    pos = {}
    for j in range(len(bq["fv_nodes"])):
        for p, f in enumerate(bq["fv_feats"][bq["fv_start"][j] : bq["fv_start"][j + 1]]):
            pos[int(f)] = p
    assert np.diff(bq["fv_start"]).min() > 96  # every node's list spans more than three chunks
    d = fr["desc"][q][: fr["n"][q]]
    for i in r["best_idx"][tie]:
        a, b = sorted(np.flatnonzero((d == d[i]).all(1)).tolist(), key=pos.get)
        assert pos[a] // 32 != pos[b] // 32 and i == a
    by_ratio = {prm["ratio"]: e["n_bow"][0, 6] for prm, e in zip(c["configs"], c["exp"])}
    assert by_ratio[1.0] == by_ratio[0.75] + 5


def test_min_inliers_above_every_frame(large):
    c = large
    prm = R.params(min_inliers=N_LARGE + 1, min_matches=0, seed=LARGE_PARAM_SEEDS[0])
    r = R.oracle_verify(c["O"], c["levelsup"], c["frames"], R.CAM, c["sf"], 0, c["table"], prm)
    assert (r["n_iters"] == 0).all() and (r["hypothesis"] == -1).all() and (r["accepted"] == 0).all() and (r["n_inliers"] == 0).all()
    assert not r["T"].any() and (r["loop_frame"] == -1).all()
    assert (r["n_corr"] > 256).any()  # the correspondences were still gathered


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _large_ctx(**kw):
    return api.Context(320, 240, N_LARGE, LEVELS_LARGE, R.SCALE, camera=api.Camera(*R.CAM, 0.1), **kw)


def _device_outputs(torch, nq, k, N, names=OUT):
    t = {n: torch.full((nq, k), 7, dtype=torch.int32, device="cuda") for n in OUT[:7] if n in names}
    if "T" in names:
        t["T"] = torch.full((nq, k, 12), 7.0, dtype=torch.float64, device="cuda")
    if "match" in names:
        t["match"] = torch.full((nq, k, N), 7, dtype=torch.int32, device="cuda")
    if "loop_frame" in names:
        t["loop_frame"] = torch.full((nq,), 7, dtype=torch.int32, device="cuda")
    return t


def _device_call(torch, LV, table, names=OUT):
    """a device table and device outputs (only `names`; the others are passed as NULL) for one call"""
    nq, k = table.shape
    return torch.from_numpy(np.ascontiguousarray(table, np.int32)).cuda(), _device_outputs(torch, nq, k, LV.ctx.n_features, names)


def _launch(LV, q_lo, call, prm):
    tab, t = call
    LV.verify_ptr(q_lo, tab.shape[0], tab.data_ptr(), tab.shape[1], [t[n].data_ptr() if n in t else 0 for n in OUT], on_device=True, **prm)


def _fetch(call):
    return {n: v.cpu().numpy() for n, v in call[1].items()}


def _device_verify(torch, LV, q_lo, table, prm, names=OUT):
    call = _device_call(torch, LV, table, names)
    torch.cuda.synchronize()
    _launch(LV, q_lo, call, prm)
    LV.ctx.synchronize()
    return _fetch(call)


def _host_verify(LV, q_lo, table, prm, names):
    """orbx_loopver_verify with a host table and only `names` among the host outputs (the others NULL)"""
    tab = np.ascontiguousarray(table, np.int32)
    nq, k, N = tab.shape[0], tab.shape[1], LV.ctx.n_features
    shapes = {n: (nq, k) for n in OUT[:7]} | dict(T=(nq, k, 12), match=(nq, k, N), loop_frame=(nq,))
    out = {n: np.full(shapes[n], 7, np.float64 if n == "T" else np.int32) for n in names}
    LV.verify_ptr(q_lo, nq, tab.ctypes.data, k, [out[n].ctypes.data if n in out else 0 for n in OUT], on_device=False, **prm)
    return out


@pytest.fixture(scope="module")
def large_gpu(large):
    import torch

    ctx = _large_ctx()
    assert np.array_equal(ctx.scaled_factors(), large["sf"])
    V = api.Vocabulary(ctx, **large["voc"])
    rec = R.to_records(ctx, large["frames"])
    LV = api.LoopVerifier.build(ctx, V, rec, len(rec), levelsup=large["levelsup"])
    yield dict(torch=torch, ctx=ctx, V=V, LV=LV, rec=rec)
    for o in (LV, V, ctx):
        o.close()


@pytest.mark.gpu
def test_cuda_verifier_equals_oracle_on_large_sets(large, large_gpu):
    c, g = large, large_gpu
    torch, ctx, V = g["torch"], g["ctx"], g["V"]
    F = len(g["rec"])
    d_rec = torch.from_numpy(g["rec"].view(np.uint8).reshape(F, -1).copy()).cuda()
    torch.cuda.synchronize()
    LVd = api.LoopVerifier.build(ctx, V, d_rec.data_ptr(), F, levelsup=c["levelsup"])
    lo, hi = 11, 47
    for LV in (g["LV"], LVd):
        for prm, exp in zip(c["configs"], c["exp"]):
            _assert_same(LV.verify(0, c["table"], **prm), exp, f"host {prm}")
            _assert_same(_device_verify(torch, LV, 0, c["table"], prm), exp, f"device {prm}")
            _assert_same(LV.verify(lo, c["table"][lo:hi], **prm), _rows(exp, lo, hi), f"sub-range {prm}")
    LVd.close()


def _stride_set(kp_dtype, n_queries: int, top_k: int, seed: int = 5) -> dict:
    """frames of at most 128 features (and a few of 2000) at N_LARGE capacity, replicated so that every frame is a query;
    each row draws its candidates at random from its group's frames, so the pair kinds mix in shuffled order"""
    B = R._Builder(seed, kp_dtype, N_LARGE, LEVELS_LARGE)
    Rc, tc = R.rot([0.2, 1, 0.1], 8.0), np.array([0.25, -0.05, 0.1])

    def pair(lms, **kw):
        return B.frame(lms, Rc, tc, spin=8.0, **kw)

    L0, L1, L2 = B.box(60), B.box(100), B.box(1500)
    groups = [
        # accepted at the first hypothesis; 19 matches (stop at min_matches); 15 correspondences (below min_inliers)
        [B.frame(L0), pair(L0[:30]), pair(L0[:19]), pair(L0[:40], no_depth=set(range(25)))],
        # 30 inliers of 100 (accepted late); 20 of 100 (never accepted in 300 hypotheses)
        [B.frame(L1)] + [pair(L1, wrong=set(B.rng.choice(100, 70, replace=False).tolist())) for _ in range(3)]
        + [pair(L1, wrong=set(range(20, 100)))],
        # 1500 matches
        [B.frame(L2, extra=N_LARGE - 1500), pair(L2, extra=0)],
    ]
    base = B.arrays()
    nb = len(base["n"])
    group_of = np.zeros(nb, int)
    for gi, fs in enumerate(groups):
        group_of[fs] = gi
    reps = -(-n_queries // nb)
    fr = {k: np.concatenate([v] * reps)[:n_queries] for k, v in base.items()}
    F = n_queries
    gid = group_of[np.arange(F) % nb]
    members = [np.flatnonzero(gid == gi) for gi in range(len(groups))]
    rng = np.random.default_rng(seed)
    table = np.full((F, top_k), -1, np.int32)
    for f in range(F):
        g = gid[f]
        if g == 2 and rng.random() < 0.9:  # the 2000-feature pairs stay few: most of their rows are empty
            continue
        n = int(rng.integers(top_k // 2, top_k + 1))
        table[f, :n] = rng.choice(members[g], n)
        rng.shuffle(table[f])
    return dict(frames=fr, table=table, levelsup=2, voc=synth.synth_vocabulary(10, 3, 21))


@pytest.mark.gpu
def test_cuda_grid_stride_reuses_cta_state_across_pair_kinds(oracle):
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    top_k = 16
    n_queries = (4 * 8 * sms) // top_k + 1  # 8 CTAs of 256 threads fill an SM's 2048 threads
    c = _stride_set(oracle.KP_DTYPE, n_queries, top_k)
    n_pairs = c["table"].size
    assert n_pairs > 4 * 8 * sms, (n_pairs, sms)
    ctx = _large_ctx()
    V = api.Vocabulary(ctx, **c["voc"])
    rec = R.to_records(ctx, c["frames"])
    LV = api.LoopVerifier.build(ctx, V, rec, len(rec), levelsup=c["levelsup"])
    O = oracle.Vocabulary(**c["voc"])
    prm = R.params(seed=13)
    exp = R.oracle_verify(O, c["levelsup"], c["frames"], R.CAM, ctx.scaled_factors(), 0, c["table"], prm)
    live = c["table"] >= 0
    acc = exp["accepted"] == 1
    kinds = dict(empty_slot=~live, below_min_matches=live & (exp["n_matches"] < prm["min_matches"]) & (exp["n_matches"] > 0),
                 corr_below_min_inliers=(exp["n_matches"] >= prm["min_matches"]) & (exp["n_corr"] < prm["min_inliers"]),
                 accepted_first=acc & (exp["hypothesis"] == 0), accepted_late=acc & (exp["hypothesis"] >= 8),
                 rejected_after_300=~acc & (exp["n_iters"] == 300), matches_over_512=exp["n_matches"] > 512)
    counts = {k: int(v.sum()) for k, v in kinds.items()}
    print(dict(n_pairs=n_pairs, sms=sms, **counts))
    assert all(counts.values()), counts
    _assert_same(_device_verify(torch, LV, 0, c["table"], prm), exp, "grid-stride device io")
    _assert_same(LV.verify(0, c["table"], **prm), exp, "grid-stride host io")
    for o in (LV, V, ctx):
        o.close()


NULL_SETS = [("T",), ("match",), ("loop_frame",), ("accepted",), ("T", "loop_frame"), ("match", "loop_frame")]


@pytest.mark.gpu
def test_cuda_verifier_with_null_outputs(large, large_gpu):
    """any output may be NULL: each subset equals the full call, for host io (whose staging offsets depend on which outputs
    are given) and for device io"""
    c, g = large, large_gpu
    torch, LV = g["torch"], g["LV"]
    prm, exp = c["configs"][0], c["exp"][0]
    for names in NULL_SETS:
        got = _host_verify(LV, 0, c["table"], prm, names)
        assert set(got) == set(names)
        for n in names:
            e = exp[n]
            assert np.array_equal(got[n].view(np.uint64), e.view(np.uint64)) if n == "T" else np.array_equal(got[n], e), f"host {names}: {n}"
        got = _device_verify(torch, LV, 0, c["table"], prm, names)
        for n in names:
            e = exp[n]
            assert np.array_equal(got[n].view(np.uint64), e.view(np.uint64)) if n == "T" else np.array_equal(got[n], e), f"device {names}: {n}"


@pytest.mark.gpu
def test_cuda_back_to_back_device_calls(large, large_gpu):
    """two device-io calls with other params and tables, enqueued with no synchronisation between them; then, on a stream
    set with ctx.set_stream, a small call followed by one whose table grows the verifier's staging buffer"""
    c, g = large, large_gpu
    torch, ctx, V = g["torch"], g["ctx"], g["V"]
    (p0, p1), (e0, e1) = c["configs"][:2], c["exp"][:2]
    lo, hi = 11, 47
    LV = api.LoopVerifier.build(ctx, V, g["rec"], len(g["rec"]), levelsup=c["levelsup"])
    a, b = _device_call(torch, LV, c["table"]), _device_call(torch, LV, c["table"][lo:hi])
    torch.cuda.synchronize()
    _launch(LV, 0, a, p0)
    _launch(LV, lo, b, p1)
    ctx.synchronize()
    _assert_same(_fetch(a), e0, "first call")
    _assert_same(_fetch(b), _rows(e1, lo, hi), "second call")
    LV.close()
    LV = api.LoopVerifier.build(ctx, V, g["rec"], len(g["rec"]), levelsup=c["levelsup"])
    a, b = _device_call(torch, LV, c["table"][lo:hi]), _device_call(torch, LV, c["table"])
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    ctx.set_stream(s.cuda_stream)
    try:
        _launch(LV, lo, a, p0)
        _launch(LV, 0, b, p1)  # more pairs than the first call: the staging buffer grows
        s.synchronize()
    finally:
        ctx.set_stream(None)
    _assert_same(_fetch(a), _rows(e0, lo, hi), "small call on a user stream")
    _assert_same(_fetch(b), e1, "growing call on a user stream")
    LV.close()


@pytest.mark.gpu
def test_cuda_verifier_at_the_benchmark_shape_through_the_device_pipeline(oracle):
    """bench.py's KITTI configuration (1241x376, 2000 features, 8 levels, synth.KITTI's camera): device records of a stereo
    sequence, a k = 10, L = 6 vocabulary built from them, the keyframe database's top 10 outside the window as a device
    table, and the verifier on it, against the oracle on 36 queries from the start, the middle and the end.  The sequence is
    16 synthetic pairs repeated as bench.py repeats its pool (candidates that are exact copies: accepted at the first
    hypothesis), then a rendered walk around a room at the same shape, whose frames overlap only partly."""
    import torch

    k = synth.KITTI
    H, W = k["height"], k["width"]
    cam = dict(w=W, h=H, fx=k["fx"], fy=k["fy"], cx=k["cx"], cy=k["cy"])
    P, n_copies, n_walk = 16, 64, 48
    pool_l, pool_r = synth.synth_stereo_pool(H, W, P, seed0=0)
    walls = S._walls(1)
    walk = [S.stereo(walls, *S.pose(i, n_walk), bl=k["bl"], **cam) for i in range(n_walk)]
    left = np.ascontiguousarray(np.concatenate([pool_l[np.arange(n_copies) % P], np.stack([a for a, _ in walk])]))
    right = np.ascontiguousarray(np.concatenate([pool_r[np.arange(n_copies) % P], np.stack([b for _, b in walk])]))
    F = len(left)
    ctx = api.Context(W, H, k["n_features"], k["n_levels"], k["scale_factor"], camera=api.Camera(k["fx"], k["fy"], k["cx"], k["cy"], k["bl"]),
                      max_batch=16)
    N, lay = ctx.n_features, ctx.record_layout()
    d_left, d_right = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
    d_rec = torch.zeros((F, lay.record_bytes), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    res = ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, W * H, None, True, d_rec.data_ptr(), lay.record_bytes, True)
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=10, L=6, seed=0)
    D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=N)
    top_k, window, levelsup = 10, 3, 4
    cand = torch.zeros((F, top_k), dtype=torch.int32, device="cuda")
    D.query_ptr(0, F, top_k, window, 0.0, [cand.data_ptr()] + [0] * 6, on_device=True)
    LV = api.LoopVerifier.build(ctx, V, d_rec.data_ptr(), F, levelsup=levelsup)
    prm = R.params(seed=17)
    ctx.synchronize()
    table = cand.cpu().numpy()
    got = _device_verify(torch, LV, 0, table, prm)
    rec = d_rec.cpu().numpy().view(ctx.record_dtype()).reshape(F)
    fr = dict(kps=rec["kps_left"], desc=rec["desc_left"], depth=rec["depth"], n=rec["n_left"])
    a, i = V.arrays(), V.info()
    O = oracle.Vocabulary(i["k"], i["L"], a["parent"], a["is_leaf"], a["desc"], a["weight"])
    camo = (ctx.camera.fx, ctx.camera.fy, ctx.camera.cx, ctx.camera.cy)
    blocks = [(0, 12), (F // 2 - 6, F // 2 + 6), (F - 12, F)]
    for lo, hi in blocks:
        exp = R.oracle_verify(O, levelsup, fr, camo, ctx.scaled_factors(), lo, table[lo:hi], prm)
        _assert_same(_rows(got, lo, hi), exp, f"queries {lo}..{hi - 1}")
    q = np.r_[tuple(np.arange(lo, hi) for lo, hi in blocks)]
    live = table[q] >= 0
    walk_rows = q >= n_copies
    stats = dict(pairs=int(live.sum()), n_matches_gt512=int((got["n_matches"][q] > 512).sum()), accepted=int(got["accepted"][q].sum()),
                 walk_pairs=int(live[walk_rows].sum()), walk_accepted=int(got["accepted"][q][walk_rows].sum()),
                 walk_hyp_gt0=int((got["hypothesis"][q][walk_rows] > 0).sum()))
    print(stats)
    assert stats["n_matches_gt512"] > 0 and stats["walk_pairs"] > 0
    for o in (LV, D, V, ctx):
        o.close()
