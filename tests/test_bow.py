"""Bag-of-words transform (SURVEY.md section 8(f) rank 3): DBoW3 Vocabulary::transform as the reference calls it
(include/ORB_SLAM2/Frame.h:224-231, levelsup = 4).

PARITY UNPINNED: DBoW3 is un-vendored and the reference ships no vocabulary.  CPU: the plain-C restatement of DBoW3's
published algorithm equals an independent, literal python restatement (dict = std::map) on synthetic vocabularies.
GPU: the CUDA kernels equal the oracle bit for bit (ids, double weights, feature lists)."""
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth


def _features(V, n, seed, flip=8):
    """descriptors near random leaves of the tree (so the descent is meaningful), plus a few random ones"""
    rng = np.random.default_rng(seed)
    leaves = np.nonzero(V.word_id >= 0)[0]
    d = V.desc[rng.choice(leaves, n)].copy()
    bits = rng.integers(0, 256, (n, flip))
    for b in range(flip):
        d[np.arange(n), bits[:, b] // 8] ^= (1 << (bits[:, b] % 8)).astype(np.uint8)
    d[:: 17] = rng.integers(0, 256, (len(d[::17]), 32), dtype=np.uint8)
    return d


def _py_transform(V, desc, levelsup):
    """literal DBoW3: per-feature descent (first minimum), BowVector::addWeight, normalize(L1), FeatureVector::addFeature"""
    bow, fv = {}, {}
    nid_level = V.L - levelsup
    for i, f in enumerate(desc):
        node, level, at = 0, 0, 0
        while True:
            level += 1
            ch = V.child_ids[V.child_start[node] : V.child_start[node + 1]]
            dist = np.unpackbits(V.desc[ch] ^ f, axis=1).sum(1)
            node = int(ch[int(np.argmin(dist))])  # argmin returns the first minimum
            if level == nid_level:
                at = node
            if V.child_start[node] == V.child_start[node + 1]:
                break
        w = float(V.weight[node])
        if w > 0:
            wid = int(V.word_id[node])
            bow[wid] = bow[wid] + w if wid in bow else w
            fv.setdefault(0 if nid_level <= 0 else at, []).append(i)
    ids = sorted(bow)
    vals = np.array([bow[k] for k in ids], np.float64)
    norm = 0.0
    for x in vals:
        norm += abs(x)
    if norm > 0:
        vals = vals / norm
    return ids, vals, fv


VOCS = [(10, 3, 1), (6, 4, 2), (3, 6, 3), (40, 2, 4)]


@pytest.mark.parametrize("kLs", VOCS, ids=[f"k{k}L{L}" for k, L, _ in VOCS])
def test_oracle_equals_literal_restatement(oracle, kLs):
    k, L, seed = kLs
    V = oracle.Vocabulary(**synth.synth_vocabulary(k, L, seed))
    assert (V.weight[V.word_id >= 0] == 0).any()  # stopped words present
    d = _features(V, 400, seed)
    for levelsup in (4, 2, 0, L, L + 3):
        r = oracle.bow_transform(V, d, levelsup)
        ids, vals, fv = _py_transform(V, d, levelsup)
        assert ids == list(r["bow_ids"]) and np.array_equal(vals, r["bow_vals"])
        assert sorted(fv) == list(r["fv_nodes"])
        for j, node in enumerate(sorted(fv)):
            assert fv[node] == list(r["fv_feats"][r["fv_start"][j] : r["fv_start"][j + 1]])
        assert abs(r["bow_vals"].sum() - 1.0) < 1e-12
    r = oracle.bow_transform(V, d[:0], 4)
    assert len(r["bow_ids"]) == 0 and len(r["fv_nodes"]) == 0


def _same(got, exp, what):
    for key in ("bow_ids", "bow_vals", "fv_nodes", "fv_start", "fv_feats"):
        assert np.array_equal(got[key], exp[key]), f"{what}: {key}"


@pytest.mark.gpu
def test_cuda_bow_equals_oracle(oracle, tmp_path):
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 6, 17)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]))
    r = ctx.stereo_frame(left, right)
    for k, L, seed in VOCS:
        voc = synth.synth_vocabulary(k, L, seed)
        # make the frame's descriptors meaningful for this tree: half of the leaves' descriptors become frame descriptors
        O = oracle.Vocabulary(**voc)
        leaves = np.nonzero(O.word_id >= 0)[0]
        rng = np.random.default_rng(seed)
        take = rng.choice(len(r.desc_left), min(len(leaves), 1200), replace=False)
        voc["desc"][leaves[: len(take)] - 1] = r.desc_left[take]
        O = oracle.Vocabulary(**voc)
        V = api.Vocabulary(ctx, **voc)
        assert V.info() == dict(k=k, L=L, n_nodes=O.n_nodes, n_words=int((O.word_id >= 0).sum()))
        for levelsup in (4, 2, 0, L + 1):
            _same(ctx.bow_transform(V, levelsup=levelsup), oracle.bow_transform(O, r.desc_left, levelsup), f"k{k} L{L} up{levelsup}")
        got = ctx.bow_transform(V)
        assert len(got["bow_ids"]) > 100 and abs(got["bow_vals"].sum() - 1.0) < 1e-12
        # the text format round trip (DBoW3 / ORB-SLAM2 ORBvoc.txt layout)
        if O.n_nodes < 3000:
            path = synth.write_vocabulary_text(str(tmp_path / f"voc_{k}_{L}.txt"), voc)
            V2 = api.Vocabulary.load_text(ctx, path)
            assert V2.info() == V.info()
            _same(ctx.bow_transform(V2), got, "text loader")
            V2.close()
        V.close()
    with pytest.raises(api.FileNotOpenError):
        api.Vocabulary.load_text(ctx, str(tmp_path / "missing.txt"))
    ctx.close()


def _read_device_bow(ctx, d, n):
    """the n frames of a bow_transform_batch_device result as bow_transform dicts"""
    N = d.stride
    nb = ctx.read_device(d.n_bow, (n,), np.int32)
    nf = ctx.read_device(d.n_fv_nodes, (n,), np.int32)
    ids = ctx.read_device(d.bow_ids, (n, N), np.int32)
    vals = ctx.read_device(d.bow_vals, (n, N), np.float64)
    fnodes = ctx.read_device(d.fv_nodes, (n, N), np.int32)
    fstart = ctx.read_device(d.fv_start, (n, N + 1), np.int32)
    ffeats = ctx.read_device(d.fv_feats, (n, N), np.int32)
    return [dict(bow_ids=ids[f, : nb[f]], bow_vals=vals[f, : nb[f]], fv_nodes=fnodes[f, : nf[f]], fv_start=fstart[f, : nf[f] + 1],
                 fv_feats=ffeats[f, : fstart[f, nf[f]]]) for f in range(n)]


@pytest.mark.gpu
def test_cuda_bow_batch_device_rgbd_and_empty(oracle):
    import torch

    c = synth.KITTI
    n = 3
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=120)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=n)
    host = ctx.stereo_batch(lefts, rights)
    voc = synth.synth_vocabulary(10, 4, 9)
    O, V = oracle.Vocabulary(**voc), api.Vocabulary(ctx, **voc)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    before = ctx.launch_count
    d = ctx.bow_transform_batch_device(V, n, 4)
    assert ctx.launch_count - before == 2
    for f, got in enumerate(_read_device_bow(ctx, d, n)):
        _same(got, oracle.bow_transform(O, host.desc_left[f][: host.n_left[f]], 4), f"frame {f}")
    # searchByBow against a frame of the batch other than frame 0 (frame 2 vs frame 0's features as the "keyframe")
    e2, e0 = oracle.bow_transform(O, host.desc_left[2][: host.n_left[2]], 4), oracle.bow_transform(O, host.desc_left[0][: host.n_left[0]], 4)
    got = ctx.search_by_bow(e0, host.desc_left[0][: host.n_left[0]], frame=2)
    exp = oracle.search_by_bow(e2, host.desc_left[2][: host.n_left[2]], e0, host.desc_left[0][: host.n_left[0]])
    for key in exp:
        assert np.array_equal(got[key], exp[key], equal_nan=True), key
    ctx.set_stream(None)
    # RGB-D frames (one image per frame): same transform
    t = synth.TUM
    rg = api.Context(t["width"], t["height"], 1000, 8, 1.2, camera=api.Camera(t["fx"], t["fy"], t["cx"], t["cy"], t["bl"], (0.0,) * 5, t["depth_scale"]))
    fr = rg.rgbd_frame(synth.synth_image(t["height"], t["width"], 3), synth.synth_depth_u16(t["height"], t["width"], 3, t["depth_scale"]))
    Vr = api.Vocabulary(rg, **voc)
    _same(rg.bow_transform(Vr), oracle.bow_transform(O, fr.desc, 4), "rgbd")
    Vr.close()
    rg.close()
    # a frame without keypoints: empty vectors
    ctx.stereo_frame(np.full((c["height"], c["width"]), 80, np.uint8), np.full((c["height"], c["width"]), 80, np.uint8))
    got = ctx.bow_transform(V)
    assert len(got["bow_ids"]) == 0 and len(got["fv_nodes"]) == 0 and len(got["fv_feats"]) == 0
    V.close()
    ctx.close()


_POP = np.array([bin(i).count("1") for i in range(256)], np.uint8)


def _shared_minima(O, desc) -> int:
    """descriptors whose descent meets, at some level, the smallest distance at two children (where the first among equals
    decides), found by a numpy descent of all of them at once"""
    node = np.zeros(len(desc), np.int64)
    tie = np.zeros(len(desc), bool)
    live = np.ones(len(desc), bool)
    kmax = int(np.diff(O.child_start).max())
    while live.any():
        i = np.nonzero(live)[0]
        c0, c1 = O.child_start[node[i]], O.child_start[node[i] + 1]
        j = c0[:, None] + np.arange(kmax)
        ok = j < c1[:, None]
        ids = O.child_ids[np.where(ok, j, c0[:, None])]
        d = _POP[O.desc[ids] ^ desc[i][:, None]].sum(-1, dtype=np.int32)
        d[~ok] = 1 << 20
        tie[i] |= (d == d.min(1)[:, None]).sum(1) > 1
        node[i] = ids[np.arange(len(i)), d.argmin(1)]
        live[i] = O.child_start[node[i]] != O.child_start[node[i] + 1]
    return int(tie.sum())


@pytest.mark.gpu
def test_cuda_bow_at_the_bench_shape(oracle):
    """bench.py's transform: 64 KITTI stereo frames of up to 2000 features in one bow_transform_batch_device call, on the
    k = 10, L = 6 synthetic vocabulary of about a million nodes"""
    import torch

    c = synth.KITTI
    n = 64
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=0)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=n)
    voc = synth.synth_vocabulary(10, 6, 0)
    O, V = oracle.Vocabulary(**voc), api.Vocabulary(ctx, **voc)
    assert O.n_nodes > 900000
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    torch.cuda.synchronize()
    res = ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    N = ctx.n_features
    desc = ctx.read_device(res.desc, (2 * n, N, 32), np.uint8)[0::2]  # image 2f = frame f's left image
    nk = ctx.read_device(res.n_kps, (2 * n,), np.int32)[0::2]
    assert nk.min() > 1000
    got = _read_device_bow(ctx, ctx.bow_transform_batch_device(V, n, 4), n)
    for f in range(n):
        _same(got[f], oracle.bow_transform(O, desc[f][: nk[f]], 4), f"frame {f}")
    assert sum(len(g["bow_ids"]) for g in got) > 50000
    for up in (0, 6):
        f = 37
        _same(ctx.bow_transform(V, frame=f, levelsup=up), oracle.bow_transform(O, desc[f][: nk[f]], up), f"frame {f} levelsup {up}")
    assert _shared_minima(O, np.concatenate([desc[f][: nk[f]] for f in range(n)])) > 0
    V.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_features", [4097, 5000, 16384])
def test_cuda_bow_past_4096_features(oracle, n_features):
    """frames of more than 4096 keypoints: bow_assemble_kernel sorts 8192 or 16384 keys in shared memory opted in past 48 KB"""
    h, w = 1200, 1600
    rng = np.random.default_rng(n_features)
    img = rng.integers(0, 256, (h, w), dtype=np.uint8)
    ctx = api.Context(w, h, n_features, 8, 1.2, camera=api.Camera(1000.0, 1000.0, w / 2, h / 2, 0.1))
    r = ctx.stereo_frame(img, np.ascontiguousarray(np.roll(img, -4, axis=1)))
    n = len(r.desc_left)
    assert n > 4096 and (n_features < 16384 or n > 8192), n
    voc = synth.synth_vocabulary(10, 4, 5)
    O0 = oracle.Vocabulary(**voc)
    leaves = np.nonzero(O0.word_id >= 0)[0]
    voc["desc"][leaves[:3000] - 1] = r.desc_left[rng.choice(n, 3000, replace=False)]  # leaves that the frame's features reach
    O, V = oracle.Vocabulary(**voc), api.Vocabulary(ctx, **voc)
    for up in (4, 0):
        _same(ctx.bow_transform(V, levelsup=up), oracle.bow_transform(O, r.desc_left, up), f"levelsup {up}")
    V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_database_at_stride_8193(oracle):
    """a keyframe database from host rows of 8193 descriptors, one frame full: the transform's sort of 16384 keys"""
    import bowdb_restatement as BR

    stride = 8193
    voc = synth.synth_vocabulary(10, 3, 6)
    O = oracle.Vocabulary(**voc)
    leaves = np.nonzero(O.word_id >= 0)[0]
    rng = np.random.default_rng(8193)
    pool = voc["desc"][rng.choice(leaves, 600, replace=False) - 1]
    counts = np.array([stride, 0, 3000, stride - 1, 40, 5000, 700], np.int32)
    desc = rng.integers(0, 256, (len(counts), stride, 32), dtype=np.uint8)
    for f, m in enumerate(counts):  # each frame from its own window of the pool: neighbours share words, far frames fewer
        desc[f, :m] = pool[(f * 60 + rng.integers(0, 200, m)) % len(pool)]
    ctx = api.Context(320, 240, 500, 4, 1.2, camera=api.Camera(300.0, 300.0, 160.0, 120.0, 0.1))
    V = api.Vocabulary(ctx, **voc)
    D = api.BowDatabase.build(ctx, V, desc, counts)
    db = BR.bow_arrays(oracle, O, desc, counts)
    assert D.info() == dict(n_frames=len(counts), n_words=db["n_words"], n_postings=int(db["n"].sum()))
    for window, min_score, top_k in [(0, 0.0, 6), (1, 0.0, 3), (0, 0.05, 2)]:
        exp = BR.oracle_query(db, db, 0, window, min_score, top_k)
        got = D.query(0, len(counts), top_k, window, min_score)
        for k in api.BOWDB_OUTPUTS:
            g, e = np.asarray(got[k]), exp[k]
            assert np.array_equal(g.view(np.uint32) if k == "cand_score" else g, e.view(np.uint32) if k == "cand_score" else e), (window, k)
    assert exp["n_scored"].max() > 0 and db["n"].max() > 150
    D.close()
    V.close()
    ctx.close()


# ---- ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255) on top of the FeatureVectors ----------------------------------
def _py_search_by_bow(oracle, f_bow, f_desc, k_bow, k_desc, cand_ok, query_ok):
    """literal merge-join of the two FeatureVectors with the reference's getBestMatch (sequential min / second rule)"""
    rows = []
    fi = ki = 0
    fn, fs, ff = f_bow["fv_nodes"], f_bow["fv_start"], f_bow["fv_feats"]
    kn, ks, kf = k_bow["fv_nodes"], k_bow["fv_start"], k_bow["fv_feats"]
    while fi < len(fn) and ki < len(kn):
        if fn[fi] > kn[ki]:
            ki += 1
        elif fn[fi] < kn[ki]:
            fi += 1
        else:
            for pk in kf[ks[ki] : ks[ki + 1]]:
                if query_ok is not None and not query_ok[pk]:
                    continue
                cand = [p for p in ff[fs[fi] : fs[fi + 1]] if cand_ok is None or cand_ok[p]]
                if not cand:
                    continue
                mn, sec, idx = 2**31 - 1, 2**31 - 1, 0
                for p in cand:
                    d = int(np.unpackbits(k_desc[pk] ^ f_desc[p]).sum())
                    if d < mn:
                        mn, idx = d, p
                    elif d < sec:
                        sec = d
                with np.errstate(invalid="ignore", divide="ignore"):
                    rows.append((pk, idx, mn, np.float32(mn) / np.float32(sec), len(cand)))
            fi += 1
            ki += 1
    return rows


def _frames_for_bow(oracle, seed):
    """two descriptor sets sharing most features (a frame and a keyframe of the same place) + a vocabulary built around them"""
    rng = np.random.default_rng(seed)
    voc = synth.synth_vocabulary(8, 3, seed)
    V = oracle.Vocabulary(**voc)
    leaves = np.nonzero(V.word_id >= 0)[0]
    base = V.desc[rng.choice(leaves, 700)].copy()

    def noisy(d, flips):
        d = d.copy()
        bits = rng.integers(0, 256, (len(d), flips))
        for b in range(flips):
            d[np.arange(len(d)), bits[:, b] // 8] ^= (1 << (bits[:, b] % 8)).astype(np.uint8)
        return d

    f_desc = noisy(base[rng.permutation(700)[:600]], 5)
    k_desc = noisy(base[rng.permutation(700)[:650]], 5)
    k_desc[:40] = f_desc[:40]  # exact copies: distance 0, NaN ratios when the runner-up is 0 too
    return voc, V, f_desc, k_desc, rng


def test_oracle_search_by_bow_equals_literal_merge_join(oracle):
    for seed in (1, 2):
        voc, V, f_desc, k_desc, rng = _frames_for_bow(oracle, seed)
        fb, kb = oracle.bow_transform(V, f_desc, 2), oracle.bow_transform(V, k_desc, 2)
        for cand_ok, query_ok in [(None, None), ((rng.random(len(f_desc)) < 0.6).astype(np.uint8), (rng.random(len(k_desc)) < 0.7).astype(np.uint8))]:
            r = oracle.search_by_bow(fb, f_desc, kb, k_desc, cand_ok, query_ok)
            exp = _py_search_by_bow(oracle, fb, f_desc, kb, k_desc, cand_ok, query_ok)
            assert len(exp) == len(r["kf_idx"]) and len(exp) > 200
            assert [e[0] for e in exp] == list(r["kf_idx"]) and [e[1] for e in exp] == list(r["best_idx"])
            assert [e[2] for e in exp] == list(r["best_dist"]) and [e[4] for e in exp] == list(r["n_cand"])
            assert np.array_equal(np.array([e[3] for e in exp], np.float32), r["ratio"], equal_nan=True)


@pytest.mark.gpu
def test_cuda_search_by_bow_equals_oracle(oracle):
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 8, 17)
    l2, r2 = synth.synth_stereo_pair(c["height"], c["width"] + 6, 8, 17)  # the "keyframe": the same scene shifted by 6 px
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=cam)
    kfr = ctx.stereo_frame(np.ascontiguousarray(l2[:, 6:]), np.ascontiguousarray(r2[:, 6:]))
    k_kps, k_desc = kfr.kps_left.copy(), kfr.desc_left.copy()
    voc = synth.synth_vocabulary(10, 3, 3)
    rng = np.random.default_rng(4)
    O0 = oracle.Vocabulary(**voc)
    leaves = np.nonzero(O0.word_id >= 0)[0]
    voc["desc"][leaves[:900] - 1] = k_desc[rng.choice(len(k_desc), 900, replace=False)]  # leaves that resemble the scene's descriptors
    O, V = oracle.Vocabulary(**voc), api.Vocabulary(ctx, **voc)
    k_bow = ctx.bow_transform(V, levelsup=2)
    fr = ctx.stereo_frame(left, right)
    with pytest.raises(ValueError):
        ctx.search_by_bow(k_bow, k_desc)  # the new frame's FeatureVector is not resident yet
    f_bow = ctx.bow_transform(V, levelsup=2)
    e_f, e_k = oracle.bow_transform(O, fr.desc_left, 2), oracle.bow_transform(O, k_desc, 2)
    kf_ok = (rng.random(len(k_desc)) < 0.7).astype(np.uint8)
    fr_ok = (rng.random(2000) < 0.6).astype(np.uint8)
    for qm, cm in [(None, None), (kf_ok, fr_ok)]:
        got = ctx.search_by_bow(k_bow, k_desc, qm, cm)
        exp = oracle.search_by_bow(e_f, fr.desc_left, e_k, k_desc, cm, qm)
        for key in exp:
            assert np.array_equal(got[key], exp[key], equal_nan=True), key
        assert len(got["kf_idx"]) > 300
    # the reference-shaped entry point: thresholds + verifyAngle, composed from the oracle
    frame = api.Frame(fr.kps_left, fr.desc_left, None, None, fr.u_right, fr.depth, fr.n_matches, {"ctx": ctx})
    m = api.ORBMatcher(0.6, True)
    got = m.searchByBow(frame, V, k_kps, k_desc, k_bow, kf_ok.astype(bool), ~fr_ok.astype(bool), levelsup=2)
    e = oracle.search_by_bow(e_f, fr.desc_left, e_k, k_desc, fr_ok, kf_ok)
    keep = ~((e["best_dist"] > 50) | (e["ratio"] > np.float32(0.6)))
    vq, vt, vd = oracle.verify_angle(e["best_idx"][keep], e["kf_idx"][keep], e["best_dist"][keep].astype(np.float32), fr.kps_left, k_kps)
    assert np.array_equal(got[:, 0], vq) and np.array_equal(got[:, 1], vt) and np.array_equal(got[:, 2], vd.astype(np.int32)) and len(got) > 50
    V.close()
    ctx.close()
