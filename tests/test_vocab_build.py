"""Vocabulary construction (orbx_vocab_build: DBoW2 / DBoW3 TemplatedVocabulary::create under the rules of include/orbx.h).

PARITY UNPINNED, as the transform: DBoW is not vendored.  CPU: the plain-C oracle_vocab_build (tests/vocab_build_oracle.c) equals a literal Python
restatement written in DBoW's recursion order (tests/vocab_build_restatement.py) on training sets built to reach every
rule, and its tree survives the ORB-SLAM2 text format.  GPU: the CUDA build equals the oracle bit for bit, on those sets
and on the device's own descriptors; the built vocabulary works with the transform and the keyframe export."""
import io
from collections import Counter

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

import vocab_build_restatement as R

FIELDS = ("parent", "is_leaf", "desc", "weight")


@pytest.fixture(scope="module")
def cases():
    return {name: R.case(name) for name in R.CASES}


def _oracle(c):
    return R.oracle_vocab_build(c["desc"], c["counts"], c["n_frames"], c["k"], c["L"], c["seed"])


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", R.CASES)
def test_oracle_equals_literal_restatement(cases, name):
    c = cases[name]
    st = Counter()
    py = R.py_vocab_build(c["desc"], c["counts"], c["n_frames"], c["k"], c["L"], c["seed"], st)
    orc = _oracle(c)
    for f in FIELDS:
        assert np.array_equal(py[f], orc[f]), f
    assert py["iters"] == orc["iters"] and py["n_capped"] == orc["n_capped"] == st["capped"] == 0
    # every training descriptor was trained into a leaf, and the two agree on which
    lf = orc["leaf_of"]
    for (f, i), node in py["leaf_of"].items():
        assert lf[f, i] == node and orc["is_leaf"][node - 1]
    assert (lf >= 0).sum() == len(py["leaf_of"]) == int(np.asarray(c["counts"])[: c["n_frames"]].sum())
    assert R.EXPECT.get(name, set()) <= {b for b, n in st.items() if n > 0}, dict(st)


def test_cases_reach_every_rule(cases):
    """every rule, over all cases and again over the cases with k > 10 alone (the k-wide paths of the kernels)"""
    seen, wide = Counter(), Counter()
    for c in cases.values():
        st = Counter()
        R.py_vocab_build(c["desc"], c["counts"], c["n_frames"], c["k"], c["L"], c["seed"], st)
        seen.update(st)
        if c["k"] > 10:
            wide.update(st)
    rules = {"node_n_le_k", "node_kmeans", "seeding_stopped_early", "assignment_tie", "converged", "empty_cluster_kept", "single_member_mean",
             "bit_majority_at_exactly_half", "early_leaf", "leaf_at_depth_L", "frame_without_keypoints", "padding_rows", "word_without_frames"}
    assert rules <= {b for b, n in seen.items() if n > 0}, dict(seen)
    assert rules <= {b for b, n in wide.items() if n > 0}, dict(wide)
    assert seen["capped"] == 0  # the ORBX_VOCAB_MAX_ITERS cap is not reached by these sets
    assert {c["k"] for c in cases.values()} >= {17, 32}


@pytest.mark.parametrize("name", ["random_k10_L3", "duplicates", "random_k3_L6"])
def test_text_format_keeps_the_tree(cases, name):
    c = cases[name]
    orc = _oracle(c)
    text = R.write_text(c["k"], c["L"], orc)
    back = R.parse_text(text)
    assert (back["k"], back["L"], back["scoring"], back["weighting"]) == (c["k"], c["L"], 0, 0)
    for f in ("parent", "is_leaf", "desc"):
        assert np.array_equal(back[f], orc[f]), f
    assert np.allclose(back["weight"], orc["weight"], rtol=1e-5, atol=0)  # "%g": 6 significant digits
    assert R.write_text(c["k"], c["L"], back) == text


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _small_ctx(**kw):
    return api.Context(320, 240, 500, 4, 1.2, camera=api.Camera(300.0, 300.0, 160.0, 120.0, 0.1), **kw)


def _assert_equal_trees(V, orc):
    got = V.arrays()
    for f in FIELDS:
        assert np.array_equal(got[f], orc[f]), f


@pytest.mark.gpu
def test_cuda_build_equals_oracle(cases):
    ctx = _small_ctx()
    for name, c in cases.items():
        stats = {}
        V = api.Vocabulary.build(ctx, c["desc"], c["counts"], n_frames=c["n_frames"], k=c["k"], L=c["L"], seed=c["seed"], stats=stats)
        orc = _oracle(c)
        _assert_equal_trees(V, orc)
        assert (stats["iters"], stats["n_capped"]) == (orc["iters"], orc["n_capped"]), name
        V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_text_round_trip(cases, tmp_path):
    ctx = _small_ctx()
    c = cases["random_k3_L6"]
    V = api.Vocabulary.build(ctx, c["desc"], c["counts"], n_frames=c["n_frames"], k=c["k"], L=c["L"], seed=c["seed"])
    p1, p2 = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
    V.save_text(p1)
    orc = _oracle(c)
    assert open(p1, "rb").read() == R.write_text(c["k"], c["L"], orc)  # the restated writer, byte for byte
    W = api.Vocabulary.load_text(ctx, p1)  # the repository's own loader
    W.save_text(p2)
    assert open(p2, "rb").read() == open(p1, "rb").read()
    got = W.arrays()
    for f in ("parent", "is_leaf", "desc"):
        assert np.array_equal(got[f], orc[f]), f
    assert W.info() == V.info()
    ctx.close()


def _kitti_images(F, seed0=40):
    c = synth.KITTI
    return synth.synth_stereo_pool(c["height"], c["width"], F, seed0=seed0, disparity=9)


def _kitti_ctx(max_batch):
    c = synth.KITTI
    return api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=max_batch)


@pytest.mark.gpu
def test_cuda_build_on_gathered_sequence_equals_oracle():
    F = 64
    lefts, rights = _kitti_images(F)
    ctx = _kitti_ctx(8)
    N = ctx.n_features
    res = ctx.sequence_stereo_ptr(F, lefts.ctypes.data, rights.ctypes.data, lefts.strides[1], lefts.strides[0])
    stats = {}
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=10, L=6, seed=11, stats=stats)
    gd = ctx.read_device(res.gathered_desc, (F, N, 32), np.uint8)
    gn = ctx.read_device(res.gathered_n, (F,), np.int32)
    assert gn.min() > 0
    orc = R.oracle_vocab_build(gd, gn, F, 10, 6, 11)
    _assert_equal_trees(V, orc)
    assert (stats["iters"], stats["n_capped"]) == (orc["iters"], orc["n_capped"])
    assert V.info()["n_words"] == int(orc["is_leaf"].sum()) > 10000
    ctx.close()


@pytest.mark.gpu
def test_cuda_training_descriptors_descend_to_their_leaves():
    """Every training descriptor on a path of converged nodes descends (orbx_bow_transform) to the leaf it was trained
    into, except (a) a descriptor with an identical twin earlier among the children of an n <= k node (the first equal
    child wins) and (b) one under a capped node.  The descent is read from the FeatureVector at every depth
    (levelsup = L - depth); a descriptor whose word has weight 0 (it occurs in every frame) is in no FeatureVector and is
    counted apart."""
    import torch

    F, k, L = 32, 10, 6
    c = synth.TUM
    H, W = c["height"], c["width"]
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], (0.0,) * 5, c["depth_scale"])
    ctx = api.Context(W, H, 1000, 8, 1.2, camera=cam, max_batch=F // 2)  # an RGB-D batch: frame f = image f
    d_gray = torch.from_numpy(np.stack([synth.synth_image(H, W, 300 + f) for f in range(F)])).cuda()
    d_depth = torch.from_numpy(np.stack([synth.synth_depth_u16(H, W, 300 + f, c["depth_scale"]) for f in range(F)])).cuda()
    torch.cuda.synchronize()
    res = ctx.rgbd_batch_device(F, d_gray.data_ptr(), W, W * H, d_depth.data_ptr(), 2 * W, 2 * W * H, api.DEPTH_U16)
    N = ctx.n_features
    V = api.Vocabulary.build(ctx, res.desc, res.n_kps, n_frames=F, stride=N, k=k, L=L, seed=3)
    desc = ctx.read_device(res.desc, (F, N, 32), np.uint8)
    n = ctx.read_device(res.n_kps, (F,), np.int32)
    orc = R.oracle_vocab_build(desc, n, F, k, L, 3)
    _assert_equal_trees(V, orc)
    par = np.concatenate([[-1], orc["parent"]])
    nd = np.concatenate([np.zeros((1, 32), np.uint8), orc["desc"]])
    capped_path = orc["node_capped"].astype(bool)
    for node in range(1, len(par)):  # parents precede their children
        capped_path[node] |= capped_path[par[node]]
    kinds = Counter()
    for f in range(F):
        deepest = np.zeros(N, np.int64)
        listed = np.zeros(N, bool)
        for depth in range(1, L + 1):
            b = ctx.bow_transform(V, frame=f, levelsup=L - depth)
            for j, node in enumerate(b["fv_nodes"]):
                feats = b["fv_feats"][b["fv_start"][j] : b["fv_start"][j + 1]]
                listed[feats] = True
                if node > 0:
                    deepest[feats] = node
        for i in range(n[f]):
            trained = orc["leaf_of"][f, i]
            if not listed[i]:
                assert orc["weight"][trained - 1] == 0.0 or capped_path[trained]
                kinds["weight_0"] += 1
            elif deepest[i] == trained:
                kinds["same_leaf"] += 1
            elif capped_path[trained]:
                kinds["under_capped_node"] += 1
            else:
                got = deepest[i]
                assert par[got] == par[trained] and got < trained and np.array_equal(nd[got], nd[trained]), (f, i, got, trained)
                kinds["earlier_identical_twin"] += 1
    assert kinds["same_leaf"] > 0.99 * n.sum(), dict(kinds)
    print(dict(kinds))
    ctx.close()


@pytest.mark.gpu
def test_cuda_two_local_ranks_build_identical_vocabularies(tmp_path):
    F = 12
    lefts, rights = _kitti_images(F, seed0=55)
    ranks = [_kitti_ctx(4) for _ in range(2)]
    comms = api.Communicator.local(ranks, F)
    results = []
    for r in range(2):
        blk = api.frame_range(F, r, 2)
        lo = lefts[blk.start : blk.stop]
        results.append(ranks[r].sequence_stereo_ptr(F, lo.ctypes.data, rights[blk.start : blk.stop].ctypes.data, lo.strides[1], lo.strides[0], comms[r]))
    texts = []
    for r in range(2):
        V = api.Vocabulary.build(ranks[r], results[r].gathered_desc, results[r].gathered_n, n_frames=F, stride=ranks[r].n_features, k=10, L=4, seed=2)
        p = str(tmp_path / f"rank{r}.txt")
        V.save_text(p)
        texts.append(open(p, "rb").read())
        V.close()
    assert texts[0] == texts[1] and len(texts[0]) > 1000
    for o in comms + ranks:
        o.close()


@pytest.mark.gpu
def test_cuda_built_vocabulary_exports_keyframes(tmp_path):
    import keyframe_proto as KP

    F = 6
    lefts, rights = _kitti_images(F, seed0=20)
    ctx = _kitti_ctx(4)
    _, gd, gn = ctx.sequence_stereo(lefts, rights)
    V = api.Vocabulary.build(ctx, gd, gn, k=10, L=6, seed=9)
    _, _, _, kf, sizes = ctx.sequence_stereo_keyframes(lefts, rights, vocab=V, id0=5)
    buf = io.BytesIO()
    api.write_keyframe_list(buf, ctx, kf, sizes, next_id=5 + F)
    lst = KP.messages()["KeyFrameList"]()
    lst.ParseFromString(buf.getvalue())
    assert len(lst.keyframes) == F and all(len(m.bow_vector.words) > 0 for m in lst.keyframes)
    # the transform on the resident vocabulary and on the one read back from its text: the same words, feature lists and
    # node ids; the weights differ only by the 6 significant digits the text keeps
    p = str(tmp_path / "voc.txt")
    V.save_text(p)
    W = api.Vocabulary.load_text(ctx, p)
    ctx.stereo_frame(lefts[0], rights[0])
    a, b = ctx.bow_transform(V), ctx.bow_transform(W)
    for f in ("bow_ids", "fv_nodes", "fv_start", "fv_feats"):
        assert np.array_equal(a[f], b[f]), f
    assert np.allclose(a["bow_vals"], b["bow_vals"], rtol=2e-5, atol=0)
    ctx.close()


@pytest.mark.gpu
def test_cuda_build_rejects_bad_arguments(cases):
    ctx = _small_ctx()
    c = cases["random_k3_L2"]
    args = (c["desc"], c["counts"])
    for k, L in [(1, 3), (0, 3), (api.VOCAB_MAX_K + 1, 2), (10, 0), (10, 10), (2, 40)]:
        with pytest.raises(ValueError, match="invalid argument"):
            api.Vocabulary.build(ctx, *args, n_frames=c["n_frames"], k=k, L=L)
    bad = np.array(c["counts"], np.int32)
    bad[0] = c["desc"].shape[1] + 1
    with pytest.raises(ValueError, match="invalid argument"):
        api.Vocabulary.build(ctx, c["desc"], bad, n_frames=c["n_frames"], k=3, L=2)
    import torch

    d_desc, d_bad = torch.from_numpy(np.ascontiguousarray(c["desc"])).cuda(), torch.from_numpy(bad).cuda()
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match=r"invalid argument \(vocabulary training set: a count lies outside 0\.\.stride"):  # the same counts in device memory
        api.Vocabulary.build(ctx, d_desc.data_ptr(), d_bad.data_ptr(), n_frames=c["n_frames"], stride=c["desc"].shape[1], k=3, L=2)
    with pytest.raises(ValueError, match="invalid argument"):
        api.Vocabulary.build(ctx, c["desc"], np.zeros_like(bad), n_frames=c["n_frames"], k=3, L=2)  # no descriptor
    # a vocabulary built on another context is refused, as a created / loaded one is
    other = _small_ctx()
    V = api.Vocabulary.build(other, *args, n_frames=c["n_frames"], k=3, L=2)
    lefts, rights = synth.synth_stereo_pool(240, 320, 2, seed0=0, disparity=9)
    with pytest.raises(ValueError, match="another context"):
        ctx.sequence_stereo_keyframes(lefts, rights, vocab=V)
    V.close()
    other.close()
    ctx.close()
