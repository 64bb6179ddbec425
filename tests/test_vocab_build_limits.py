"""Vocabulary construction (orbx_vocab_build) and the bag-of-words sort at their size limits.

The training sets of tests/vocab_build_restatement.py's LIMIT_CASES reach what the sets written for the rules do not:
  - k = 31 at three levels (the k-wide centre arrays, counters and ballots; k = 17 and 32 are in CASES, where the literal
    restatement checks them too);
  - roots of exactly 4096, 4097 and 8193 descriptors: a full last k-means tile, a last tile of one, three tiles;
  - frame rows of 4096, 4097, 8193 and 16384 descriptors, one of them full: the IDF step's one-CTA sort of P = 4096,
    8192 and 16384 keys (above 48 KB of shared memory from 4097 on);
  - 70,500 frames and 1,059,382 descriptors: a root of 259 tiles, so that each thread of vocab_kpp_pick_kernel sums two
    tiles and walks them to the cut, and a second 65535-frame chunk of the IDF step.
CPU: a census over oracle_vocab_build's outputs shows each set reaches its limit.  GPU: the CUDA build equals the oracle bit
for bit on every set, from host rows and, for the largest two, from device pointers; and every bag-of-words entry point
refuses a frame row above ORBX_BOW_MAX_STRIDE before it enqueues anything, leaving the context usable."""
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

import vocab_build_restatement as R
from test_vocab_build import _assert_equal_trees, _small_ctx

TILE = 4096          # kTile of csrc/orbx_vocab.cu: descriptors per k-means tile
PICK_THREADS = 256   # threads of vocab_kpp_pick_kernel, each summing ceil(tiles / 256) tiles
IDF_CHUNK = 65535    # frames per launch of the IDF step (grid.y)


@pytest.fixture(scope="module")
def limits():
    """name -> (case, oracle_vocab_build of it)"""
    out = {}
    for name in R.LIMIT_CASES:
        c = R.case(name)
        out[name] = (c, R.oracle_vocab_build(c["desc"], c["counts"], c["n_frames"], c["k"], c["L"], c["seed"]))
    return out


def _n(c):
    return int(np.asarray(c["counts"])[: c["n_frames"]].sum())


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_tile_cases_end_on_the_tile_edges(limits):
    for name, (n, last) in {"tile_4096": (4096, TILE), "tile_4097": (4097, 1), "tile_8193": (8193, 1)}.items():
        c, orc = limits[name]
        assert _n(c) == n and (n - 1) % TILE + 1 == last, name
        assert orc["iters"][0] > 1 and orc["root_picks"].min() >= 0, name  # the root ran k-means with k picks


def test_many_frames_root_picks_walk_inside_a_threads_tiles(limits):
    c, orc = limits["many_frames"]
    n = _n(c)
    tiles = -(-n // TILE)
    per = -(-tiles // PICK_THREADS)
    assert n > PICK_THREADS * TILE and per == 2, (n, tiles)
    picks = orc["root_picks"][1:]  # pick 0 is r_0 % n, without a walk
    assert (picks >= 0).all()
    # the root's segment starts at tile 0: a pick in a tile t with t % per != 0 is found past the first tile of a thread's range
    assert ((picks // TILE) % per != 0).any(), picks


def test_many_frames_has_words_of_the_second_idf_chunk(limits):
    c, orc = limits["many_frames"]
    F = c["n_frames"]
    assert F >= 70000 and F > IDF_CHUNK
    leaf_of = orc["leaf_of"]
    frame = np.broadcast_to(np.arange(F)[:, None], leaf_of.shape)
    trained = leaf_of >= 0
    first = np.full(len(orc["parent"]) + 1, F, np.int64)
    np.minimum.at(first, leaf_of[trained], frame[trained])
    node = np.arange(1, len(orc["parent"]) + 1)
    late = node[(first[node] >= IDF_CHUNK) & (first[node] < F) & (orc["weight"] > 0)]
    assert len(late) > 0  # words whose every training frame is in the second chunk, with N_i > 0
    # and words of the first chunk, for contrast
    assert ((first[node] < IDF_CHUNK) & (orc["weight"] > 0)).any()


@pytest.mark.parametrize("name", R.WIDE_STRIDE_CASES)
def test_wide_stride_sets_have_a_full_and_an_empty_row(limits, name):
    c, orc = limits[name]
    stride = c["desc"].shape[1]
    counts = np.asarray(c["counts"])[: c["n_frames"]]
    assert (counts == stride).any() and (counts == 0).any()
    assert stride <= api.BOW_MAX_STRIDE and (orc["weight"] > 0).any()


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _build(ctx, c, **kw):
    stats = {}
    V = api.Vocabulary.build(ctx, c["desc"], c["counts"], n_frames=c["n_frames"], k=c["k"], L=c["L"], seed=c["seed"], stats=stats, **kw)
    return V, stats


def _equals_oracle(V, stats, orc, what):
    _assert_equal_trees(V, orc)
    assert (stats["iters"], stats["n_capped"]) == (orc["iters"], orc["n_capped"]), what


@pytest.mark.gpu
def test_cuda_build_equals_oracle_at_the_limits(limits):
    ctx = _small_ctx()
    for name, (c, orc) in limits.items():
        V, stats = _build(ctx, c)
        _equals_oracle(V, stats, orc, name)
        V.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["many_frames", "wide_stride_16384"])
def test_cuda_build_from_device_pointers_at_the_limits(limits, name):
    import torch

    c, orc = limits[name]
    ctx = _small_ctx()
    d_desc, d_n = torch.from_numpy(c["desc"]).cuda(), torch.from_numpy(np.asarray(c["counts"], np.int32)).cuda()
    torch.cuda.synchronize()
    stats = {}
    V = api.Vocabulary.build(ctx, d_desc.data_ptr(), d_n.data_ptr(), n_frames=c["n_frames"], stride=c["desc"].shape[1], k=c["k"], L=c["L"],
                             seed=c["seed"], stats=stats)
    _equals_oracle(V, stats, orc, name)
    V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_text_round_trip_k32(tmp_path):
    c = R.case("k32_L2")
    orc = R.oracle_vocab_build(c["desc"], c["counts"], c["n_frames"], c["k"], c["L"], c["seed"])
    ctx = _small_ctx()
    V, _ = _build(ctx, c)
    p1, p2 = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
    V.save_text(p1)
    assert open(p1, "rb").read() == R.write_text(32, 2, orc)
    W = api.Vocabulary.load_text(ctx, p1)
    W.save_text(p2)
    assert open(p2, "rb").read() == open(p1, "rb").read()
    got = W.arrays()
    for f in ("parent", "is_leaf", "desc"):
        assert np.array_equal(got[f], orc[f]), f
    assert W.info() == V.info() and V.info()["k"] == 32
    ctx.close()


def _still_usable(ctx, limits, pair, before):
    """after a refusal: the same stereo frame as before it, and a stride-16384 build equal to the oracle, on the same context"""
    r = ctx.stereo_frame(*pair)
    assert np.array_equal(r.desc_left, before.desc_left) and r.n_matches == before.n_matches
    c, orc = limits["wide_stride_16384"]
    V, stats = _build(ctx, c)
    _equals_oracle(V, stats, orc, "after a refusal")
    V.close()


@pytest.mark.gpu
def test_cuda_bow_entry_points_refuse_rows_the_sort_cannot_hold(limits):
    pair = synth.synth_stereo_pair(240, 320, 0, 9)
    voc = synth.synth_vocabulary(10, 3, 1)
    ctx = _small_ctx()
    V = api.Vocabulary(ctx, **voc)
    before = ctx.stereo_frame(*pair)
    assert before.n_matches > 0
    for stride in (api.BOW_MAX_STRIDE + 1, 65535):
        desc, counts = np.zeros((2, stride, 32), np.uint8), np.array([1, stride], np.int32)
        with pytest.raises(ValueError, match="invalid argument.*ORBX_BOW_MAX_STRIDE"):
            api.Vocabulary.build(ctx, desc, counts, k=10, L=2)
        _still_usable(ctx, limits, pair, before)
        with pytest.raises(ValueError, match="invalid argument.*ORBX_BOW_MAX_STRIDE"):
            api.BowDatabase.build(ctx, V, desc, counts)
        _still_usable(ctx, limits, pair, before)
    V.close()
    ctx.close()
    # a context whose frames hold more features than the sort: the transform and the loop verifier refuse it.  A noise
    # image of 1600 x 1200 over 8 levels fills all 16385 features (the shape of test_bow's 16384-feature context).
    noise = np.random.default_rng(1).integers(0, 256, (1200, 1600), dtype=np.uint8)
    big_pair = (noise, np.ascontiguousarray(np.roll(noise, -4, axis=1)))
    big = api.Context(1600, 1200, api.BOW_MAX_STRIDE + 1, 8, 1.2, camera=api.Camera(1000.0, 1000.0, 800.0, 600.0, 0.1))
    W = api.Vocabulary(big, **voc)
    before = big.stereo_frame(*big_pair)
    assert len(before.desc_left) > api.BOW_MAX_STRIDE
    with pytest.raises(ValueError, match="ORBX_BOW_MAX_STRIDE"):
        big.bow_transform(W)
    _still_usable(big, limits, big_pair, before)
    with pytest.raises(ValueError, match="ORBX_BOW_MAX_STRIDE"):
        api.LoopVerifier.build(big, W, np.zeros(1, big.record_dtype()), 1)
    _still_usable(big, limits, big_pair, before)
    W.close()
    big.close()
