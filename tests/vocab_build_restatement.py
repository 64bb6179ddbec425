"""A literal restatement of the vocabulary construction (DBoW2 / DBoW3 TemplatedVocabulary::create under the rules of
include/orbx.h, orbx_vocab_build), the ctypes binding of the plain-C checker oracle_vocab_build (tests/vocab_build_oracle.c), the ORB-SLAM2 text writer, and the training
sets the tests run on.

The restatement is written the way DBoW writes it: a recursive HKmeansStep over Python lists, nodes appended to a list in
creation order, children consecutive, splits depth first.  It counts the branches it takes (`stats`), so every case can
assert which rules it reaches.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile
from collections import Counter

import numpy as np

MAX_ITERS = 100  # ORBX_VOCAB_MAX_ITERS
GOLDEN = 0x9E3779B97F4A7C15
M64 = (1 << 64) - 1
HERE = os.path.dirname(os.path.abspath(__file__))


def splitmix64(x: int) -> int:
    z = (x + GOLDEN) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def _dist(a: bytes, b: bytes) -> int:
    return bin(int.from_bytes(a, "little") ^ int.from_bytes(b, "little")).count("1")


def _bit(x: bytes, b: int) -> int:
    return (x[b >> 3] >> (b & 7)) & 1


def py_vocab_build(desc, counts, n_frames: int, k: int, L: int, seed: int, stats: Counter | None = None):
    """-> dict(parent, is_leaf, desc, weight) in record order (record i = node i + 1), iters (per level), n_capped, leaf_of
    (frame, i) -> node id"""
    st = stats if stats is not None else Counter()
    feats, where = [], []
    for f in range(n_frames):
        if counts[f] == 0:
            st["frame_without_keypoints"] += 1
        for i in range(int(counts[f])):
            feats.append(bytes(desc[f][i]))
            where.append((f, i))
    if len(desc) > n_frames:
        st["padding_rows"] += 1
    nodes = [dict(parent=-1, children=[], desc=bytes(32))]  # node 0 = root
    iters = [0] * L
    leaf_of = {}
    capped = [0]

    def hkmeans_step(parent_id, key, members, level):
        n = len(members)
        if n <= k:
            st["node_n_le_k"] += 1
            clusters = [feats[m] for m in members]
            groups = [[m] for m in members]
        else:
            st["node_kmeans"] += 1
            # initiateClustersKMpp, integer form
            clusters = [feats[members[splitmix64(key) % n]]]
            min_dist = [_dist(feats[m], clusters[0]) for m in members]
            while len(clusters) < k:
                S = sum(min_dist)
                if S == 0:
                    st["seeding_stopped_early"] += 1
                    break
                cut = 1 + splitmix64(key ^ ((len(clusters) * GOLDEN) & M64)) % S
                run = 0
                for i, d in enumerate(min_dist):
                    run += d
                    if run >= cut:
                        break
                clusters.append(feats[members[i]])
                min_dist = [min(md, _dist(feats[m], clusters[-1])) for md, m in zip(min_dist, members)]
            last, p = None, 0
            while True:
                p += 1
                groups = [[] for _ in clusters]
                current = []
                for m in members:
                    ds = [_dist(feats[m], c) for c in clusters]
                    best = min(ds)
                    if ds.count(best) > 1:
                        st["assignment_tie"] += 1
                    c = ds.index(best)  # the first among equals
                    groups[c].append(m)
                    current.append(c)
                if last is not None and current == last:
                    st["converged"] += 1
                    break
                if p == MAX_ITERS:
                    st["capped"] += 1
                    capped[0] += 1
                    break
                last = current
                # FORB::meanValue
                new = []
                for c, g in zip(clusters, groups):
                    if not g:
                        st["empty_cluster_kept"] += 1
                        new.append(c)
                        continue
                    if len(g) == 1:
                        st["single_member_mean"] += 1
                    half = (len(g) + 1) // 2
                    out = bytearray(32)
                    for b in range(256):
                        s = sum(_bit(feats[m], b) for m in g)
                        if s >= half:
                            out[b >> 3] |= 1 << (b & 7)
                            if s == half and len(g) > 1:
                                st["bit_majority_at_exactly_half"] += 1
                    new.append(bytes(out))
                clusters = new
            iters[level - 1] = max(iters[level - 1], p)
        first = len(nodes)
        for c in clusters:
            nodes.append(dict(parent=parent_id, children=[], desc=c))
            nodes[parent_id]["children"].append(len(nodes) - 1)
        for ci, g in enumerate(groups):
            child = first + ci
            if level < L and len(g) > 1:
                hkmeans_step(child, splitmix64((key + ci + 1) & M64), g, level + 1)
            else:
                st["early_leaf" if level < L else "leaf_at_depth_L"] += 1
                for m in g:
                    leaf_of[where[m]] = child

    hkmeans_step(0, splitmix64(seed), list(range(len(feats))), 1)
    # createWords + setNodeWeights (TF_IDF) with the transform's descent
    word = {}
    for i, nd in enumerate(nodes):
        if i > 0 and not nd["children"]:
            word[i] = len(word)
    ni = Counter()
    for f in range(n_frames):
        seen = set()
        for i in range(int(counts[f])):
            x, node = bytes(desc[f][i]), 0
            while nodes[node]["children"]:
                ch = nodes[node]["children"]
                ds = [_dist(x, nodes[c]["desc"]) for c in ch]
                node = ch[ds.index(min(ds))]
            seen.add(word[node])
        ni.update(seen)
    rec = dict(parent=[], is_leaf=[], desc=[], weight=[])
    for i in range(1, len(nodes)):
        nd = nodes[i]
        rec["parent"].append(nd["parent"])
        rec["is_leaf"].append(int(not nd["children"]))
        rec["desc"].append(np.frombuffer(nd["desc"], np.uint8))
        w = 0.0
        if i in word and ni[word[i]] > 0:
            w = math.log(n_frames / ni[word[i]])
        elif i in word:
            st["word_without_frames"] += 1
        rec["weight"].append(w)
    return dict(parent=np.array(rec["parent"], np.int32), is_leaf=np.array(rec["is_leaf"], np.uint8), desc=np.array(rec["desc"], np.uint8).reshape(-1, 32),
                weight=np.array(rec["weight"], np.float64), iters=iters, n_capped=capped[0], leaf_of=leaf_of)


_lib = None


def _oracle_lib():
    """tests/vocab_build_oracle.c, compiled once per process with the host C compiler (the flags of oracle/Makefile) into a
    temporary directory that is removed again once the library is loaded"""
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="vocab_build_oracle_")
        try:
            so = os.path.join(tmp, "libvocab_build_oracle.so")
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", "-o", so, os.path.join(HERE, "vocab_build_oracle.c"), "-lm"],
                           check=True, capture_output=True)
            lib = C.CDLL(so)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        lib.oracle_vocab_build.restype = C.c_int
        lib.oracle_vocab_build.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int] + [C.c_void_p] * 9
        _lib = lib
    return _lib


def oracle_vocab_build(desc, counts, n_frames: int, k: int, L: int, seed: int):
    """oracle_vocab_build (tests/vocab_build_oracle.c) -> the same dict as py_vocab_build, leaf_of as an (n_frames, stride)
    array (-1 = padding), plus node_capped per node id and root_picks (the root's k-means++ picks as positions among the
    training descriptors in frame order, -1 past the last)"""
    f = _oracle_lib().oracle_vocab_build
    d = np.ascontiguousarray(desc, np.uint8)
    cnt = np.ascontiguousarray(counts, np.int32)
    stride = d.shape[1]
    cap = max(1, int(cnt[:n_frames].sum())) * L + 1
    par, leaf, nd, w = np.zeros(cap, np.int32), np.zeros(cap, np.uint8), np.zeros((cap, 32), np.uint8), np.zeros(cap, np.float64)
    iters, ncap = np.zeros(L, np.int32), np.zeros(1, np.int32)
    leaf_of, node_capped, picks = np.zeros((n_frames, stride), np.int32), np.zeros(cap + 1, np.uint8), np.zeros(k, np.int32)
    n = f(d.ctypes.data, cnt.ctypes.data, n_frames, stride, k, L, seed & M64, cap, par.ctypes.data, leaf.ctypes.data, nd.ctypes.data, w.ctypes.data,
          iters.ctypes.data, ncap.ctypes.data, leaf_of.ctypes.data, node_capped.ctypes.data, picks.ctypes.data)
    assert n > 0, "oracle_vocab_build refused the input"
    return dict(parent=par[:n].copy(), is_leaf=leaf[:n].copy(), desc=nd[:n].copy(), weight=w[:n].copy(), iters=iters.tolist(), n_capped=int(ncap[0]),
                leaf_of=leaf_of, node_capped=node_capped[: n + 1].copy(), root_picks=picks)


def write_text(k: int, L: int, rec: dict) -> bytes:
    """ORB-SLAM2 TemplatedVocabulary::saveToTextFile: "k L  scoring weighting", then "parent isLeaf " + FORB::toString (a
    blank after every byte) + " " + weight as the stream prints a double ("%g")"""
    lines = [f"{k} {L}  0 0"]
    for p, lf, d, w in zip(rec["parent"], rec["is_leaf"], rec["desc"], rec["weight"]):
        lines.append(f"{int(p)} {int(lf)} " + "".join(f"{int(x)} " for x in d) + " " + ("%g" % float(w)))
    return ("\n".join(lines) + "\n").encode()


def parse_text(text: bytes) -> dict:
    """what a whitespace-separated reader (operator>>) takes from write_text's output"""
    lines = text.decode().split("\n")
    k, L, scoring, weighting = (int(x) for x in lines[0].split())
    rows = [ln.split() for ln in lines[1:] if ln.strip()]
    return dict(k=k, L=L, scoring=scoring, weighting=weighting, parent=np.array([int(r[0]) for r in rows], np.int32),
                is_leaf=np.array([int(r[1]) for r in rows], np.uint8), desc=np.array([[int(x) for x in r[2:34]] for r in rows], np.uint8).reshape(-1, 32),
                weight=np.array([float(r[34]) for r in rows], np.float64))


# ---- training sets ------------------------------------------------------------------------------------------------
def _frames(feats: np.ndarray, counts, stride: int, pad_rows: int = 0, seed: int = 0):
    """rows [F + pad_rows][stride][32] holding feats frame by frame (random bytes beyond each count and in the padding)"""
    rng = np.random.default_rng(seed + 1000)
    counts = np.asarray(counts, np.int32)
    F = len(counts)
    desc = rng.integers(0, 256, (F + pad_rows, stride, 32), dtype=np.uint8)
    assert counts.sum() == len(feats)
    desc[:F][np.arange(stride) < counts[:, None]] = feats
    full = np.concatenate([counts, rng.integers(1, stride + 1, pad_rows).astype(np.int32)])
    return desc, full


def _clustered(n: int, n_centres: int, flip: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    centres = rng.integers(0, 256, (n_centres, 32), dtype=np.uint8)
    d = centres[rng.integers(0, n_centres, n)].copy()
    bits = np.unpackbits(d, axis=1, bitorder="little")
    for i in range(n):
        bits[i, rng.choice(256, rng.integers(0, flip + 1), replace=False)] ^= 1
    return np.packbits(bits, axis=1, bitorder="little")


def _flip(d: np.ndarray, flip: int, rng) -> np.ndarray:
    """every row with up to `flip` bits flipped at random positions (a position drawn twice flips back), vectorised"""
    d = d.copy()
    m = rng.integers(0, flip + 1, len(d))
    pos = rng.integers(0, 256, (len(d), max(flip, 1)))
    rows = np.arange(len(d))
    for j in range(flip):
        on = m > j
        d[rows[on], pos[on, j] >> 3] ^= (1 << (pos[on, j] & 7)).astype(np.uint8)
    return d


def _two_level(n: int, n_top: int, n_sub: int, seed: int, spread: int = 40, flip: int = 8, decay: float = 0.85):
    """n descriptors around n_top groups of n_sub sub-centres each: sub-centres within `spread` bits of their group's centre,
    descriptors within `flip` bits of a sub-centre.  Group sizes fall geometrically by `decay`, so that some groups hold
    fewer than k descriptors and others more than k clusters.  -> (descriptors, group of each)"""
    rng = np.random.default_rng(seed)
    top = rng.integers(0, 256, (n_top, 32), dtype=np.uint8)
    sub = _flip(np.repeat(top, n_sub, axis=0), spread, rng)
    w = decay ** np.arange(n_top)
    g = rng.choice(n_top, n, p=w / w.sum())
    return _flip(sub[g * n_sub + rng.integers(0, n_sub, n)], flip, rng), g


def _spread(n: int, n_frames: int, seed: int) -> np.ndarray:
    """n descriptors over n_frames frames of uneven counts, frame 1 empty"""
    rng = np.random.default_rng(seed)
    cut = np.sort(rng.choice(np.arange(1, n), n_frames - 2, replace=False))
    counts = np.diff(np.concatenate([[0], cut, [n]]))
    return np.insert(counts, 1, 0).astype(np.int32)


def case(name: str):
    """-> dict(desc, counts, n_frames, k, L, seed): training rows plus the parameters of one named case"""
    if name.startswith("random_k"):  # random_k{k}_L{L}
        k, L = (int(x) for x in name[len("random_k") :].split("_L"))
        counts = [31, 0, 17, 40, 9, 28]
        feats = _clustered(sum(counts), 12, 40, 7 * k + L)
        desc, full = _frames(feats, counts, 40, pad_rows=2, seed=k + L)
        return dict(desc=desc, counts=full, n_frames=len(counts), k=k, L=L, seed=k * 100 + L)
    if name == "duplicates":  # four distinct descriptors repeated: k-means++ runs out of distinct points
        rng = np.random.default_rng(3)
        base = rng.integers(0, 256, (4, 32), dtype=np.uint8)
        counts = [20, 0, 25]
        feats = base[rng.integers(0, 4, sum(counts))]
        desc, full = _frames(feats, counts, 25, pad_rows=1, seed=3)
        return dict(desc=desc, counts=full, n_frames=3, k=10, L=3, seed=5)
    if name == "all_identical":
        rng = np.random.default_rng(4)
        counts = [12, 13]
        feats = np.repeat(rng.integers(0, 256, (1, 32), dtype=np.uint8), sum(counts), axis=0)
        desc, full = _frames(feats, counts, 16, seed=4)
        return dict(desc=desc, counts=full, n_frames=2, k=3, L=4, seed=6)
    if name == "n_le_k_root":  # fewer descriptors than k, two of them equal
        rng = np.random.default_rng(5)
        feats = rng.integers(0, 256, (7, 32), dtype=np.uint8)
        feats[5] = feats[2]
        desc, full = _frames(feats, [3, 0, 4], 6, pad_rows=3, seed=5)
        return dict(desc=desc, counts=full, n_frames=3, k=10, L=2, seed=7)
    if name == "even_members":  # pairs of near twins: even clusters whose bit counts land on exactly m/2
        rng = np.random.default_rng(6)
        base = rng.integers(0, 256, (6, 32), dtype=np.uint8)
        feats = np.repeat(base, 4, axis=0)
        bits = np.unpackbits(feats, axis=1, bitorder="little")
        for i in range(len(feats)):
            bits[i, rng.choice(256, 30, replace=False)] ^= 1
        feats = np.packbits(bits, axis=1, bitorder="little")
        desc, full = _frames(feats, [8, 8, 8], 8, seed=6)
        return dict(desc=desc, counts=full, n_frames=3, k=3, L=3, seed=8)
    if name == "k32_root_eq_k":  # exactly k = 32 descriptors, two equal: the root's children are its descriptors, a full warp
        rng = np.random.default_rng(40)
        feats = rng.integers(0, 256, (32, 32), dtype=np.uint8)
        feats[29] = feats[6]
        desc, full = _frames(feats, [10, 0, 22], 24, pad_rows=1, seed=40)
        return dict(desc=desc, counts=full, n_frames=3, k=32, L=2, seed=41)
    if name == "k32_root_k_plus_1":  # k-means++ picks 32 centres from 33 descriptors
        rng = np.random.default_rng(42)
        feats = _flip(np.repeat(rng.integers(0, 256, (3, 32), dtype=np.uint8), 11, axis=0), 60, rng)
        desc, full = _frames(feats, [16, 17], 20, pad_rows=2, seed=42)
        return dict(desc=desc, counts=full, n_frames=2, k=32, L=2, seed=43)
    if name in ("k32_L2", "k31_L3", "k17_L2"):
        k, L = (int(x) for x in name[1:].split("_L"))
        n, n_top, n_sub = {32: (2600, 20, 48), 31: (4000, 45, 40), 17: (2200, 12, 30)}[k]
        feats, _ = _two_level(n, n_top, n_sub, seed=k)
        # a group of 60 copies of 6 distinct descriptors: a node with more than k descriptors but fewer than k distinct ones
        rng = np.random.default_rng(k + 1)
        feats[rng.choice(n, 60, replace=False)] = rng.integers(0, 256, (6, 32), dtype=np.uint8)[np.arange(60) % 6]
        counts = _spread(n, 9, seed=k)
        desc, full = _frames(feats, counts, int(counts.max()) + 3, pad_rows=2, seed=k)
        return dict(desc=desc, counts=full, n_frames=len(counts), k=k, L=L, seed=k * 7)
    if name.startswith("tile_"):  # a root of exactly n descriptors: k-means tiles of kTile = 4096, the last one full / of one / three tiles
        n = int(name[5:])
        feats, _ = _two_level(n, 14, 12, seed=n)
        counts = _spread(n, 11, seed=n)
        desc, full = _frames(feats, counts, int(counts.max()), pad_rows=1, seed=n)
        return dict(desc=desc, counts=full, n_frames=len(counts), k=10, L=2, seed=n)
    if name.startswith("wide_stride_"):  # frame rows past 4096 descriptors: one full row, one empty, in the IDF step's sort
        stride = int(name[len("wide_stride_") :])
        counts = np.array([stride, 0, stride // 3, 1, stride - 5], np.int32)
        feats, _ = _two_level(int(counts.sum()), 16, 10, seed=stride)
        desc, full = _frames(feats, counts, stride, pad_rows=1, seed=stride)
        return dict(desc=desc, counts=full, n_frames=len(counts), k=10, L=3, seed=stride)
    if name == "many_frames":
        # 70,500 frames of up to 16 descriptors, 1,065,000 in all: the root spans 261 k-means tiles (more than one per thread
        # of the pick kernel's 256) and the IDF step runs a second chunk of frames (>= 65535).  Frames from 65535 on draw
        # half their descriptors from 4 groups no earlier frame uses, so some words are reached from the second chunk only.
        F, stride = 70500, 16
        counts = np.full(F, stride, np.int32)
        counts[::3] = 14
        counts[::50] = 0
        counts[65535] = stride
        n = int(counts.sum())
        feats, _ = _two_level(n, 12, 8, seed=70, decay=0.97)
        late_lo = int(counts[:65535].sum())
        rng = np.random.default_rng(71)
        new, _ = _two_level(n - late_lo, 4, 3, seed=72, decay=1.0)
        take = rng.random(n - late_lo) < 0.5
        feats[late_lo:][take] = new[take]
        desc, full = _frames(feats, counts, stride, pad_rows=1, seed=73)
        return dict(desc=desc, counts=full, n_frames=F, k=10, L=2, seed=74)
    raise KeyError(name)


RANDOM_CASES = [f"random_k{k}_L{L}" for k in (2, 3, 10) for L in (1, 2, 3, 6)]
# branching factors above 10, small enough for the literal restatement
WIDE_K_CASES = ["k32_root_eq_k", "k32_root_k_plus_1", "k32_L2", "k17_L2"]
CASES = RANDOM_CASES + ["duplicates", "all_identical", "n_le_k_root", "even_members"] + WIDE_K_CASES
# the size limits of the device build, checked against the C oracle only (the restatement would take minutes)
TILE_CASES = ["tile_4096", "tile_4097", "tile_8193"]
WIDE_STRIDE_CASES = [f"wide_stride_{s}" for s in (4096, 4097, 8193, 16384)]
LIMIT_CASES = ["k31_L3"] + TILE_CASES + WIDE_STRIDE_CASES + ["many_frames"]

# the branches each case must reach (beyond the ones every case reaches)
EXPECT = {
    "duplicates": {"seeding_stopped_early", "padding_rows", "frame_without_keypoints", "node_kmeans"},
    "all_identical": {"seeding_stopped_early", "leaf_at_depth_L", "converged"},
    "n_le_k_root": {"node_n_le_k", "early_leaf", "padding_rows", "frame_without_keypoints"},
    "even_members": {"bit_majority_at_exactly_half", "node_kmeans"},
    "random_k10_L2": {"empty_cluster_kept", "node_n_le_k", "early_leaf", "assignment_tie", "word_without_frames"},
    "random_k2_L6": {"empty_cluster_kept", "single_member_mean", "early_leaf", "leaf_at_depth_L"},
    "k32_root_eq_k": {"node_n_le_k", "early_leaf", "padding_rows", "frame_without_keypoints"},
    "k32_root_k_plus_1": {"node_kmeans", "node_n_le_k", "padding_rows"},
}
# No case reaches the ORBX_VOCAB_MAX_ITERS cap (the most passes any node takes here is 9); the tests assert that the cap
# count the builds report matches the passes they count.
