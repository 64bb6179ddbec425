"""A literal restatement of the keyframe database (orbx_bowdb_*: the first stage of ORB-SLAM2's
KeyFrameDatabase::DetectLoopCandidates with DBoW3's L1Scoring::score, under the rules of include/orbx.h), the ctypes binding
of the plain-C checker oracle_bowdb_query (tests/bowdb_oracle.c), and the crafted databases the tests run on.

The restatement is written the way ORB-SLAM2 writes it: an inverted file of per-word lists filled in frame order, the
mnLoopQuery / mnLoopWords fields of every keyframe, BowVectors as dicts in ascending word id (std::map), and DBoW's
merge-join with lower_bound via bisect.  It counts the branches it takes (`stats`), so every case can assert which rules
it reaches.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile
from bisect import bisect_left
from collections import Counter

import numpy as np

from orb_slam2_ros2_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))


class _KeyFrame:
    def __init__(self, fid: int, bow: dict):
        self.mnId, self.mBowVec = fid, bow
        self.mnLoopQuery, self.mnLoopWords = -1, 0


def l1_score(v1: dict, v2: dict) -> float:
    """DBoW3 L1Scoring::score(v1, v2)"""
    k1, k2 = list(v1), list(v2)
    a = b = 0
    score = 0.0
    while a < len(k1) and b < len(k2):
        vi, wi = v1[k1[a]], v2[k2[b]]
        if k1[a] == k2[b]:
            score += abs(vi - wi) - abs(vi) - abs(wi)
            a += 1
            b += 1
        elif k1[a] < k2[b]:
            a = bisect_left(k1, k2[b], a)
        else:
            b = bisect_left(k2, k1[a], b)
    score = -score / 2.0
    return score


def bow_dicts(ids, vals, n) -> list:
    return [{int(w): float(x) for w, x in zip(ids[f][: n[f]], vals[f][: n[f]])} for f in range(len(n))]


def py_query(bows: list, queries: list, window: int, min_score: float, top_k: int, stats: Counter | None = None):
    """bows[f] = frame f's BowVector (dict); queries = [(query id, BowVector, frame)], frame None = not a database member
    (nothing excluded).  -> dict of arrays as oracle_query returns them"""
    st = stats if stats is not None else Counter()
    kfs = [_KeyFrame(f, b) for f, b in enumerate(bows)]
    inverted = {}
    for kf in kfs:  # KeyFrameDatabase::add
        for w in kf.mBowVec:
            inverted.setdefault(w, []).append(kf)
    if len(kfs) == 1:
        st["one_frame_database"] += 1
    minScore = np.float32(min_score)
    out = dict(cand_frame=[], cand_score=[], cand_common=[], n_sharing=[], max_common=[], n_scored=[], n_kept=[])
    for qid, qbow, qframe in queries:
        connected = set() if qframe is None or window < 0 else {g for g in range(len(kfs)) if abs(g - qframe) <= window}
        lKFsSharingWords = []
        shares_connected = False
        for w in qbow:
            for kfi in inverted.get(w, []):
                if kfi.mnLoopQuery != qid:
                    kfi.mnLoopWords = 0
                    if kfi.mnId not in connected:
                        kfi.mnLoopQuery = qid
                        lKFsSharingWords.append(kfi)
                    else:
                        shares_connected = True
                        if qframe is not None and window > 0 and abs(kfi.mnId - qframe) == window:
                            st["window_edge_excluded"] += 1
                kfi.mnLoopWords += 1
        res = dict(n_sharing=len(lKFsSharingWords), max_common=0, n_scored=0, n_kept=0)
        lScoreAndMatch = []
        if not lKFsSharingWords:
            st["empty_sharing"] += 1
            if shares_connected:
                st["shares_only_connected"] += 1
        else:
            if qframe is not None and window >= 0 and any(abs(k.mnId - qframe) == window + 1 for k in lKFsSharingWords):
                st["window_edge_plus_one_listed"] += 1
            maxCommonWords = max(k.mnLoopWords for k in lKFsSharingWords)
            share = np.float32(maxCommonWords) * np.float32(0.8)
            minCommonWords = int(share)
            st["min_common_whole" if float(share) == minCommonWords else "min_common_truncated"] += 1
            for kfi in lKFsSharingWords:
                if kfi.mnLoopWords == minCommonWords:
                    st["common_eq_min_common_rejected"] += 1
                    if float(share) == minCommonWords:
                        st["common_eq_whole_min_common_rejected"] += 1
                if kfi.mnLoopWords > minCommonWords:
                    res["n_scored"] += 1
                    si = np.float32(l1_score(qbow, kfi.mBowVec))
                    if si >= minScore:
                        if si == minScore:
                            st["score_eq_min_score_kept"] += 1
                        lScoreAndMatch.append((si, kfi))
            res["max_common"], res["n_kept"] = maxCommonWords, len(lScoreAndMatch)
            lScoreAndMatch.sort(key=lambda p: (-float(p[0]), p[1].mnId))
            scores = [float(s) for s, _ in lScoreAndMatch]
            if len(set(scores)) < len(scores):
                st["tied_scores"] += 1
            if lScoreAndMatch:
                st["top_k_below_n_kept" if top_k < len(lScoreAndMatch) else "top_k_at_or_above_n_kept"] += 1
        for key in ("n_sharing", "max_common", "n_scored", "n_kept"):
            out[key].append(res[key])
        row = lScoreAndMatch[:top_k]
        out["cand_frame"].append([k.mnId for _, k in row] + [-1] * (top_k - len(row)))
        out["cand_score"].append([float(s) for s, _ in row] + [0.0] * (top_k - len(row)))
        out["cand_common"].append([k.mnLoopWords for _, k in row] + [0] * (top_k - len(row)))
    dt = dict(cand_frame=np.int32, cand_score=np.float32, cand_common=np.int32)
    return {k: np.array(v, dt.get(k, np.int32)).reshape(len(queries), top_k) if k in dt else np.array(v, np.int32) for k, v in out.items()}


_lib = None


def _oracle_lib():
    """tests/bowdb_oracle.c, compiled once per process with the host C compiler (the flags of oracle/Makefile) into a
    temporary directory that is removed again once the library is loaded"""
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="bowdb_oracle_")
        try:
            so = os.path.join(tmp, "libbowdb_oracle.so")
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", "-o", so, os.path.join(HERE, "bowdb_oracle.c"), "-lm"],
                           check=True, capture_output=True)
            lib = C.CDLL(so)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        lib.oracle_bowdb_query.restype = C.c_int
        lib.oracle_bowdb_query.argtypes = ([C.c_void_p] * 3 + [C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 3 + [C.c_int64, C.c_int32, C.c_int64, C.c_int32,
                                           C.c_float, C.c_int32] + [C.c_void_p] * 4)
        _lib = lib
    return _lib


def oracle_query(db: dict, q: dict, q_frame0: int, window: int, min_score: float, top_k: int) -> dict:
    """oracle_bowdb_query: db / q = dict(ids [F][stride], vals, n) BowVector arrays; query i is frame q_frame0 + i"""
    ids, vals, n = (np.ascontiguousarray(db[k], t) for k, t in (("ids", np.int32), ("vals", np.float64), ("n", np.int32)))
    qi, qv, qn = (np.ascontiguousarray(q[k], t) for k, t in (("ids", np.int32), ("vals", np.float64), ("n", np.int32)))
    nq = len(qn)
    cf, cs, cc = np.zeros((nq, top_k), np.int32), np.zeros((nq, top_k), np.float32), np.zeros((nq, top_k), np.int32)
    cnt = np.zeros((nq, 4), np.int32)
    rc = _oracle_lib().oracle_bowdb_query(ids.ctypes.data, vals.ctypes.data, n.ctypes.data, ids.shape[1], len(n), int(db["n_words"]), qi.ctypes.data,
                                          qv.ctypes.data, qn.ctypes.data, qi.shape[1], nq, q_frame0, window, min_score, top_k, cf.ctypes.data,
                                          cs.ctypes.data, cc.ctypes.data, cnt.ctypes.data)
    assert rc == 0, "oracle_bowdb_query refused the input"
    return dict(cand_frame=cf, cand_score=cs, cand_common=cc, n_sharing=cnt[:, 0].copy(), max_common=cnt[:, 1].copy(), n_scored=cnt[:, 2].copy(),
                n_kept=cnt[:, 3].copy())


def bow_arrays(oracle, O, desc, counts, levelsup: int = 4) -> dict:
    """every frame's BowVector by oracle_bow_transform -> dict(ids [F][stride], vals, n, n_words)"""
    F, stride = len(counts), desc.shape[1]
    ids, vals, n = np.zeros((F, stride), np.int32), np.zeros((F, stride), np.float64), np.zeros(F, np.int32)
    for f in range(F):
        r = oracle.bow_transform(O, desc[f][: counts[f]], levelsup)
        m = len(r["bow_ids"])
        ids[f, :m], vals[f, :m], n[f] = r["bow_ids"], r["bow_vals"], m
    return dict(ids=ids, vals=vals, n=n, n_words=int((O.word_id >= 0).sum()))


# ---- crafted databases --------------------------------------------------------------------------------------------
def word_descriptors(oracle, voc: dict):
    """-> (descriptor of each usable word in ascending word id, descriptors whose word is stopped): a leaf's descriptor is
    taken when its oracle descent ends in a single word"""
    O = oracle.Vocabulary(**voc)
    words, stopped = {}, []
    for r in np.nonzero(voc["is_leaf"])[0]:
        d = voc["desc"][r][None]
        b = oracle.bow_transform(O, d, 4)
        if len(b["bow_ids"]) == 1:
            words.setdefault(int(b["bow_ids"][0]), d[0])
        elif len(b["bow_ids"]) == 0:
            stopped.append(d[0])
    return O, [words[w] for w in sorted(words)], stopped


# frames of the crafted loop database as (first word, last word) runs of the word pool; 'stopped' / 'empty' / ('dup', f)
LOOP_FRAMES = [
    [(0, 10), (20, 23)],  # 0: shares all 10 words of frame 5: max_common 10 -> min_common 8 (whole)
    [(0, 8), (23, 26)],   # 1: 8 == min_common: rejected by the strict >
    [(0, 9), (26, 28)],   # 2: 9: scored
    [(0, 9), (28, 30)],   # 3: |3 - 5| = 2 = window + 1: listed
    [(0, 10)],            # 4: |4 - 5| = 1 = window: connected
    [(0, 10)],            # 5: the main query
    [(0, 10), (30, 31)],  # 6: |6 - 5| = window: connected
    "empty",              # 7: no keypoints
    "stopped",            # 8: keypoints whose words are all stopped
    ("dup", 0),           # 9: frame 0 again: a tie with frame 0, ordered by frame id
    [(0, 3), (31, 34)],   # 10: 3 shared: below min_common
    [(40, 47)],           # 11: shares only with 12
    [(40, 47), (47, 48)], # 12: shares only with 11 (connected at window 1)
    [(60, 67)],           # 13: max_common 7 -> min_common 5 (truncated from 5.6)
    [(70, 72)],           # 14
    [(60, 67), (72, 74)], # 15: 7 shared with 13
    [(60, 65), (74, 76)], # 16: 5 == min_common: rejected
    [(60, 66), (76, 78)], # 17: 6: scored
]


def _assemble(frames, pool, stopped, stride: int, seed: int):
    rng = np.random.default_rng(seed)
    F = len(frames)
    desc = rng.integers(0, 256, (F, stride, 32), dtype=np.uint8)
    counts = np.zeros(F, np.int32)
    for f, spec in enumerate(frames):
        if spec == "empty":
            continue
        if spec == "stopped":
            rows = [stopped[i % len(stopped)] for i in range(3)]
        elif isinstance(spec, tuple):
            rows = list(desc[spec[1]][: counts[spec[1]]])
        else:
            rows = []
            for a, b in spec:
                for w in range(a, b):
                    rows += [pool[w]] * (1 + (w * 7 + f * 3) % 3)  # repeats: term frequencies differ between frames
        rows = [rows[i] for i in rng.permutation(len(rows))] if not isinstance(spec, tuple) else rows
        assert len(rows) <= stride
        desc[f, : len(rows)] = rows
        counts[f] = len(rows)
    return desc, counts


def case(oracle, name: str) -> dict:
    """-> dict(voc, desc, counts, configs=[(window, min_score, top_k)], queries=(lo, hi)) of one named database"""
    voc = synth.synth_vocabulary(10, 3, 21)
    O, pool, stopped = word_descriptors(oracle, voc)
    assert len(pool) > 80 and stopped
    if name == "loop":
        desc, counts = _assemble(LOOP_FRAMES, pool, stopped, 32, 1)
        F = len(counts)
        db = bow_arrays(oracle, O, desc, counts)
        # min_score equal to one kept score of the main query (frame 5, window 1)
        r = py_query(bow_dicts(db["ids"], db["vals"], db["n"]), [(5, bow_dicts(db["ids"][5:6], db["vals"][5:6], db["n"][5:6])[0], 5)], 1, 0.0, F)
        mid = float(r["cand_score"][0][1])
        configs = [(1, 0.0, 3), (1, 0.0, F), (1, mid, F), (0, 0.0, 2), (3, 0.0, 5), (1, -1.0, 1)]
        return dict(voc=voc, O=O, desc=desc, counts=counts, db=db, configs=configs)
    if name == "one_frame":
        desc, counts = _assemble([[(0, 6)]], pool, stopped, 16, 2)
        return dict(voc=voc, O=O, desc=desc, counts=counts, db=bow_arrays(oracle, O, desc, counts), configs=[(0, 0.0, 1)])
    raise KeyError(name)


CASES = ["loop", "one_frame"]
