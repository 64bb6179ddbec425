"""ORBMatcher::searchByStereo (src/ORBMatcher.cc:18-81, with createRowIndexDB / getBestMatch / pixelSADMatch / getPitch /
SAD at :841-1011) restated line by line in Python, with the float and double steps of oracle_search_by_stereo, plus a
census of the branch every left keypoint ends in.

Outcomes, one per left keypoint:
  row_outside      cvRound(y) of the undistorted left keypoint is not an image row (the reference indexes rowIdxDB out
                   of range; no candidates here, as in the kernel and the oracle)
  no_candidate     no right keypoint in the row band with minU < x < maxU
  dist_gt_75       best Hamming distance > 75 (mnMeanThreshold)
  octave_mismatch  the octaves differ by more than one
  window_outside   the left 11x11 or the right 11x21 SAD window leaves its level image (the reference throws in
                   cv::Mat::rowRange; dropped, DESIGN section 2)
  sad_edge         the SAD minimum is at shift -5 or +5: no parabola, uRight = the right keypoint's x
  parabola         the parabola refinement (or its |delta| >= 1 reset) gives uRight
  fallback         uRight ended at or right of the left x, so uRight = the right keypoint's x (the `disp <= 0` branch)
Counters across keypoints:
  hamming_tie           the best distance is shared by several candidates (the first, lowest index, wins)
  sad_tie               the smallest SAD is shared by several shifts (the first wins)
  minU_excluded_better  a right keypoint of the row band at or left of minU is strictly closer than the chosen one
  dist_eq_75            the best distance is exactly 75 (kept: the test is `> 75`)
  x_eq_maxU             a right keypoint of the row band lies exactly at the left x (excluded: the test is `x < maxU`)

Not reachable, so not counted: the clamps of uRight to [0, W - 1] and the second `disp <= 0` return.  Right keypoints lie
at least 16 level pixels, i.e. 16 * sf, inside the image and |delta| < sf, so uRight stays inside; and the fallback's
uRight is the right keypoint's x, which the strict `x < maxU` filter put left of the left x.
"""
from __future__ import annotations

from collections import Counter

import numpy as np

f32, f64 = np.float32, np.float64
OUTCOMES = ("row_outside", "no_candidate", "dist_gt_75", "octave_mismatch", "window_outside", "sad_edge", "parabola", "fallback")
COUNTERS = ("hamming_tie", "sad_tie", "minU_excluded_better", "dist_eq_75", "x_eq_maxU")


def cv_round(v) -> int:
    return int(np.rint(f32(v)))  # lrintf: round half to even


def cv_floor(v) -> int:
    return int(np.floor(f32(v)))


def create_row_index_db(kr, sf, rows):
    """:915-932 -> list over image rows of the right keypoint indices whose band covers the row, ascending"""
    db = [[] for _ in range(rows)]
    for j in range(len(kr)):
        r = f32(2.0 * f64(sf[kr["octave"][j]]))
        row = cv_round(kr["y"][j])  # unsigned row
        max_row = min(rows, cv_round(f32(f32(row) + r) + f32(1)))
        min_row = max(0, cv_round(f32(row) - r))
        for y in range(min_row, max_row):
            db[y].append(j)
    return [np.asarray(r, np.int64) for r in db]


_POPC = np.array([bin(v).count("1") for v in range(256)], np.int64)


def _distance(a, b):
    """:941-956, the bit count of a ^ b over the 32 bytes, against each row of b"""
    return _POPC[a[None, :] ^ b].sum(1)


def _sad(li, lx, ly, ri, rx, ry):
    """:893-905 on the centre-subtracted 11x11 patches; every term is an integer, so the double sum is exact"""
    a = li[ly - 5 : ly + 6, lx - 5 : lx + 6].astype(np.int64) - int(li[ly, lx])
    b = ri[ry - 5 : ry + 6, rx - 5 : rx + 6].astype(np.int64) - int(ri[ry, rx])
    return f32(np.abs(a - b).sum())


def search_by_stereo(left_levels, right_levels, sf, kl, dl, kr, dr, fx, bf, width, height):
    """left_levels / right_levels: the un-blurred pyramid level images; kl: the undistorted left keypoints.
    -> dict(n_matches, u_right, depth, match_idx, outcome (per left keypoint), census (Counter))"""
    fx, bf = f32(fx), f32(bf)
    nl = len(kl)
    ur, dp = np.full(nl, -1.0), np.full(nl, -1.0)
    mi = np.full(nl, -1, np.int64)
    outcome = []
    census = Counter({k: 0 for k in OUTCOMES + COUNTERS})
    db = create_row_index_db(kr, sf, height)
    krx = kr["x"].astype(f32)
    n_matches = 0
    for i in range(nl):
        lx_f, ly_f, lo = f32(kl["x"][i]), f32(kl["y"][i]), int(kl["octave"][i])
        max_u = lx_f
        min_u = lx_f - fx if lx_f - fx > f32(0) else f32(0)
        row = cv_round(ly_f)
        if row < 0 or row >= height:
            outcome.append("row_outside")
            census["row_outside"] += 1
            continue
        band = db[row]
        xr = krx[band]
        inside = (xr < max_u) & (xr > min_u)
        cand = band[inside]
        census["x_eq_maxU"] += int((xr == max_u).any())
        d = _distance(dl[i], dr[cand])
        best_d = int(d.min()) if len(cand) else 1 << 30
        below = band[(xr <= min_u) & (xr < max_u)]
        if len(below) and int(_distance(dl[i], dr[below]).min()) < best_d:
            census["minU_excluded_better"] += 1
        if not len(cand):
            outcome.append("no_candidate")
            census["no_candidate"] += 1
            continue
        best_j = int(cand[int(np.argmin(d))])  # argmin == the first minimum over ascending indices
        census["hamming_tie"] += int((d == best_d).sum() > 1)
        census["dist_eq_75"] += int(best_d == 75)
        if best_d > 75:
            outcome.append("dist_gt_75")
            census["dist_gt_75"] += 1
            continue
        ro = int(kr["octave"][best_j])
        if lo > ro + 1 or lo < ro - 1:
            outcome.append("octave_mismatch")
            census["octave_mismatch"] += 1
            continue
        rx_f, ry_f = f32(kr["x"][best_j]), f32(kr["y"][best_j])
        li, ri = left_levels[lo], right_levels[ro]
        lx, ly = cv_floor(lx_f / f32(sf[lo])), cv_floor(ly_f / f32(sf[lo]))
        rx, ry = cv_floor(rx_f / f32(sf[ro])), cv_floor(ry_f / f32(sf[ro]))
        if lx - 5 < 0 or ly - 5 < 0 or lx + 5 >= li.shape[1] or ly + 5 >= li.shape[0] or rx - 10 < 0 or ry - 5 < 0 or rx + 10 >= ri.shape[1] or ry + 5 >= ri.shape[0]:
            outcome.append("window_outside")
            census["window_outside"] += 1
            continue
        # pixelSADMatch :841-881
        scores = [_sad(li, lx, ly, ri, rx + s, ry) for s in range(-5, 6)]
        min_score, best = f32(3.402823466e38), 0
        for k, s in enumerate(scores):
            if s < min_score:
                min_score, best = s, k
        census["sad_tie"] += int(sum(s == min_score for s in scores) > 1)
        delta = f32(0)
        if 0 < best < 10:
            s1, s2, s3 = scores[best - 1], scores[best], scores[best + 1]
            delta = f32(f64(0.5) * f64(f32(s1 - s3)) / f64(f32(f32(s1 + s3) - f32(f32(2) * s2))))
            delta = f32(delta * f32(sf[ro])) if f32(-1) < delta < f32(1) else f32(0)
        label = "parabola" if 0 < best < 10 else "sad_edge"
        right_u = f32(rx_f + delta)
        right_u = right_u if right_u > f32(0) else f32(0)
        lim = f32(width) - f32(1)
        right_u = right_u if right_u < lim else lim
        disp = f32(lx_f - right_u)
        if disp <= f32(0):
            right_u = rx_f
            disp = f32(lx_f - right_u)
            assert disp > f32(0)  # the second `return` of the branch: unreachable, see the module comment
            label = "fallback"
        outcome.append(label)
        census[label] += 1
        ur[i] = f64(right_u)
        dp[i] = f64(f32(bf / disp))
        mi[i] = best_j
        n_matches += 1
    return dict(n_matches=n_matches, u_right=ur, depth=dp, match_idx=mi, outcome=outcome, census=census)
