"""A literal restatement of loop verification (orbx_loopver_*: the check of ORB-SLAM2's LoopClosing::ComputeSim3 --
searchByBow with the candidate as the keyframe, verifyAngle, and Sim3Solver's RANSAC with Horn's closed form at a fixed scale,
under the rules of include/orbx.h), the ctypes binding of the plain-C checker oracle_loopver (tests/loopver_oracle.c), and
the crafted record sets the tests run on.

The restatement is written the way ORB-SLAM2 writes it: Sim3Solver::iterate runs one hypothesis after another, the sample
indices come out of a vector (`vAvailableIndices[randi] = vAvailableIndices.back(); pop_back()`), Horn's N goes through a
plain cyclic Jacobi loop, and SetRansacParameters computes the iteration count.  The matching stage is the already pinned
oracle_search_by_bow / oracle_verify_angle / oracle_bow_transform.  It counts the rules it reaches (`stats`).
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

from orb_slam2_ros2_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
COUNTS = ("n_bow", "n_matches", "n_corr", "n_iters", "hypothesis", "n_inliers", "accepted")
JACOBI_SWEEPS = 16  # ORBX_LOOPVER_JACOBI_SWEEPS
GOLDEN = 0x9E3779B97F4A7C15
M64 = (1 << 64) - 1


def splitmix64(x: int) -> int:
    z = (x + GOLDEN) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


# ---- the restatement ---------------------------------------------------------------------------------------------
def ransac_iterations(n: int, min_inliers: int, max_iterations: int, probability: float) -> int:
    """Sim3Solver::SetRansacParameters; 0 when there are fewer correspondences than min_inliers (iterate() returns at once)"""
    if n < min_inliers:
        return 0
    if n == min_inliers:
        it = 1.0
    else:
        epsilon = float(np.float32(min_inliers) / np.float32(n))
        it = float(math.ceil(math.log(1 - probability) / math.log(1 - math.pow(epsilon, 3))))
    return 1 if it < 1 else max_iterations if it > max_iterations else int(it)


def slot_sum(xs, slots) -> float:
    p = [0.0] * 32
    for x, s in zip(xs, slots):
        p[s % 32] += x
    s = 16
    while s:
        for l in range(s):
            p[l] += p[l + s]
        s >>= 1
    return p[0]


def horn(P1, P2, slots):
    """Sim3Solver::ComputeSim3(P1 = query points, P2 = candidate points) with mbFixScale; R from the quaternion's homogeneous
    form.  -> 15 floats: R row-major, t (T12: candidate -> query), -R^T t"""
    m = len(P1)
    O1 = [slot_sum([p[d] for p in P1], slots) / m for d in range(3)]
    O2 = [slot_sum([p[d] for p in P2], slots) / m for d in range(3)]
    Mm = [[slot_sum([(P2[k][a] - O2[a]) * (P1[k][b] - O1[b]) for k in range(m)], slots) for b in range(3)] for a in range(3)]
    N11 = Mm[0][0] + Mm[1][1] + Mm[2][2]
    N12 = Mm[1][2] - Mm[2][1]
    N13 = Mm[2][0] - Mm[0][2]
    N14 = Mm[0][1] - Mm[1][0]
    N22 = Mm[0][0] - Mm[1][1] - Mm[2][2]
    N23 = Mm[0][1] + Mm[1][0]
    N24 = Mm[2][0] + Mm[0][2]
    N33 = -Mm[0][0] + Mm[1][1] - Mm[2][2]
    N34 = Mm[1][2] + Mm[2][1]
    N44 = -Mm[0][0] - Mm[1][1] + Mm[2][2]
    A = [[N11, N12, N13, N14], [N12, N22, N23, N24], [N13, N23, N33, N34], [N14, N24, N34, N44]]
    V = [[1.0 if i == j else 0.0 for j in range(4)] for i in range(4)]
    for _sweep in range(JACOBI_SWEEPS):
        if all(A[p][q] == 0 for p in range(4) for q in range(p + 1, 4)):
            break
        for p in range(3):
            for q in range(p + 1, 4):
                if A[p][q] == 0:
                    continue
                theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q])
                t = 1.0 / (abs(theta) + math.sqrt(theta * theta + 1.0))
                if theta < 0:
                    t = -t
                c = 1.0 / math.sqrt(t * t + 1.0)
                s = t * c
                for k in range(4):
                    akp, akq = A[k][p], A[k][q]
                    A[k][p], A[k][q] = c * akp - s * akq, s * akp + c * akq
                for k in range(4):
                    apk, aqk = A[p][k], A[q][k]
                    A[p][k], A[q][k] = c * apk - s * aqk, s * apk + c * aqk
                A[p][q] = A[q][p] = 0.0
                for k in range(4):
                    vkp, vkq = V[k][p], V[k][q]
                    V[k][p], V[k][q] = c * vkp - s * vkq, s * vkp + c * vkq
    mx = 0
    for i in range(1, 4):
        if A[i][i] > A[mx][mx]:
            mx = i
    w, x, y, z = V[0][mx], V[1][mx], V[2][mx], V[3][mx]
    ww, xx, yy, zz = w * w, x * x, y * y, z * z
    n2 = ww + xx + yy + zz
    R = [(ww + xx - yy - zz) / n2, 2.0 * (x * y - w * z) / n2, 2.0 * (x * z + w * y) / n2,
         2.0 * (x * y + w * z) / n2, (ww - xx + yy - zz) / n2, 2.0 * (y * z - w * x) / n2,
         2.0 * (x * z - w * y) / n2, 2.0 * (y * z + w * x) / n2, (ww - xx - yy + zz) / n2]
    t = [O1[r] - (R[3 * r] * O2[0] + R[3 * r + 1] * O2[1] + R[3 * r + 2] * O2[2]) for r in range(3)]
    ti = [-(R[r] * t[0] + R[3 + r] * t[1] + R[6 + r] * t[2]) for r in range(3)]
    return R + t + ti


def check_inlier(T, Xc, Xq, uvc, uvq, thr_c, thr_q, cam, stats):
    """Sim3Solver::CheckInliers for one correspondence, against the keypoint positions"""
    fx, fy, cx, cy = cam
    Y = [T[3 * r] * Xc[0] + T[3 * r + 1] * Xc[1] + T[3 * r + 2] * Xc[2] + T[9 + r] for r in range(3)]
    Z = [T[r] * Xq[0] + T[3 + r] * Xq[1] + T[6 + r] * Xq[2] + T[12 + r] for r in range(3)]
    if Y[2] <= 0 or Z[2] <= 0:
        stats["point_behind_camera"] += 1
    with np.errstate(all="ignore"):
        iy, iz = (1.0 / Y[2] if Y[2] != 0 else math.copysign(math.inf, Y[2])), (1.0 / Z[2] if Z[2] != 0 else math.copysign(math.inf, Z[2]))
        du1, dv1 = uvq[0] - (fx * (Y[0] * iy) + cx), uvq[1] - (fy * (Y[1] * iy) + cy)
        du2, dv2 = uvc[0] - (fx * (Z[0] * iz) + cx), uvc[1] - (fy * (Z[1] * iz) + cy)
        e1, e2 = du1 * du1 + dv1 * dv1, du2 * du2 + dv2 * dv2
    return e1 < thr_q and e2 < thr_c


def py_verify(oracle, O, levelsup, fr: dict, cam, sf, q_lo: int, table, prm: dict, stats: Counter | None = None) -> dict:
    """fr = dict(kps [F][N], desc [F][N][32], depth [F][N], n [F]); table [nq][top_k] -> dict of oracle_verify's outputs"""
    st = stats if stats is not None else Counter()
    F, N = fr["kps"].shape
    table = np.asarray(table)
    nq, top_k = table.shape
    bows = [oracle.bow_transform(O, fr["desc"][f][: fr["n"][f]], levelsup) for f in range(F)]
    sig = [float(np.float32(sf[l]) * np.float32(sf[l])) if l < len(sf) else 1.0 for l in range(64)]
    ratio = np.float32(prm["ratio"])
    out = {k: np.zeros((nq, top_k), np.int32) for k in COUNTS}
    out["hypothesis"][:] = -1
    out.update(T=np.zeros((nq, top_k, 12)), match=np.full((nq, top_k, N), -1, np.int32), loop_frame=np.full(nq, -1, np.int32))
    seed_key = splitmix64(prm["seed"] & M64)
    for qi in range(nq):
        qf = q_lo + qi
        accepted = []
        for sl in range(top_k):
            cf = int(table[qi, sl])
            if cf < 0:
                st["empty_slot"] += 1
                continue
            if cf == qf:
                st["candidate_is_query"] += 1
            nqf, ncf = fr["n"][qf], fr["n"][cf]
            kq, kc = fr["kps"][qf][:nqf], fr["kps"][cf][:ncf]
            # searchByBow(pFrame = query, pKframe = candidate, bLoop): keep iff dist <= 50 && !(ratio > mfRatio)
            r = oracle.search_by_bow(bows[qf], fr["desc"][qf][:nqf], bows[cf], fr["desc"][cf][:ncf])
            keep = ~((r["best_dist"] > 50) | (r["ratio"] > ratio))
            qi_, ti_, _ = oracle.verify_angle(r["best_idx"][keep], r["kf_idx"][keep], r["best_dist"][keep].astype(np.float32), kq, kc)
            out["n_bow"][qi, sl], out["n_matches"][qi, sl] = int(keep.sum()), len(qi_)
            if len(qi_) < int(keep.sum()):
                st["rotation_check_drops"] += 1
            for a, b in zip(qi_, ti_):
                out["match"][qi, sl, b] = a
            nmatches = len(qi_)
            if nmatches < prm["min_matches"]:
                st["matches_below_min" if nmatches == prm["min_matches"] - 1 else "matches_far_below_min"] += 1
                continue
            if nmatches == prm["min_matches"]:
                st["matches_at_min"] += 1
            # Sim3Solver's constructor: the matches whose two features have a depth
            P1, P2, uvq, uvc, thq, thc = [], [], [], [], [], []
            for a, b in zip(qi_, ti_):
                zq, zc = float(fr["depth"][qf][a]), float(fr["depth"][cf][b])
                if not (zq > 0 and zc > 0):
                    st["zero_depth_dropped"] += 1
                    continue
                pq, pc = kq[a], kc[b]
                P1.append([(float(pq["x"]) - cam[2]) * zq / cam[0], (float(pq["y"]) - cam[3]) * zq / cam[1], zq])
                P2.append([(float(pc["x"]) - cam[2]) * zc / cam[0], (float(pc["y"]) - cam[3]) * zc / cam[1], zc])
                uvq.append((float(pq["x"]), float(pq["y"])))
                uvc.append((float(pc["x"]), float(pc["y"])))
                thq.append(9.210 * sig[int(pq["octave"])])
                thc.append(9.210 * sig[int(pc["octave"])])
            n = len(P1)
            out["n_corr"][qi, sl] = n
            nit = ransac_iterations(n, prm["min_inliers"], prm["max_iterations"], prm["probability"])
            if n < prm["min_inliers"]:
                st["corr_below_min_inliers"] += 1
            elif n == prm["min_inliers"]:
                st["corr_eq_min_inliers_one_iteration"] += 1
            # Sim3Solver::iterate
            K = splitmix64((splitmix64((seed_key + qf + 1) & M64) + cf + 1) & M64)
            best_n, best_h, best_T, acc = 0, -1, None, False
            for h in range(nit):
                vAvailableIndices = list(range(n))
                idx = []
                for j in range(3):
                    randi = splitmix64(K ^ (((3 * h + j) * GOLDEN) & M64)) % (n - j)
                    idx.append(vAvailableIndices[randi])
                    vAvailableIndices[randi] = vAvailableIndices[-1]
                    vAvailableIndices.pop()
                S1, S2 = [P1[i] for i in idx], [P2[i] for i in idx]
                d1, d2 = np.subtract(S2[1], S2[0]), np.subtract(S2[2], S2[0])
                if S2[0] == S2[1] or S2[1] == S2[2] or S2[0] == S2[2]:
                    st["coincident_sample"] += 1
                elif np.linalg.norm(np.cross(d1, d2)) <= 1e-6 * float(np.linalg.norm(d1) * np.linalg.norm(d2)):
                    st["collinear_sample"] += 1  # three distinct points on a line, up to the float32 rounding of their keypoints
                T = horn(S1, S2, [0, 1, 2])
                nin = sum(check_inlier(T, P2[i], P1[i], uvc[i], uvq[i], thc[i], thq[i], cam, st) for i in range(n))
                if nin == prm["min_inliers"]:
                    st["inliers_eq_min_not_accepted"] += 1
                if nin >= best_n:
                    if nin == best_n and best_h >= 0:
                        st["tied_best"] += 1
                    best_n, best_h, best_T = nin, h, T
                    if nin > prm["min_inliers"]:
                        acc = True
                        if nin == prm["min_inliers"] + 1:
                            st["accepted_at_min_plus_one"] += 1
                        break
            out["n_iters"][qi, sl] = best_h + 1 if acc else nit
            out["hypothesis"][qi, sl] = best_h
            out["n_inliers"][qi, sl] = best_n if best_h >= 0 else 0
            out["accepted"][qi, sl] = int(acc)
            if best_h < 0:
                continue
            if best_n >= 3:
                inl = [i for i in range(n) if check_inlier(best_T, P2[i], P1[i], uvc[i], uvq[i], thc[i], thq[i], cam, Counter())]
                Tf = horn([P1[i] for i in inl], [P2[i] for i in inl], inl)
            else:
                st["refit_from_samples"] += 1
                Tf = best_T
            out["T"][qi, sl] = Tf[:12]
            if acc:
                accepted.append((best_h // 5, sl, cf))
        if accepted:
            rnd, sl, cf = min(accepted)
            out["loop_frame"][qi] = cf
            if any(s < sl for _, s, _ in accepted):
                st["loop_frame_by_round"] += 1
    return out


# ---- the C oracle -------------------------------------------------------------------------------------------------
_lib = None


def _oracle_lib():
    """tests/loopver_oracle.c and oracle/orb_oracle.c, compiled once per process with the host C compiler (the flags of
    oracle/Makefile) into a temporary directory that is removed again once the library is loaded"""
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="loopver_oracle_")
        try:
            so = os.path.join(tmp, "libloopver_oracle.so")
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", so,
                            os.path.join(HERE, "loopver_oracle.c"), os.path.join(ROOT, "oracle", "orb_oracle.c"), "-lm"], check=True, capture_output=True)
            lib = C.CDLL(so)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        lib.oracle_loopver.restype = C.c_int
        lib.oracle_loopver.argtypes = ([C.c_void_p, C.c_int, C.c_int32, C.c_int32] + [C.c_void_p] * 4 + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_int64, C.c_int32,
                                       C.c_void_p, C.c_int32, C.c_float, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_uint64] + [C.c_void_p] * 5)
        _lib = lib
    return _lib


def oracle_verify(O, levelsup: int, fr: dict, cam, sf, q_lo: int, table, prm: dict) -> dict:
    """oracle_loopver -> dict of LOOPVER_OUTPUTS, and first_best [nq][top_k]: the first hypothesis that reached the
    reported hypothesis's inlier count (-1 without one)"""
    kps = np.ascontiguousarray(fr["kps"])
    desc, depth, n = (np.ascontiguousarray(fr[k], t) for k, t in (("desc", np.uint8), ("depth", np.float64), ("n", np.int32)))
    F, N = kps.shape
    tab = np.ascontiguousarray(table, np.int32)
    nq, top_k = tab.shape
    sfa = np.ascontiguousarray(sf, np.float32)
    counts, T, match, lf = np.zeros((nq, top_k, 7), np.int32), np.zeros((nq, top_k, 12)), np.zeros((nq, top_k, N), np.int32), np.zeros(nq, np.int32)
    first = np.zeros((nq, top_k), np.int32)
    rc = _oracle_lib().oracle_loopver(C.addressof(O._c), levelsup, F, N, kps.ctypes.data, desc.ctypes.data, depth.ctypes.data, n.ctypes.data, cam[0], cam[1],
                                      cam[2], cam[3], sfa.ctypes.data, len(sfa), q_lo, nq, tab.ctypes.data, top_k, prm["ratio"], prm["min_matches"],
                                      prm["min_inliers"], prm["max_iterations"], prm["probability"], prm["seed"] & M64, counts.ctypes.data, T.ctypes.data,
                                      match.ctypes.data, lf.ctypes.data, first.ctypes.data)
    assert rc == 0
    out = {k: counts[:, :, i].copy() for i, k in enumerate(COUNTS)}
    out.update(T=T, match=match, loop_frame=lf, first_best=first)
    return out


def params(ratio=0.75, min_matches=20, min_inliers=20, max_iterations=300, probability=0.99, seed=0) -> dict:
    return dict(ratio=ratio, min_matches=min_matches, min_inliers=min_inliers, max_iterations=max_iterations, probability=probability, seed=seed)


# ---- crafted record sets ------------------------------------------------------------------------------------------
CAM = (300.0, 300.0, 160.0, 120.0)  # fx fy cx cy (float32-exact)
N_FEATURES, N_LEVELS, SCALE = 128, 4, 1.2


def rot(axis, deg) -> np.ndarray:
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    t = math.radians(deg)
    return np.eye(3) + math.sin(t) * K + (1 - math.cos(t)) * K @ K


class _Builder:
    """frames of landmarks (3-D point + descriptor + base angle) seen from known poses X_cam = R X_world + t"""

    def __init__(self, seed: int, kp_dtype, n_features: int = N_FEATURES, n_levels: int = N_LEVELS, voc=None, levelsup: int = 0):
        """voc, levelsup: when given, a landmark's copy with flipped bits keeps its landmark's FeatureVector node and a word
        that is not stopped"""
        self.rng = np.random.default_rng(seed)
        self.kp_dtype = kp_dtype
        self.N, self.n_levels = n_features, n_levels
        self.voc, self.levelsup = voc, levelsup
        if voc is not None:
            self.bits = np.unpackbits(voc["desc"], axis=1)
            self.children = [np.flatnonzero(voc["parent"] == p) for p in range(len(voc["parent"]) + 1)]
        self.frames = []

    def landmarks(self, P) -> list:
        P = np.asarray(P, float)
        return [dict(X=P[i], d=self.rng.integers(0, 256, 32, dtype=np.uint8), a=float(self.rng.uniform(-170, 170))) for i in range(len(P))]

    def box(self, n, z=(3.0, 7.0)) -> list:
        return self.landmarks(np.stack([self.rng.uniform(-2, 2, n), self.rng.uniform(-1.5, 1.5, n), self.rng.uniform(*z, n)], 1))

    def node(self, d) -> int:
        """the FeatureVector node descriptor d descends to (oracle_bow_descend), or -1 for a stopped word"""
        b, node, at, level = np.unpackbits(d), 0, 0, 0
        while len(self.children[node]):
            level += 1
            c = self.children[node]
            node = int(c[(self.bits[c] != b).sum(1).argmin()]) + 1  # record i is node i + 1
            if level == self.voc["L"] - self.levelsup:
                at = node
        return at if self.voc["weight"][node - 1] > 0 else -1

    def copy_desc(self, d, flip: int):
        """d with `flip` random bits flipped, in d's node"""
        while True:
            c = d.copy()
            for b in self.rng.choice(256, flip, replace=False):
                c[b // 8] ^= np.uint8(1 << (b % 8))
            if self.voc is None or self.node(c) == self.node(d):
                return c

    def frame(self, lms, R=np.eye(3), t=(0, 0, 0), spin=0.0, no_depth=(), wrong=(), bad_angle=(), extra=20, turn=None, flip=0) -> int:
        """features: every landmark (those in `wrong` at a random point instead), `extra` distractors; no_depth: landmark
        positions in `lms` whose feature has no depth; bad_angle: positions whose angle breaks the rotation check; turn:
        {position: degrees} added to those landmarks' angles as given; flip: bits flipped in each landmark's descriptor"""
        feats = []
        bad = sorted(bad_angle)
        for i, lm in enumerate(lms):
            X = np.asarray(R) @ lm["X"] + np.asarray(t, float)
            if i in wrong:
                X = np.array([self.rng.uniform(-3, 3), self.rng.uniform(-2, 2), self.rng.uniform(2, 9)])
            ang = lm["a"] - spin + (60.0 + 40.0 * bad.index(i) if i in bad_angle else 0.0)  # one rotation bin each
            if turn is not None:
                ang += turn.get(i, 0.0)
            ang = (ang + 180.0) % 360.0 - 180.0
            feats.append((X, self.copy_desc(lm["d"], flip) if flip else lm["d"], ang, -1.0 if i in no_depth else X[2]))
        for _ in range(extra):
            X = np.array([self.rng.uniform(-2, 2), self.rng.uniform(-1.5, 1.5), self.rng.uniform(3, 7)])
            feats.append((X, self.rng.integers(0, 256, 32, dtype=np.uint8), float(self.rng.uniform(-170, 170)), X[2]))
        assert len(feats) <= self.N
        order = self.rng.permutation(len(feats))
        kps = np.zeros(self.N, self.kp_dtype)
        desc = np.zeros((self.N, 32), np.uint8)
        depth = np.zeros(self.N)
        for j, k in enumerate(order):
            X, d, ang, z = feats[k]
            kps[j]["x"], kps[j]["y"] = np.float32(CAM[0] * X[0] / X[2] + CAM[2]), np.float32(CAM[1] * X[1] / X[2] + CAM[3])
            kps[j]["angle"], kps[j]["octave"], kps[j]["size"] = ang, int(self.rng.integers(0, self.n_levels)), 7.0
            desc[j], depth[j] = d, z
        self.frames.append((kps, desc, depth, len(feats)))
        return len(self.frames) - 1

    def arrays(self) -> dict:
        return dict(kps=np.stack([f[0] for f in self.frames]), desc=np.stack([f[1] for f in self.frames]), depth=np.stack([f[2] for f in self.frames]),
                    n=np.array([f[3] for f in self.frames], np.int32))


def crafted(kp_dtype, seed: int = 3) -> dict:
    """-> dict(frames, table, configs=[params], truth={(query, candidate): (R, t)})"""
    B = _Builder(seed, kp_dtype)
    truth, rows = {}, []
    Rc, tc = rot([0.2, 1, 0.1], 8.0), np.array([0.25, -0.05, 0.1])
    L0 = B.box(60)

    def pair(lms, **kw):
        f = B.frame(lms, Rc, tc, spin=8.0, **kw)
        return f

    # query 0: 19 / 20 / 21 matches, all with depth: below min_matches, n_corr == min_inliers (one iteration), accepted at 21
    q0 = B.frame(L0)
    rows.append((q0, [pair(L0[:19]), pair(L0[:20]), pair(L0[:21])]))
    # query 1: most depths missing; one wrong point among 21 (20 inliers: never accepted, every hypothesis ties); half wrong
    q1 = B.frame(L0)
    rows.append((q1, [pair(L0[:40], no_depth=set(range(25))), pair(L0[:21], wrong={20}), pair(L0, wrong=set(range(0, 60, 2)), bad_angle={1, 3, 5, 7, 9})]))
    # query 2: collinear landmarks; the query itself as a candidate; an empty slot
    line = B.landmarks([[-1.5 + 0.1 * i, 0.5 - 0.03 * i, 4.0 + 0.05 * i] for i in range(30)])
    q2 = B.frame(line)
    rows.append((q2, [pair(line), q2, -1]))
    # query 3: coincident landmarks (ten features at one point) and a few without depth
    co = B.landmarks([[0.3, 0.2, 5.0]] * 10 + list(np.stack([np.linspace(-1.5, 1.5, 16), np.sin(np.arange(16)), np.linspace(3, 6, 16)], 1)))
    q3 = B.frame(co)
    rows.append((q3, [pair(co, no_depth={12, 13}), -1, pair(co[:12])]))
    # queries 4..7: several half-wrong candidates each, so that an earlier slot is accepted in a later round of five
    for _ in range(4):
        L = B.box(70)
        q = B.frame(L)
        rows.append((q, [pair(L, wrong=set(B.rng.choice(70, 36, replace=False).tolist())) for _ in range(3)]))
    # every frame is a query; frames without a row get an empty one, a frame of another row, or themselves
    fr = B.arrays()
    F = len(fr["n"])
    table = np.full((F, 3), -1, np.int32)
    for q, cands in rows:
        table[q] = cands
    truth[(q0, rows[0][1][2])] = (Rc.T, -Rc.T @ tc)
    table[rows[0][1][2]] = [rows[0][1][2], -1, q0]  # a candidate frame queried against itself and its query
    configs = [params(), params(seed=7), params(min_inliers=8, min_matches=12, seed=11), params(ratio=0.6, max_iterations=4, seed=5),
               params(min_inliers=3, min_matches=3, max_iterations=40, probability=0.5, seed=2)]
    return dict(frames=fr, table=table, configs=configs, truth=truth, levelsup=2, voc=synth.synth_vocabulary(10, 3, 21))


def crafted_large(kp_dtype, N: int = 2000, n_levels: int = 8, seed: int = 1, param_seeds=(0, 0, 0)) -> dict:
    """record sets at the benchmark's frame size that reach the verifier's block structure -> the dict of crafted() (no truth).

    Scene A: a query of N features (1400 landmarks, five of them twice, 595 distractors) and ten candidates of
    0 / 255 / 256 / 257 / 512 / 513 / N features, and three whose rotation check keeps 256 and 257 of 296 and 297 kept rows
    (bins 10, 15 and 20 tie behind bin 0: bin 20 is dropped) or whose depths leave 256 and 257 correspondences.  With
    levelsup 2 the FeatureVector node is one of the root's 10 children, so a row's candidates span several 32-lane chunks,
    and the landmark copies differ by 3 bits from their originals.  Angles are multiples of 0.5 degrees, so angle
    differences fall on bin edges; a few lie 2^-24 and 0.5 degrees below 360.
    Scene R: eight queries of 200 features, each with six candidates of 25-40 % inliers in shuffled slots (accepted at a
    hypothesis spread over many rounds of eight), one with exactly min_inliers = 20 inliers of 60 (never accepted: the
    maxima tie across rounds), one with 20 inliers of 150 (runs to max_iterations), and itself.
    configs: max_iterations 300, 157 and 299 (ratio 1.0: the rows whose two best distances tie are kept), seeds param_seeds."""
    voc = synth.synth_vocabulary(10, 3, 21)
    B = _Builder(seed, kp_dtype, N, n_levels, voc=voc, levelsup=2)
    rows = []
    Rc, tc = rot([0.2, 1, 0.1], 8.0), np.array([0.25, -0.05, 0.1])

    def lms(n):
        L = B.box(n)
        for lm in L:
            lm["a"] = round(2.0 * lm["a"]) / 2.0
            while B.node(lm["d"]) < 0:  # a stopped word has no FeatureVector entry
                lm["d"] = B.rng.integers(0, 256, 32, dtype=np.uint8)
        return L

    def cand(L, **kw):
        return B.frame(L, Rc, tc, flip=3, **kw)

    # scene A
    LA = lms(1400)
    for lm in LA[5:10]:
        lm["a"] = 0.5
    qa = B.frame(LA + LA[:5], no_depth=set(range(1300, 1310)), extra=N - 1405)
    empty = B.frame([], extra=0)
    sizes = [cand(LA[10 : 10 + n], extra=0) for n in (255, 256, 257, 512, 513)]
    edge = {i: 2.0**-24 for i in (5, 6, 7)} | {8: 0.5, 9: 0.5}
    full = cand(LA, extra=N - 1400, turn=edge, no_depth=set(range(1200, 1260)))

    def tied(main, no_depth=()):
        g = {main + i: -120.0 for i in range(40)} | {main + 40 + i: -180.0 for i in range(40)} | {main + 80 + i: -240.0 for i in range(40)}
        return cand(LA[10 : 10 + main + 120], extra=0, turn=g, no_depth=no_depth)

    rows.append((qa, [empty] + sizes + [full, tied(176), tied(177, no_depth={0}), cand(LA[10:310], extra=0, no_depth=set(range(43)))]))
    # scene R
    for _ in range(8):
        L = lms(160)
        q = B.frame(L, extra=40)
        cs = []
        for _ in range(6):
            n_in = int(B.rng.integers(26, 41))
            n = min(int(B.rng.integers(int(n_in / 0.4), int(n_in / 0.25) + 1)), 120)
            cs.append(cand(L[:n], spin=12.0, wrong=set(B.rng.choice(n, n - n_in, replace=False).tolist())))
        cs.append(cand(L[:60], spin=12.0, wrong=set(range(20, 60))))
        cs.append(cand(L[:150], spin=12.0, wrong=set(range(20, 150))))
        order = B.rng.permutation(len(cs))
        rows.append((q, [cs[i] for i in order] + [q, -1]))
    fr = B.arrays()
    F = len(fr["n"])
    table = np.full((F, 10), -1, np.int32)
    for q, cands in rows:
        table[q, : len(cands)] = cands
    table[empty, :2] = [qa, sizes[0]]  # a query without features
    s0, s1, s2 = param_seeds
    configs = [params(seed=s0), params(max_iterations=157, seed=s1), params(ratio=1.0, max_iterations=299, seed=s2)]
    return dict(frames=fr, table=table, configs=configs, levelsup=2, voc=voc)


def to_records(ctx, fr: dict) -> np.ndarray:
    """the frames as orbx_record_layout records of ctx (left keypoints, descriptors and depth; the rest zero)"""
    rec = np.zeros(len(fr["n"]), ctx.record_dtype())
    rec["n_left"], rec["kps_left"], rec["desc_left"], rec["depth"] = fr["n"], fr["kps"], fr["desc"], fr["depth"]
    return rec
