"""Seeded ray-cast stereo sequences of a closed room, for loop verification with known relative poses.

A room is an axis-aligned box 5 m wide, 2 m high and 5 m deep (x right, y down, z forward) whose six walls carry their own
seeded texture (synth.synth_image, 100 texels per metre, sampled bilinearly).  A rectified stereo camera (baseline BL along
its x axis) walks a circle of radius 1.2 m around the room's centre and turns by 360 / n degrees per frame, looking along
its walk, so the last frames come back to the view of the first.  The true loops checked against the truth are the pairs
20 degrees apart across the seam (0.42 m between the cameras): closer pairs move too little for the pose check to mean much.  A second room with other textures, seen from the
same poses, gives the unrelated frames.  X_cam = R_cw (X_world - C) for a camera with centre C.
"""
from __future__ import annotations

import math

import numpy as np

from orb_slam2_ros2_b200 import api, synth

import stereo_scenes

W, H = 640, 480
FX = FY = 600.0
CX, CY = 320.0, 240.0
BL = 0.4
N_FEATURES, N_LEVELS, SCALE = 1000, 8, 1.2
LEVELSUP = 4  # with an L = 4 vocabulary the FeatureVector node is the root: every query feature is a candidate of a row
ROOM = np.array([[-2.5, 2.5], [-1.0, 1.0], [0.0, 5.0]])
CENTRE = np.array([0.0, 0.0, 2.5])
N_LOOP, N_OTHER = 36, 6
LOOP_DEG = 20.0


def _walls(seed: int) -> list:
    """textures of the walls x-, x+, y-, y+, z-, z+ (100 texels per metre along the two in-plane axes)"""
    dims = [(2, 5), (2, 5), (5, 5), (5, 5), (2, 5), (2, 5)]  # (first, second) in-plane extent in metres
    return [synth.synth_image(int(a * 100) + 2, int(b * 100) + 2, seed * 10 + i).astype(np.float32) for i, (a, b) in enumerate(dims)]


def pose(i: int, n: int = N_LOOP):
    """-> (R_cw, C) of frame i of an n-frame walk: on a circle of radius 1.2 m, looking along it (the walls are seen at a
    slant, so the depth varies across the view and the pose is well conditioned)"""
    th = 2 * math.pi * i / n
    C = CENTRE + 1.2 * np.array([math.sin(th), 0.0, math.cos(th)])
    th += math.pi / 2
    fwd = np.array([math.sin(th), 0.0, math.cos(th)])
    right = np.array([math.cos(th), 0.0, -math.sin(th)])  # x axis; y stays world y (down)
    R_wc = np.stack([right, [0.0, 1.0, 0.0], fwd], 1)
    return R_wc.T, C


def render(walls: list, R_cw: np.ndarray, C: np.ndarray) -> np.ndarray:
    """one 8-bit view: every pixel centre's ray from C hits the box from inside"""
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    d = np.stack([(u - CX) / FX, (v - CY) / FY, np.ones_like(u)], -1) @ R_cw  # world directions R_wc d, as rows
    t_best = np.full(u.shape, np.inf)
    img = np.zeros(u.shape, np.float32)
    hit_axis = np.full(u.shape, -1)
    for ax in range(3):
        for side in range(2):
            with np.errstate(divide="ignore", invalid="ignore"):
                t = (ROOM[ax, side] - C[ax]) / d[..., ax]
            ok = (t > 0) & (t < t_best)
            t_best = np.where(ok, t, t_best)
            hit_axis = np.where(ok, 2 * ax + side, hit_axis)
    P = C + d * t_best[..., None]
    planes = {0: (1, 2), 1: (0, 2), 2: (1, 0)}  # in-plane axes of the walls normal to x, y, z
    for wall in range(6):
        m = hit_axis == wall
        if not m.any():
            continue
        a, b = planes[wall // 2]
        ta = (P[..., a][m] - ROOM[a, 0]) * 100.0
        tb = (P[..., b][m] - ROOM[b, 0]) * 100.0
        img[m] = stereo_scenes._bilinear(walls[wall], tb, ta)
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def stereo(walls, R_cw, C):
    R_wc = R_cw.T
    return render(walls, R_cw, C), render(walls, R_cw, C + R_wc[:, 0] * BL)


def relative_pose(seq: dict, q: int, c: int):
    """ground truth T (candidate camera -> query camera): X_q = R X_c + t"""
    (Rq, Cq), (Rc, Cc) = seq["poses"][q], seq["poses"][c]
    return Rq @ Rc.T, Rq @ (Cc - Cq)


def is_loop(seq: dict, q: int, c: int) -> bool:
    if seq["room"][q] != seq["room"][c] or q == c:
        return False
    dyaw = abs(((seq["yaw"][q] - seq["yaw"][c]) + 180.0) % 360.0 - 180.0)
    return abs(dyaw - LOOP_DEG) < 1.0 and abs(q - c) > 4


def context(max_batch: int = 1) -> api.Context:
    return api.Context(W, H, N_FEATURES, N_LEVELS, SCALE, camera=api.Camera(FX, FY, CX, CY, BL), max_batch=max_batch)


def loop_sequence(oracle, with_images: bool = False, seed: int = 1) -> dict:
    """N_LOOP frames of room A around the loop, then N_OTHER frames of room B.  Without images: the oracle's extraction and
    stereo depth of every frame, a synthetic vocabulary, and a table of true loops and unrelated pairs (truth / unrelated)."""
    walls_a, walls_b = _walls(seed), _walls(seed + 50)
    poses, rooms, yaws, lefts, rights = [], [], [], [], []
    for i in range(N_LOOP + N_OTHER):
        j = i if i < N_LOOP else (i - N_LOOP) * (N_LOOP // N_OTHER)
        R_cw, C = pose(j)
        l, r = stereo(walls_a if i < N_LOOP else walls_b, R_cw, C)
        poses.append((R_cw, C)), rooms.append(0 if i < N_LOOP else 1), yaws.append(360.0 * j / N_LOOP), lefts.append(l), rights.append(r)
    seq = dict(poses=poses, room=rooms, yaw=yaws, left=np.stack(lefts), right=np.stack(rights))
    if with_images:
        return seq
    F = len(lefts)
    kps = np.zeros((F, N_FEATURES), oracle.KP_DTYPE)
    desc = np.zeros((F, N_FEATURES, 32), np.uint8)
    depth = np.full((F, N_FEATURES), -1.0)
    n = np.zeros(F, np.int32)
    bf = float(np.float32(FX) * np.float32(BL))
    for f in range(F):
        L = oracle.extract(lefts[f], N_FEATURES, N_LEVELS, SCALE)
        Rr = oracle.extract(rights[f], N_FEATURES, N_LEVELS, SCALE)
        _, _, dp, _ = oracle.search_by_stereo(L, Rr, FX, bf)
        m = len(L.kps)
        kps[f, :m], desc[f, :m], depth[f, :m], n[f] = L.kps, L.desc, dp, m
    voc = synth.synth_vocabulary(10, 4, 5)
    seq.update(frames=dict(kps=kps, desc=desc, depth=depth, n=n), O=oracle.Vocabulary(**voc), voc=voc, levelsup=LEVELSUP,
               cam=(FX, FY, CX, CY), sf=oracle.scale_factors(SCALE, N_LEVELS))
    # rows: query q with its true loop candidates first, then frames of the other room
    table = np.full((F, 4), -1, np.int32)
    truth, unrelated = {}, []
    for q in list(range(3)) + list(range(N_LOOP - 2, N_LOOP)):
        loops = [c for c in range(N_LOOP) if is_loop(seq, q, c)][:2]
        others = [N_LOOP + (q % N_OTHER), N_LOOP + ((q + 1) % N_OTHER)]
        table[q, : len(loops)] = loops
        table[q, 2:] = others
        for sl, c in enumerate(loops):
            truth[(q, sl)] = relative_pose(seq, q, c)
        unrelated += [(q, 2), (q, 3)]
    seq.update(table=table, truth=truth, unrelated=unrelated)
    return seq
