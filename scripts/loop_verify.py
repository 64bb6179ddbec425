"""Cost of loop verification (orbx_loopver_*) on two workloads, each through the whole device pipeline: orbx_sequence_stereo
with the records on the device, a device vocabulary from gathered_desc / gathered_n, the keyframe database, query_range for
every frame (top_k candidates outside the window) into a device table, then the verifier on that table.

  kitti   bench.py's F-frame KITTI-shaped sequence (1241x376, 2000 features, 8 levels; frame f = synthetic pair f mod --pool),
          vocabulary k = 10, L = 6, levelsup 4, window 50, top_k 10.  Every candidate is an exact copy of its query's pair: the
          matching-bound case (every pair is accepted at its first hypothesis).
  loop    a rendered loop of --loop-frames frames (tests/loop_scenes.py, 640x480, 1000 features), vocabulary k = 10, L = 4, window
          --loop-window, top_k 10: the candidates overlap their query only partly, so fewer pairs are accepted and more
          hypotheses run than on the copies.  It is not RANSAC-bound: on a B200 its pairs averaged 2.8 hypotheses.

Prints one JSON line: the GPU's name and power limit (read in the same run) and, per workload, build_ms (host clock around
the blocking call, best of 3 after a warm-up), verify_ms (CUDA events around the device-table, device-output call, best of
--repeats after a warm-up), pairs/s, the mean n_matches / n_corr / n_iters over the non-empty pairs, the accepted pairs and
the queries with a loop_frame, and oracle_loopver (tests/loopver_oracle.c, one host core) against the device on the first
--oracle-queries queries: equality of every output (T as bits) and the oracle's time.

    python scripts/loop_verify.py [--frames 4541] [--pool 256] [--loop-frames 300] [--loop-window 25] [--repeats 5] [--oracle-queries 8]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from vocab_build import gpu_identity  # noqa: E402  (scripts/vocab_build.py)


def run(torch, O, api, R, ctx, d_left, d_right, F, k, L, levelsup, window, top_k, repeats, oracle_queries, seed=0):
    N, lay = ctx.n_features, ctx.record_layout()
    d_rec = torch.zeros((F, lay.record_bytes), dtype=torch.uint8, device="cuda")
    H, W = ctx.height, ctx.width
    res = ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, W * H, None, True, d_rec.data_ptr(), lay.record_bytes, True)
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=k, L=L, seed=seed)
    D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=N)
    cand = torch.zeros((F, top_k), dtype=torch.int32, device="cuda")
    D.query_ptr(0, F, top_k, window, 0.0, [cand.data_ptr()] + [0] * 6)
    ctx.synchronize()

    def build():
        t = time.perf_counter()
        LV = api.LoopVerifier.build(ctx, V, d_rec.data_ptr(), F, levelsup=levelsup)
        return LV, (time.perf_counter() - t) * 1e3

    build()[0].close()  # warm-up: module load, allocations
    builds = []
    for _ in range(3):
        LV, ms = build()
        builds.append(ms)
        LV.close()
    LV, _ = build()
    out = {n: torch.zeros((F, top_k), dtype=torch.int32, device="cuda") for n in api.LOOPVER_OUTPUTS[:7]}
    out.update(T=torch.zeros((F, top_k, 12), dtype=torch.float64, device="cuda"), match=torch.zeros((F, top_k, N), dtype=torch.int32, device="cuda"),
               loop_frame=torch.zeros(F, dtype=torch.int32, device="cuda"))
    ptrs = [out[n].data_ptr() for n in api.LOOPVER_OUTPUTS]
    s = torch.cuda.Stream()
    ctx.set_stream(s.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    LV.verify_ptr(0, F, cand.data_ptr(), top_k, ptrs, seed=seed)  # warm-up
    times = []
    for _ in range(repeats):
        e0.record(s)
        LV.verify_ptr(0, F, cand.data_ptr(), top_k, ptrs, seed=seed)
        e1.record(s)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ctx.set_stream(None)
    got = {n: v.cpu().numpy() for n, v in out.items()}
    table = cand.cpu().numpy()
    best = min(times)
    live = table >= 0

    # oracle (one host core) against the device on the first queries: only the frames they use are read back
    Q = min(oracle_queries, F)
    used = sorted(set(range(Q)) | {int(g) for g in table[:Q].ravel() if g >= 0})
    rec = np.zeros(F, ctx.record_dtype())
    rec[used] = d_rec[torch.tensor(used, device="cuda")].cpu().numpy().view(ctx.record_dtype()).reshape(len(used))
    fr = dict(kps=rec["kps_left"], desc=rec["desc_left"], depth=rec["depth"], n=rec["n_left"])
    a, i = V.arrays(), V.info()
    OV = O.Vocabulary(i["k"], i["L"], a["parent"], a["is_leaf"], a["desc"], a["weight"])
    cam = (ctx.camera.fx, ctx.camera.fy, ctx.camera.cx, ctx.camera.cy)
    t = time.perf_counter()
    exp = R.oracle_verify(OV, levelsup, fr, cam, ctx.scaled_factors(), 0, table[:Q], R.params(seed=seed))
    oracle_ms = (time.perf_counter() - t) * 1e3
    equal = all(np.array_equal(got[n][:Q].view(np.uint64) if n == "T" else got[n][:Q], exp[n].view(np.uint64) if n == "T" else exp[n])
                for n in api.LOOPVER_OUTPUTS)
    r = dict(frames=F, pairs=int(live.sum()), build_ms=round(min(builds), 2), build_ms_runs=[round(x, 2) for x in builds], verify_ms=round(best, 3),
             verify_ms_runs=[round(x, 3) for x in times], pairs_per_s=round(int(live.sum()) / (best / 1e3)),
             mean_n_matches=round(float(got["n_matches"][live].mean()), 2), mean_n_corr=round(float(got["n_corr"][live].mean()), 2),
             mean_n_iters=round(float(got["n_iters"][live].mean()), 2), accepted=int(got["accepted"].sum()),
             queries_with_loop_frame=int((got["loop_frame"] >= 0).sum()),
             oracle_subset=dict(queries=Q, pairs=int(live[:Q].sum()), oracle_ms_one_core=round(oracle_ms, 1), equal=equal))
    for o in (LV, D, V):
        o.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--pool", type=int, default=256)
    ap.add_argument("--loop-frames", type=int, default=300)
    ap.add_argument("--loop-window", type=int, default=25)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--oracle-queries", type=int, default=8)
    args = ap.parse_args()

    import torch

    from oracle import oracle_py as O
    from orb_slam2_ros2_b200 import api, synth

    import loop_scenes as S
    import loopver_restatement as R

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the device verifier")
    ident = gpu_identity()
    out = dict(**ident)

    c = synth.KITTI
    H, W, F, P = c["height"], c["width"], args.frames, args.pool
    ctx = api.Context(W, H, 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=64)
    pool_l, pool_r = synth.synth_stereo_pool(H, W, P, seed0=0)
    idx = np.arange(F) % P
    d_left = torch.from_numpy(np.ascontiguousarray(pool_l[idx])).cuda()
    d_right = torch.from_numpy(np.ascontiguousarray(pool_r[idx])).cuda()
    torch.cuda.synchronize()
    out["kitti"] = dict(workload=f"{F}-frame KITTI-shaped stereo sequence (frame f = synthetic pair f mod {P}, as bench.py), vocabulary k=10 L=6, "
                                 f"levelsup 4, window 50, top_k 10", **run(torch, O, api, R, ctx, d_left, d_right, F, 10, 6, 4, 50, 10, args.repeats,
                                                                            args.oracle_queries))
    del d_left, d_right
    ctx.close()

    n = args.loop_frames
    walls = S._walls(1)
    lefts, rights = zip(*(S.stereo(walls, *S.pose(i, n)) for i in range(n)))
    ctx = S.context(max_batch=16)
    d_left = torch.from_numpy(np.ascontiguousarray(np.stack(lefts))).cuda()
    d_right = torch.from_numpy(np.ascontiguousarray(np.stack(rights))).cuda()
    torch.cuda.synchronize()
    out["loop"] = dict(workload=f"rendered {n}-frame loop in a 5 m room (640x480, 1000 features), vocabulary k=10 L=4, levelsup {S.LEVELSUP}, "
                                f"window {args.loop_window}, top_k 10", **run(torch, O, api, R, ctx, d_left, d_right, n, 10, 4, S.LEVELSUP,
                                                                               args.loop_window, 10, args.repeats, args.oracle_queries))
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
