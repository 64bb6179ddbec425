"""Build and query cost of the keyframe database (orbx_bowdb_*) on bench.py's workload: the F-frame KITTI-shaped stereo
sequence (1241x376, 2000 features, 8 levels x1.2; frame f = synthetic pair f mod --pool, as bench.py builds it) through
orbx_sequence_stereo, a device vocabulary of ORBvoc.txt's shape (k = 10, L = 6) from gathered_desc / gathered_n, then the
database from the same arrays and loop candidates for every frame.  Prints one JSON line:
  build_ms (host clock around the call, which blocks), query_ms for all F frames (CUDA events around the device-output
  query, best of --repeats after a warm-up), queries per second, the mean n_sharing / n_scored, whether every frame's top 10
  are the 10 lowest-id copies of its pair outside the window (all with one score), the GPU's name and power limit (read in
  the same run), and oracle_bowdb_query (tests/bowdb_oracle.c, one host core) against the device for the first
  --oracle-frames queries over the whole database: equality and the oracle's time.

    python scripts/bowdb_query.py [--frames 4541] [--pool 256] [--window 50] [--top-k 10] [--repeats 5] [--oracle-frames 256]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--pool", type=int, default=256)
    ap.add_argument("--window", type=int, default=50)
    ap.add_argument("--top-k", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--oracle-frames", type=int, default=256)
    args = ap.parse_args()

    import torch

    from oracle import oracle_py as O
    from orb_slam2_ros2_b200 import api, synth

    import bowdb_restatement as R

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the device database")
    ident = gpu_identity()
    c = synth.KITTI
    H, W, F, P, K, win = c["height"], c["width"], args.frames, args.pool, args.top_k, args.window
    ctx = api.Context(W, H, 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=64)
    N = ctx.n_features
    pool_l, pool_r = synth.synth_stereo_pool(H, W, P, seed0=0)
    idx = np.arange(F) % P
    d_left = torch.from_numpy(np.ascontiguousarray(pool_l[idx])).cuda()
    d_right = torch.from_numpy(np.ascontiguousarray(pool_r[idx])).cuda()
    torch.cuda.synchronize()
    res = ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, W * H, None, True)
    del d_left, d_right
    V = api.Vocabulary.build(ctx, res.gathered_desc, res.gathered_n, n_frames=F, stride=N, k=10, L=6, seed=0)

    def build():
        t = time.perf_counter()
        D = api.BowDatabase.build(ctx, V, res.gathered_desc, res.gathered_n, n_frames=F, stride=N)
        return D, (time.perf_counter() - t) * 1e3

    build()[0].close()  # warm-up: module load, allocations
    builds = []
    for _ in range(3):
        D, ms = build()
        builds.append(ms)
        D.close()
    D, _ = build()
    info = D.info()

    out = {k: torch.zeros((F, K) if k.startswith("cand") else (F,), dtype=torch.float32 if k == "cand_score" else torch.int32, device="cuda")
           for k in api.BOWDB_OUTPUTS}
    ptrs = [out[k].data_ptr() for k in api.BOWDB_OUTPUTS]
    s = torch.cuda.Stream()
    ctx.set_stream(s.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.query_ptr(0, F, K, win, 0.0, ptrs)  # warm-up
    times = []
    for _ in range(args.repeats):
        e0.record(s)
        D.query_ptr(0, F, K, win, 0.0, ptrs)
        e1.record(s)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ctx.set_stream(None)
    got = {k: v.cpu().numpy() for k, v in out.items()}
    best = min(times)

    # every frame: its top K are the K lowest-id copies of its pair outside the window, with one score
    copies_ok = True
    for f in range(F):
        exp = [g for g in range(f % P, F, P) if abs(g - f) > win][:K]
        row = got["cand_frame"][f]
        if list(row[: len(exp)]) != exp or len(set(got["cand_score"][f][: len(exp)].tolist())) > 1:
            copies_ok = False
            break

    # oracle (one host core) against the device: the first --oracle-frames queries over the whole database
    Fo = min(args.oracle_frames, F)
    gd = ctx.read_device(res.gathered_desc, (F, N, 32), np.uint8)
    gn = ctx.read_device(res.gathered_n, (F,), np.int32)
    a, i = V.arrays(), V.info()
    OV = O.Vocabulary(i["k"], i["L"], a["parent"], a["is_leaf"], a["desc"], a["weight"])
    t = time.perf_counter()
    db = R.bow_arrays(O, OV, gd, gn)
    transform_ms = (time.perf_counter() - t) * 1e3
    t = time.perf_counter()
    exp = R.oracle_query(db, {k: db[k][:Fo] for k in ("ids", "vals", "n")}, 0, win, 0.0, K)
    oracle_ms = (time.perf_counter() - t) * 1e3
    equal = all(np.array_equal(got[k][:Fo].view(np.uint32) if k == "cand_score" else got[k][:Fo],
                               exp[k].view(np.uint32) if k == "cand_score" else exp[k]) for k in api.BOWDB_OUTPUTS)

    print(json.dumps(dict(
        workload=f"loop candidates of every frame of a {F}-frame KITTI-shaped stereo sequence (1241x376, 2000 features; frame f = synthetic pair f mod {P}, "
                 f"as bench.py) against all of them, window {win}, top_k {K}, min_score 0; vocabulary k=10, L=6 built on the device from the same descriptors",
        **ident, frames=F, n_words=info["n_words"], n_postings=info["n_postings"],
        build_ms=round(min(builds), 2), build_ms_runs=[round(x, 2) for x in builds],
        query_ms=round(best, 3), query_ms_runs=[round(x, 3) for x in times], queries_per_s=round(F / (best / 1e3)),
        mean_n_sharing=round(float(got["n_sharing"].mean()), 2), mean_n_scored=round(float(got["n_scored"].mean()), 2),
        top_k_are_lowest_copies_with_one_score=copies_ok,
        oracle_subset=dict(queries=Fo, oracle_query_ms_one_core=round(oracle_ms, 1), oracle_transform_ms_one_core=round(transform_ms, 1), equal=equal),
    )))
    D.close()
    V.close()
    ctx.close()


if __name__ == "__main__":
    main()
