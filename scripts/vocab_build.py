"""Build time of a bag-of-words vocabulary on the device (orbx_vocab_build) from the gathered descriptors of bench.py's
workload: the F-frame KITTI-shaped stereo sequence (1241x376, 2000 features, 8 levels x1.2; frame f = synthetic pair f mod
--pool, as bench.py builds it) through orbx_sequence_stereo, then a vocabulary of ORBvoc.txt's shape (k = 10, L = 6) from
gathered_desc / gathered_n.  Prints one JSON line:
  build_ms (host clock around the call, which blocks), level_ms / idf_ms (CUDA events inside it), iterations per level,
  capped nodes, training descriptors per second, the tree's size, the GPU's name and power limit (read in the same run), and
  oracle_vocab_build (the plain-C checker in tests/vocab_build_oracle.c, one host core) against the same device build on the
  first --oracle-frames frames: both times and whether the trees are equal.

    python scripts/vocab_build.py [--frames 4541] [--pool 256] [--k 10] [--L 6] [--repeats 3] [--oracle-frames 64]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_identity() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--pool", type=int, default=256)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--L", type=int, default=6)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--oracle-frames", type=int, default=64)
    args = ap.parse_args()

    import torch

    from orb_slam2_ros2_b200 import api, synth

    import vocab_build_restatement as R

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the device build")
    ident = gpu_identity()
    c = synth.KITTI
    H, W, F, P = c["height"], c["width"], args.frames, args.pool
    ctx = api.Context(W, H, 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=64)
    N = ctx.n_features
    pool_l, pool_r = synth.synth_stereo_pool(H, W, P, seed0=0)
    idx = np.arange(F) % P
    d_left = torch.from_numpy(np.ascontiguousarray(pool_l[idx])).cuda()
    d_right = torch.from_numpy(np.ascontiguousarray(pool_r[idx])).cuda()
    torch.cuda.synchronize()
    res = ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, W * H, None, True)
    del d_left, d_right
    gn = ctx.read_device(res.gathered_n, (F,), np.int32)
    n_desc = int(gn.sum())

    def build(desc, counts, n_frames):
        st = {}
        t = time.perf_counter()
        V = api.Vocabulary.build(ctx, desc, counts, n_frames=n_frames, stride=N, k=args.k, L=args.L, seed=args.seed, stats=st)
        return V, (time.perf_counter() - t) * 1e3, st

    V, _, _ = build(res.gathered_desc, res.gathered_n, F)  # warm-up: module load, allocations
    info = V.info()
    V.close()
    runs = []
    for _ in range(args.repeats):
        V, ms, st = build(res.gathered_desc, res.gathered_n, F)
        runs.append((ms, st))
        V.close()
    ms_all = [r[0] for r in runs]
    best_ms, st = min(runs, key=lambda r: r[0])

    # oracle on a subset (host, one core) vs the device on the same subset
    Fo = min(args.oracle_frames, F)
    gd = ctx.read_device(res.gathered_desc, (Fo, N, 32), np.uint8)
    t = time.perf_counter()
    orc = R.oracle_vocab_build(gd, gn[:Fo], Fo, args.k, args.L, args.seed)
    oracle_ms = (time.perf_counter() - t) * 1e3
    Vs, sub_ms, _ = build(gd, gn[:Fo], Fo)
    got = Vs.arrays()
    equal = all(np.array_equal(got[f], orc[f]) for f in ("parent", "is_leaf", "desc", "weight"))
    Vs.close()

    print(json.dumps(dict(
        workload=f"gathered left descriptors of a {F}-frame KITTI-shaped stereo sequence (1241x376, 2000 features; frame f = synthetic pair f mod {P}, "
                 f"as bench.py), k={args.k}, L={args.L}, seed={args.seed}",
        **ident, frames=F, training_descriptors=n_desc, n_nodes=info["n_nodes"], n_words=info["n_words"],
        build_ms=round(best_ms, 2), build_ms_runs=[round(x, 2) for x in ms_all],
        level_ms=[round(x, 3) for x in st["level_ms"][: args.L]], idf_ms=round(st["level_ms"][args.L], 3), iters_per_level=st["iters"],
        capped_nodes=st["n_capped"], descriptors_per_s=round(n_desc / (best_ms / 1e3)),
        oracle_subset=dict(frames=Fo, descriptors=int(gn[:Fo].sum()), oracle_ms_one_core=round(oracle_ms, 1), device_ms=round(sub_ms, 2), trees_equal=equal),
    )))
    ctx.close()


if __name__ == "__main__":
    main()
