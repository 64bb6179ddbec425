"""Cost of the offline map export: orbx_sequence_stereo vs orbx_sequence_stereo_keyframes on bench.py's workload.

    python scripts/sequence_keyframes.py [--frames 4541] [--batch 64] [--pool 256] [--reps 3]

Prints ONE JSON line:
  * device-resident frames/s of both calls, alternated in this process (images, raw records, keyframe records in HBM), and
    their ratio; the vocabulary has ORBvoc.txt's shape (synth.synth_vocabulary(10, 6, ...): k = 10, L = 6), levelsup = 4;
  * mean keyframe record bytes against the stride (orbx_serialized_capacity_bow);
  * per 64 frames (one device batch): CUDA-event times of the bag-of-words transform (descent + assembly) and of the BoW
    serialiser, and the split of the transform into its two kernels from torch.profiler (a separate, traced run);
  * the GPU's name and power limit (nvidia-smi), which belong to every number above.
Needs a CUDA device; there is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from orb_slam2_ros2_b200 import api, synth  # noqa: E402


def gpu_info(index: int) -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    parts = [p.strip() for p in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return dict(zip(("gpu_name", "power_limit", "sm_clock_max"), parts)) if len(parts) == 3 else {"gpu_query_error": q.stderr.strip()}


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--pool", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3, help="timed passes of each call, alternated")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sequence_keyframes.py: no CUDA device")
    c = synth.KITTI
    H, W, N, B, F = c["height"], c["width"], c["n_features"], args.batch, args.frames
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    ctx = api.Context(W, H, N, c["n_levels"], c["scale_factor"], c["ini_th"], c["min_th"], camera=cam, max_batch=B)
    V = api.Vocabulary(ctx, **synth.synth_vocabulary(10, 6, 1))

    pool_l, pool_r = synth.synth_stereo_pool(H, W, args.pool, seed0=0)
    idx = np.arange(F) % args.pool
    d_left, d_right = torch.from_numpy(pool_l[idx]).cuda(), torch.from_numpy(pool_r[idx]).cuda()
    fsz = W * H
    rs, ks = ctx.record_layout().record_bytes, ctx.serialized_capacity_bow()
    d_rec = torch.empty((F, rs), dtype=torch.uint8, device="cuda")
    d_kf = torch.empty((F, ks), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(F, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    def plain():
        ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, fsz, None, True, d_rec.data_ptr(), rs, True)

    def keyframes():
        ctx.sequence_stereo_keyframes_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, fsz, d_kf.data_ptr(), ks, d_sz.data_ptr(), V, 4, 0, True, 0, True, None,
                                          True, d_rec.data_ptr(), rs, True)

    def timed(fn) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        fn()  # returns once every record has landed
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    plain()
    rec_plain = d_rec.clone()
    keyframes()
    torch.cuda.synchronize()
    same_records = bool(torch.equal(rec_plain, d_rec))
    t_plain, t_kf = [], []
    for _ in range(args.reps):
        t_plain.append(timed(plain))
        t_kf.append(timed(keyframes))
    sizes = d_sz.cpu().numpy()

    # per 64 frames: one device batch, then the BoW transform and the BoW serialiser alone, CUDA events over 20 launches each
    nb = min(64, B)
    ctx.stereo_batch_device(nb, d_left.data_ptr(), d_right.data_ptr(), W, fsz)
    out = torch.empty((nb, ks), dtype=torch.uint8, device="cuda")
    osz = torch.empty(nb, dtype=torch.int64, device="cuda")
    reps = 20

    def ev_ms(fn):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps * (64 / nb)

    bow_ms = ev_ms(lambda: ctx.bow_transform_batch_device(V, nb))
    ser_ms = ev_ms(lambda: ctx.serialize_keyframes_bow_device(nb, 0, out.data_ptr(), ks, osz.data_ptr()))
    plain_ser_ms = ev_ms(lambda: ctx.serialize_keyframes_device(nb, 0, out.data_ptr(), ks, osz.data_ptr()))

    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.bow_transform_batch_device(V, nb)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        for key, tag in (("bow_descend", "bow_descend_kernel"), ("bow_assemble", "bow_assemble_kernel")):
            if tag in e.key:
                kern[key] = round(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1000.0 / reps * (64 / nb), 4)

    fps_plain, fps_kf = F / (np.median(t_plain) / 1e3), F / (np.median(t_kf) / 1e3)
    res = dict(
        metric="keyframe_export_throughput_ratio",
        frames=F, batch=B, vocabulary="synth_vocabulary(10, 6, 1): ORBvoc.txt's shape (k=10, L=6)", levelsup=4,
        plain_frames_per_s=round(fps_plain, 1), keyframes_frames_per_s=round(fps_kf, 1), ratio=round(fps_kf / fps_plain, 4),
        plain_ms=[round(t, 2) for t in t_plain], keyframes_ms=[round(t, 2) for t in t_kf],
        raw_records_identical=same_records,
        mean_record_bytes=round(float(sizes.mean()), 1), max_record_bytes=int(sizes.max()), stride=ks,
        per_64_frames_ms=dict(bow_transform_events=round(bow_ms, 4), bow_serialiser_events=round(ser_ms, 4), plain_serialiser_events=round(plain_ser_ms, 4),
                              **{f"{k}_profiler": v for k, v in kern.items()}),
        **gpu_info(torch.cuda.current_device()),
    )
    ctx.set_stream(None)
    V.close()
    ctx.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
