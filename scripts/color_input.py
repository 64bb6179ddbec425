"""Colour input (orbx_set_input_format) against gray on the benchmark's KITTI shape, all in one process, formats alternating.

    python scripts/color_input.py [--frames 4541] [--rounds 3] [--out FILE]

For gray, BGR8 and BGRA8:
  * pyramid_level0 ms of one 64-frame batch (orbx_profile_stereo_batch_device, median of 10);
  * sequence_stereo frames/s over the sequence with inputs and records in HBM (bench.py's `value` path);
  * frames/s of the sequence from pinned host memory (records back to pinned memory), next to the bare H2D copy ceiling of
    the same input bytes: colour moves 3 or 4 times the bytes over PCIe, so this path is expected to be slower;
  * single-pair host-to-host p50 through the library, and for colour also cv2.cvtColor x 2 followed by the gray call.
Prints one JSON line (card name and power limit included) and writes it to --out.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from orb_slam2_ros2_b200 import api, synth  # noqa: E402

C = synth.KITTI
H, W, N = C["height"], C["width"], C["n_features"]
FMTS = {"gray": api.FORMAT_GRAY8, "bgr8": api.FORMAT_BGR8, "bgra8": api.FORMAT_BGRA8}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def pool(n):
    """n colour pairs (BGR): each channel is the synth stereo recipe with its own seed, one common disparity"""
    ls, rs = [], []
    for i in range(n):
        ch = [synth.synth_stereo_pair(H, W, 1000 + i + 101 * c, 17) for c in range(3)]
        ls.append(np.stack([c[0] for c in ch], -1))
        rs.append(np.stack([c[1] for c in ch], -1))
    return np.stack(ls), np.stack(rs)


def as_format(bgr, name):
    if name == "gray":
        return np.stack([cv2.cvtColor(x, cv2.COLOR_BGR2GRAY) for x in bgr])
    if name == "bgr8":
        return bgr
    alpha = np.random.default_rng(5).integers(0, 256, bgr.shape[:-1] + (1,), dtype=np.uint8)
    return np.concatenate([bgr, alpha], -1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--host-frames", type=int, default=512)
    ap.add_argument("--pool", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("color_input.py: no CUDA device")
    cv2.setNumThreads(1)
    F, Fh, P, B = args.frames, args.host_frames, args.pool, 64
    cam = api.Camera(C["fx"], C["fy"], C["cx"], C["cy"], C["bl"])
    bl, br = pool(P)
    idx = torch.from_numpy(np.arange(F) % P).cuda()
    hidx = np.arange(Fh) % P
    data = {}
    for name, fmt in FMTS.items():
        pl, pr = as_format(bl, name), as_format(br, name)
        dl, dr = torch.from_numpy(pl).cuda()[idx], torch.from_numpy(pr).cuda()[idx]
        hl = torch.empty((Fh,) + pl.shape[1:], dtype=torch.uint8, pin_memory=True)
        hr = torch.empty_like(hl, pin_memory=True)
        np.take(pl, hidx, axis=0, out=hl.numpy())
        np.take(pr, hidx, axis=0, out=hr.numpy())
        ctx = api.Context(W, H, N, C["n_levels"], C["scale_factor"], camera=cam, max_batch=B)
        one = api.Context(W, H, N, C["n_levels"], C["scale_factor"], camera=cam, max_batch=1)
        ctx.set_input_format(fmt)
        one.set_input_format(fmt)
        data[name] = dict(pl=pl, pr=pr, dl=dl, dr=dr, hl=hl, hr=hr, ctx=ctx, one=one, row=W * api.FORMAT_BPP[fmt])
    gray_one = data["gray"]["one"]
    rs = data["gray"]["ctx"].record_layout().record_bytes
    d_rec = torch.empty((F, rs), dtype=torch.uint8, device="cuda")
    h_rec = torch.empty((Fh, rs), dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    res = {k: dict(level0_ms=[], seq_fps=[], e2e_fps=[], copy_fps=[], pair_p50_ms=[], cvt_pair_p50_ms=[]) for k in FMTS}

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t

    for rnd in range(args.rounds + 1):  # round 0 warms every path up and is not reported
        for name, d in data.items():
            ctx, row = d["ctx"], d["row"]
            fs = row * H
            lv = sorted(ctx.profile_stereo_batch_device(B, d["dl"].data_ptr(), d["dr"].data_ptr(), row, fs)["pyramid_level0"] for _ in range(10))
            t_seq = timed(lambda: ctx.sequence_stereo_ptr(F, d["dl"].data_ptr(), d["dr"].data_ptr(), row, fs, None, True, d_rec.data_ptr(), rs, True))
            t_e2e = timed(lambda: ctx.sequence_stereo_ptr(Fh, d["hl"].data_ptr(), d["hr"].data_ptr(), row, fs, None, False, h_rec.data_ptr(), rs, False))
            sl, sr = torch.empty_like(d["hl"], device="cuda"), torch.empty_like(d["hr"], device="cuda")
            t_copy = timed(lambda: (sl.copy_(d["hl"], non_blocking=True), sr.copy_(d["hr"], non_blocking=True)))
            del sl, sr
            lat, cvt = [], []
            for i in range(args.pairs):
                l, r = d["pl"][i % P], d["pr"][i % P]
                t = time.perf_counter()
                d["one"].stereo_frame(l, r)
                lat.append(time.perf_counter() - t)
                if name != "gray":
                    code = cv2.COLOR_BGR2GRAY if name == "bgr8" else cv2.COLOR_BGRA2GRAY
                    t = time.perf_counter()
                    gray_one.stereo_frame(cv2.cvtColor(l, code), cv2.cvtColor(r, code))
                    cvt.append(time.perf_counter() - t)
            if rnd == 0:
                continue
            r_ = res[name]
            r_["level0_ms"].append(lv[len(lv) // 2])
            r_["seq_fps"].append(F / t_seq)
            r_["e2e_fps"].append(Fh / t_e2e)
            r_["copy_fps"].append(Fh / t_copy)
            r_["pair_p50_ms"].append(1e3 * float(np.median(lat)))
            if cvt:
                r_["cvt_pair_p50_ms"].append(1e3 * float(np.median(cvt)))
    out = dict(script="color_input", card=card(), frames=F, host_frames=Fh, batch=B, shape=[W, H], rounds=args.rounds,
               results={k: {m: [round(x, 4) for x in v] for m, v in r.items() if v} for k, r in res.items()})
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    for d in data.values():
        d["ctx"].close()
        d["one"].close()


if __name__ == "__main__":
    main()
