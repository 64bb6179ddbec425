#!/usr/bin/env python
"""bench.py -- stereo frames/s of the ORB front-end (extract L+R + stereo match, 2000 features) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--frames F] [--transport nccl|peer] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (pyramid+blur, FAST, quadtree, orientation+BRIEF, stereo match) over the synthetic
4541-frame KITTI-00-length stereo sequence (BASELINE.json configs[2]; per frame it is configs[0]), sharded by frame over the
N GPUs in contiguous blocks through the library's own sequence entry (orbx_sequence_stereo): strong scaling.  `value` is
whole-job frames/s with every rank's block resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` is
the same call with the block in pinned host memory and the per-frame records landing in pinned host memory (copies inside
the timed region).  The only exchange between ranks is the gather of the left descriptors, issued by the library (NCCL
send/recv pieces on a side stream, or peer-memory stores fused into the record-packing kernel).  The line also carries the
other BASELINE configurations (`configs`: TUM RGB-D, 1080p, the feature-count latency sweep), the roofline of the dominant
kernel, the CPU baseline and a `check` block that verifies the timed work (gathered descriptors against single-frame calls,
checksums across ranks, bit flips against the oracle).

`--impl reference` times the reference's own CPU implementation (oracle/_ref: the reference's ORBExtractor.cc and the
searchByStereo lines of ORBMatcher.cc compiled unmodified) on the host cores of the same box, on a bounded sample of the
same sequence per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from orb_slam2_ros2_b200 import synth  # noqa: E402

METRIC = "stereo frames/s (extract+stereo match, 2000 feats)"
UNIT = "frames/s"
CFG = synth.KITTI


SEQ_FRAMES = 4541  # KITTI odometry sequence 00 (BASELINE.json configs[2])


def workload_config(args):
    c = CFG
    return {
        "workload": f"synthetic {args.frames}-frame KITTI-00-length stereo sequence 1241x376, 2000 features, 8 levels x1.2: ORB extraction (L+R) + stereo "
                    "matching per frame, frames sharded over the GPUs in contiguous blocks of ceil(F/N) (BASELINE.json configs[2] = configs[0] per frame)",
        "frames_per_step": args.frames,
        "pool_pairs": args.pool,
        "frame_source": f"frame f = synthetic pair f mod {args.pool} ({args.pool} distinct pairs, seeds fixed: every rank count sees the same sequence)",
        "l2_policy": f"inputs larger than L2: every rank's block of the sequence is materialised ({args.frames * 2 * c['width'] * c['height'] / 1e9:.2f} GB "
                     "over all ranks, read once per step) and ~370 MB of pyramid intermediates are rewritten per 64 frames",
        "device_slots": args.batch,
        "parallelism": "frame blocks per rank, no data-path collective; left descriptors (+ counts) of all frames gathered on every rank by the library "
                       f"({args.transport}: " + ("grouped ncclSend/ncclRecv of 64-frame pieces on a side stream" if args.transport == "nccl" else
                                                 "stores into every rank's gathered array through CUDA-IPC peer pointers from the record-packing kernel") + ")",
    }


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout=5.0):
        """nvidia-smi needs a moment to attach; block until it has written its first line"""
        t0 = time.time()
        while self.proc and time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return
            except OSError:
                pass
            time.sleep(0.02)

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [q.strip() for q in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------
_ref_pool = {}


def cpu_reference_run(n_frames: int, workers: int, pool_pairs: int = 8):
    """times oracle/_ref (the compiled reference) on `n_frames` stereo frames; returns (fps, cores, kind, sample)"""
    from oracle import oracle_py as O  # the CPU baseline leg is one of the places allowed to execute oracle/

    if pool_pairs not in _ref_pool:
        _ref_pool[pool_pairs] = synth.synth_stereo_pool(CFG["height"], CFG["width"], pool_pairs, seed0=0)  # the first pairs of the sequence
    lefts, rights = _ref_pool[pool_pairs]
    with tempfile.TemporaryDirectory() as td:
        tp = O.write_template_file(os.path.join(td, "brief_template.txt"))
        if O.have_ref():
            O.ref_set_camera(CFG["fx"], CFG["fy"], CFG["cx"], CFG["cy"], CFG["bl"], None)
            secs, _ = O.ref_bench_stereo(lefts, rights, tp, n_frames, workers, CFG["n_features"], CFG["n_levels"], CFG["scale_factor"])
            kind = "reference"
            cores = min(os.cpu_count() or 1, 2 * workers)
        else:  # the reference could not be compiled where this tree was built: time the scalar C port instead
            t0 = time.perf_counter()
            for i in range(n_frames):
                el = O.extract(lefts[i % pool_pairs])
                er = O.extract(rights[i % pool_pairs])
                O.search_by_stereo(el, er, np.float32(CFG["fx"]), np.float32(CFG["fx"]) * np.float32(CFG["bl"]))
            secs = time.perf_counter() - t0
            kind, cores = "port", 1
    sample = (f"{n_frames} frames of the same KITTI-shaped sequence ({pool_pairs} distinct pairs), {workers} frames in flight x the reference's 2 extractor "
              "threads (Frame.cc:100-105); the reference's own ORBExtractor.cc / ORBMatcher.cc compiled unmodified, its three OpenCV primitives "
              "(cv::resize, cv::GaussianBlur, cv::FAST) are scalar restatements -- no C++ OpenCV in this image; a SIMD OpenCV build is ~2x faster on them")
    return n_frames / secs, cores, kind, sample


def opencv_primitives_timing(fps: float, workers: int):
    """How much of the CPU arm is the scalar restatement of the three OpenCV primitives?  Times cv::resize + cv::GaussianBlur +
    cv::FAST of ONE image of the workload (all pyramid levels) twice on one host core: the oracle's scalar C restatements (what
    oracle/_ref links) and cv2's SIMD code (per 30-px cell like the reference: cv::FAST on the cell's sub-matrix, iniTh then minTh
    for empty cells), and turns the difference into an ESTIMATE of the arm with a SIMD OpenCV build (same threads, same frames in
    flight: per-image time = workers / fps)."""
    try:
        import cv2
        from oracle import oracle_py as O
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)}
    img = synth.synth_stereo_pair(CFG["height"], CFG["width"], 0)[0]
    rc, lw, lh = O.level_sizes(CFG["width"], CFG["height"], CFG["scale_factor"], CFG["n_levels"])
    cv2.setNumThreads(1)

    def scalar():
        lv = [img] + [O.resize_linear(img, int(lw[l]), int(lh[l])) for l in range(1, CFG["n_levels"])]
        for a in lv:
            O.gaussian_blur7(a)
            O.fast_cells(a, CFG["ini_th"], CFG["min_th"])

    det = {t: cv2.FastFeatureDetector_create(threshold=t, nonmaxSuppression=True) for t in (CFG["ini_th"], CFG["min_th"])}

    def simd():
        lv = [img] + [cv2.resize(img, (int(lw[l]), int(lh[l])), interpolation=cv2.INTER_LINEAR) for l in range(1, CFG["n_levels"])]
        for a in lv:
            cv2.GaussianBlur(a, (7, 7), 2, 2, borderType=cv2.BORDER_REFLECT_101)
            h, w = a.shape
            bw, bh = w - 32, h - 32  # the 16-px margin of src/ORBExtractor.cc:334-343
            nc, nr = bw // 30, bh // 30
            wc, hc = bw // nc, bh // nr
            for i in range(nr):
                for j in range(nc):
                    y0, x0 = 16 + i * hc, 16 + j * wc
                    cell = a[y0 : min(y0 + hc + 6, h - 16), x0 : min(x0 + wc + 6, w - 16)]
                    if not det[CFG["ini_th"]].detect(cell):
                        det[CFG["min_th"]].detect(cell)

    def best(f, reps=3):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            f()
            ts.append(time.perf_counter() - t0)
        return min(ts)

    t_scalar, t_simd = best(scalar), best(simd)
    t_img = workers / fps  # seconds one extractor thread spends per image in the measured arm
    est = workers / max(t_img - (t_scalar - t_simd), 1e-9) if t_scalar > t_simd else fps
    return {"scalar_ms_per_image": 1e3 * t_scalar, "cv2_simd_ms_per_image": 1e3 * t_simd, "cv2_version": cv2.__version__,
            "estimated_value_with_simd_opencv": est,
            "note": "one host core, min of 3; cv2 timing includes the Python call overhead of ~2.5k cv::FAST calls per image (conservative); the estimate "
                    "replaces the scalar primitives' time inside the measured per-image time, everything else (quadtree, BRIEF, stereo matching: the "
                    "reference's own code) unchanged"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    workers = max(1, ncpu // 2)
    per_step = 64  # a bounded sample of the sequence per step: 64 frames = the GPU arm's device-slot batch
    for _ in range(min(args.warmup, 1)):
        cpu_reference_run(max(workers, 8), workers)
    t0 = time.perf_counter()
    fps_list = []
    kind = cores = sample = None
    for _ in range(args.steps):
        fps, cores, kind, sample = cpu_reference_run(per_step, workers)
        fps_list.append(fps)
    wall = time.perf_counter() - t0
    value = float(args.steps * per_step / sum(per_step / f for f in fps_list))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * per_step / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args),  # identical to the GPU arm's; what a CPU "step" actually ran is in cpu_baseline.sample
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": sample + f"; {per_step} frames per step x {args.steps} steps (ms_per_step is the time of one such sample)",
                         "opencv_primitives": opencv_primitives_timing(value, workers)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
class CudaArray:
    """expose a raw device pointer to torch through __cuda_array_interface__"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def bench_matchers(ctx, api, torch, stream, d_left, d_right, B, W, H, N, fsz, cpu=True, th=15.0, reps=20):
    """ORBMatcher::searchByProjection's inner step (findFeaturesInArea + exclusion + getBestMatch) for N queries per frame
    against the B device-resident frames of one stereo batch: queries = each frame's own keypoints as "seen in the last
    frame" (moved by N(0, 3) px, 6 descriptor bits flipped), 30 % of the frame's keypoints excluded."""
    ctx.set_stream(stream.cuda_stream)
    res = ctx.stereo_batch_device(B, d_left.data_ptr(), d_right.data_ptr(), W, fsz)
    kps = ctx.read_device(res.kps_und, (2 * B, N), api.KP_DTYPE)[0::2]
    desc = ctx.read_device(res.desc, (2 * B, N, 32), np.uint8)[0::2]
    nk = ctx.read_device(res.n_kps, (2 * B,), np.int32)[0::2]
    qs, qds, exs = np.zeros((B, N), api.AREA_QUERY_DTYPE), np.zeros((B, N, 32), np.uint8), np.zeros((B, N), np.uint8)
    for f in range(B):
        q, qd, ex, _ = synth.synth_area_queries(kps[f][: nk[f]], desc[f][: nk[f]], N, 500 + f, W, H, CFG["n_levels"], th)
        qs[f], qds[f], exs[f, : len(ex)] = q, qd, ex
    with torch.cuda.stream(stream):
        t_q = torch.from_numpy(qs.view(np.uint8).reshape(B, -1)).cuda()
        t_d, t_x = torch.from_numpy(qds).cuda(), torch.from_numpy(exs).cuda()
        o = [torch.zeros((B, N), dtype=torch.int32, device="cuda") for _ in range(3)]
        o_ratio = torch.zeros((B, N), dtype=torch.float32, device="cuda")

        def launch():
            ctx.search_in_area_batch_device(B, N, t_q.data_ptr(), t_d.data_ptr(), 0, t_x.data_ptr(), o[0].data_ptr(), o[1].data_ptr(), o_ratio.data_ptr(),
                                            o[2].data_ptr())

        for _ in range(3):
            launch()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        e0.record(stream)
        for _ in range(reps):
            launch()
        e1.record(stream)
        stream.synchronize()
    ms = e0.elapsed_time(e1) / reps
    n_cand = o[2].cpu().numpy()
    accepted = int(((o[0].cpu().numpy() >= 0) & (o[1].cpu().numpy() < 50) & (o_ratio.cpu().numpy() < 0.6)).sum())
    alg = B * N * (24 + 32 + 16) + int(n_cand.sum()) * (32 + 4 + 2)  # queries in, results out, per candidate: descriptor + octave + grid entry
    peak, _ = measured_peaks()
    out = {
        "metric": "area-search queries/s (findFeaturesInArea + getBestMatch, %d queries/frame, th=%g)" % (N, th), "value": B * N / (ms * 1e-3),
        "unit": "queries/s", "kernel": "area_match", "kernel_ms": ms, "frames_per_launch": B, "mean_candidates": float(n_cand.mean()),
        "accepted_per_frame": accepted / B, "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg},
    }
    # result serialisation (SURVEY 8(f) rank 4): one KeyFrameData record per frame, assembled on the device
    cap = ctx.serialized_capacity()
    with torch.cuda.stream(stream):
        rec = torch.zeros((B, cap), dtype=torch.uint8, device="cuda")
        rec_sizes = torch.zeros(B, dtype=torch.int64, device="cuda")
        for _ in range(3):
            ctx.serialize_keyframes_device(B, 1, rec.data_ptr(), cap, rec_sizes.data_ptr())
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        s0.record(stream)
        for _ in range(reps):
            ctx.serialize_keyframes_device(B, 1, rec.data_ptr(), cap, rec_sizes.data_ptr())
        s1.record(stream)
        stream.synchronize()
    ser_ms = s0.elapsed_time(s1) / reps
    ser_bytes = int(rec_sizes.sum().item())
    out["serialize"] = {"metric": "KeyFrameData records/s (proto3 wire format, %d keypoints each)" % N, "value": B / (ser_ms * 1e-3), "unit": "records/s",
                        "kernel": "serialize", "kernel_ms": ser_ms, "bytes_per_record": ser_bytes / B,
                        "roofline": {"bound": "hbm", "achieved": (ser_bytes + B * N * (28 + 32 + 16)) / (ser_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                     "frac": (ser_bytes + B * N * (28 + 32 + 16)) / (ser_ms * 1e-3) / 1e9 / peak}}
    # bag-of-words transform (SURVEY 8(f) rank 3) with a synthetic vocabulary of ORBvoc.txt's shape (k = 10, L = 6, ~1 M nodes)
    voc = synth.synth_vocabulary(10, 6, 0)
    V = api.Vocabulary(ctx, **voc)
    with torch.cuda.stream(stream):
        for _ in range(3):
            ctx.bow_transform_batch_device(V, B, 4)
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        b0.record(stream)
        for _ in range(reps):
            dbow = ctx.bow_transform_batch_device(V, B, 4)
        b1.record(stream)
        stream.synchronize()
    bow_ms = b0.elapsed_time(b1) / reps
    n_words = ctx.read_device(dbow.n_bow, (B,), np.int32)
    vi = V.info()
    # per descriptor: its 32 bytes + L levels x k children x 32-byte node descriptors; per frame: 16 B per BowVector entry + 8 B per feature
    bow_alg = B * N * (32 + 6 * 10 * 32) + int(n_words.sum()) * 12 + B * N * 8
    out["bow"] = {"metric": "frames/s of DBoW3 transform (k=10, L=6 synthetic vocabulary, %d descriptors per frame, levelsup 4)" % N,
                  "value": B / (bow_ms * 1e-3), "unit": "frames/s", "kernels": ["bow_descend", "bow_assemble"], "ms_per_launch_pair": bow_ms,
                  "frames_per_launch": B, "vocabulary_nodes": vi["n_nodes"], "mean_words_per_frame": float(n_words.mean()),
                  "roofline": {"bound": "hbm", "achieved": bow_alg / (bow_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                               "frac": bow_alg / (bow_ms * 1e-3) / 1e9 / peak}, "parity": "unpinned (DBoW3 is un-vendored; oracle = restated published algorithm)"}
    if cpu:
        from oracle import oracle_py as O

        OV = O.Vocabulary(**voc)
        t0 = time.perf_counter()
        for f in range(min(B, 8)):
            O.bow_transform(OV, desc[f][: nk[f]], 4)
        out["bow"]["cpu_baseline"] = {"value": min(B, 8) / (time.perf_counter() - t0), "unit": "frames/s", "cores": 1, "kind": "port",
                                      "sample": "%d frames" % min(B, 8)}
        t0 = time.perf_counter()
        ur = ctx.read_device(res.u_right, (B, N), np.float64)
        dpt = ctx.read_device(res.depth, (B, N), np.float64)
        t0 = time.perf_counter()
        for f in range(min(B, 16)):
            O.serialize_keyframe(kps[f][: nk[f]], desc[f][: nk[f]], ur[f][: nk[f]], dpt[f][: nk[f]], 1 + f, ctx.grid_info()[2:], None, True)
        out["serialize"]["cpu_baseline"] = {"value": min(B, 16) / (time.perf_counter() - t0), "unit": "records/s", "cores": 1, "kind": "port",
                                            "sample": "%d records" % min(B, 16)}
        bounds = ctx.grid_info()[2:]
        sf = ctx.scaled_factors()
        t0 = time.perf_counter()
        nf = min(B, 8)
        for f in range(nf):
            O.search_in_area(kps[f][: nk[f]], desc[f][: nk[f]], bounds, sf, qs[f], qds[f], exs[f][: nk[f]])
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": nf * N / dt, "unit": "queries/s", "cores": 1, "kind": "port", "sample": "%d frames x %d queries (incl. initGrid per frame)" % (nf, N)}
    return out


def _events(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


_pinned_keep = []


def pinned_outputs(torch, n_features):
    """the nine output arrays of orbx_stereo_batch for one frame, in pinned host memory -> their addresses"""
    N = n_features
    t = {"kl": torch.empty((N, 28), dtype=torch.uint8, pin_memory=True), "dl": torch.empty((N, 32), dtype=torch.uint8, pin_memory=True),
         "kr": torch.empty((N, 28), dtype=torch.uint8, pin_memory=True), "dr": torch.empty((N, 32), dtype=torch.uint8, pin_memory=True),
         "ur": torch.empty(N, dtype=torch.float64, pin_memory=True), "dp": torch.empty(N, dtype=torch.float64, pin_memory=True),
         "c": torch.zeros(4, dtype=torch.int32, pin_memory=True)}
    _pinned_keep.append(t)
    c = t["c"].data_ptr()
    return [t["kl"].data_ptr(), t["dl"].data_ptr(), c, t["kr"].data_ptr(), t["dr"].data_ptr(), c + 4, t["ur"].data_ptr(), t["dp"].data_ptr(), c + 8]


def oracle_flip_check(api, O, ctx_result_kps, ctx_result_desc, img, nf, nl, sc):
    """descriptor bit flips / inexact angles of one image against the oracle (north_star: flips "traced ... and counted")"""
    e = O.extract(img, nf, nl, sc)
    n = len(e.kps)
    same = len(ctx_result_kps) == n and all(np.array_equal(ctx_result_kps[f], e.kps[f]) for f in ("x", "y", "size", "response", "octave", "class_id"))
    flips = int(np.unpackbits(ctx_result_desc[:n] ^ e.desc).sum()) if len(ctx_result_desc) >= n else -1
    dang = np.abs(ctx_result_kps["angle"][:n] - e.kps["angle"]) if len(ctx_result_kps) >= n else np.array([1e9])
    dang = np.minimum(dang, 360.0 - dang)
    return {"keypoints": n, "keypoints_bit_exact": bool(same), "descriptor_bit_flips": flips, "inexact_angles": int((dang != 0).sum()),
            "max_angle_error_rad": float(np.radians(dang.max(initial=0.0)))}


def bench_other_configs(args, api, torch, stream, local_rank, with_oracle):
    """BASELINE.json configs[1], [3], [4] on one GPU: TUM-shaped RGB-D throughput, the feature-count latency sweep and the
    1920x1080 / 5000 features / 12 levels stress case -- each with frames/s (or p50 ms), algorithmic bytes, roofline fraction
    and a bit-flip count against the oracle on one frame."""
    peak, _ = measured_peaks()
    O = None
    if with_oracle:
        from oracle import oracle_py as O  # checker only
    out = {}

    def timed_ms(fn, reps):
        for _ in range(3):
            fn()
        e0, e1 = _events(torch)
        stream.synchronize()
        e0.record(stream)
        for i in range(reps):
            fn(i)
        e1.record(stream)
        stream.synchronize()
        return e0.elapsed_time(e1) / reps

    # configs[1]: TUM-shaped RGB-D 640x480, 1000 features, depth lookup path (Frame.cc:125-159)
    c = synth.TUM
    B, P = 64, 128
    g = np.stack([synth.synth_image(c["height"], c["width"], 3000 + i) for i in range(P)])
    d = np.stack([synth.synth_depth_u16(c["height"], c["width"], 3000 + i, c["depth_scale"]) for i in range(P)])
    with torch.cuda.stream(stream):
        dg, dd = torch.from_numpy(g).cuda(), torch.from_numpy(d.view(np.int16)).cuda()
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], tuple(c["dist"]), c["depth_scale"])
    ctx = api.Context(c["width"], c["height"], c["n_features"], c["n_levels"], c["scale_factor"], camera=cam, max_batch=B, device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    fs = c["width"] * c["height"]

    def tum_step(i=0):
        o = (i % (P // B)) * B
        ctx.rgbd_batch_device(B, dg.data_ptr() + o * fs, c["width"], fs, dd.data_ptr() + 2 * o * fs, 2 * c["width"], 2 * fs, api.DEPTH_U16)

    ms = timed_ms(tum_step, 20)
    alg = ctx.algorithmic_bytes(False) + 18 * c["n_features"]
    fps = B / (ms * 1e-3)
    one = api.Context(c["width"], c["height"], c["n_features"], c["n_levels"], c["scale_factor"], camera=cam, max_batch=1, device=local_rank)
    r = one.rgbd_frame(g[0], d[0])
    lat = []
    for i in range(40):
        t0 = time.perf_counter()
        one.rgbd_frame(g[i % P], d[i % P])
        lat.append(1e3 * (time.perf_counter() - t0))
    out["tum_rgbd"] = {
        "workload": "synthetic TUM-shaped RGB-D frames 640x480, 1000 features, 8 levels, TUM distortion, uint16 depth / 5208 (BASELINE.json configs[1])",
        "value": fps, "unit": "frames/s", "frames_per_launch": B, "pool_frames": P, "ms_per_step": ms, "algorithmic_bytes_per_frame": alg,
        "roofline": {"bound": "hbm", "achieved": alg * fps / 1e9, "peak": peak, "unit": "GB/s", "frac": alg * fps / 1e9 / peak},
        "p50_ms_host_to_host": float(np.median(lat[10:])), "depth_valid_fraction": float((r.depth > 0).mean()),
        "check": oracle_flip_check(api, O, r.kps_raw, r.desc, g[0], c["n_features"], c["n_levels"], c["scale_factor"]) if O else None,
    }
    ctx.close()
    one.close()
    del dg, dd

    # configs[4]: 1920x1080 stereo, 5000 features, 12 levels
    c = synth.HD
    B, P = 16, 32
    l, r_ = synth.synth_stereo_pool(c["height"], c["width"], P, seed0=4000)
    with torch.cuda.stream(stream):
        dl, dr = torch.from_numpy(l).cuda(), torch.from_numpy(r_).cuda()
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    ctx = api.Context(c["width"], c["height"], c["n_features"], c["n_levels"], c["scale_factor"], camera=cam, max_batch=B, device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    fs = c["width"] * c["height"]

    def hd_step(i=0):
        o = (i % (P // B)) * B
        ctx.stereo_batch_device(B, dl.data_ptr() + o * fs, dr.data_ptr() + o * fs, c["width"], fs)

    ms = timed_ms(hd_step, 20)
    stages = ctx.profile_stereo_batch_device(B, dl.data_ptr(), dr.data_ptr(), c["width"], fs)
    alg = ctx.algorithmic_bytes(True)
    fps = B / (ms * 1e-3)
    one = api.Context(c["width"], c["height"], c["n_features"], c["n_levels"], c["scale_factor"], camera=cam, max_batch=1, device=local_rank)
    one.set_stream(stream.cuda_stream)
    lat = []
    for i in range(40):
        e0, e1 = _events(torch)
        e0.record(stream)
        one.stereo_batch_device(1, dl.data_ptr() + (i % P) * fs, dr.data_ptr() + (i % P) * fs, c["width"], fs)
        e1.record(stream)
        stream.synchronize()
        lat.append(e0.elapsed_time(e1))
    one.set_stream(None)
    res = one.stereo_frame(l[0], r_[0])
    out["hd_1080p"] = {
        "workload": "synthetic 1920x1080 stereo pairs, 5000 features, 12 levels x1.2 (BASELINE.json configs[4])",
        "value": fps, "unit": "frames/s", "frames_per_launch": B, "pool_pairs": P, "ms_per_step": ms, "algorithmic_bytes_per_frame": alg, "stage_ms": stages,
        "roofline": {"bound": "hbm", "achieved": alg * fps / 1e9, "peak": peak, "unit": "GB/s", "frac": alg * fps / 1e9 / peak},
        "p50_ms_device_single_pair": float(np.median(lat[10:])), "matches_first_pair": int(res.n_matches),
        "check": oracle_flip_check(api, O, res.kps_left, res.desc_left, l[0], c["n_features"], c["n_levels"], c["scale_factor"]) if O else None,
    }
    ctx.close()
    one.close()
    del dl, dr

    # configs[3]: per-frame latency sweep over the feature count on KITTI-shaped stereo, single GPU (left and right run in the same launches)
    c = synth.KITTI
    P = 16
    l, r_ = synth.synth_stereo_pool(c["height"], c["width"], P, seed0=0)
    with torch.cuda.stream(stream):
        dl, dr = torch.from_numpy(l).cuda(), torch.from_numpy(r_).cuda()
    hl, hr = torch.from_numpy(l).pin_memory(), torch.from_numpy(r_).pin_memory()
    fs = c["width"] * c["height"]
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    sweep = {}
    for nf in (500, 1000, 2000, 4000):
        one = api.Context(c["width"], c["height"], nf, c["n_levels"], c["scale_factor"], camera=cam, max_batch=1, device=local_rank)
        row = {}
        for graph in (True, False):
            one.set_graph(graph)
            one.set_stream(stream.cuda_stream)
            dev = []
            for i in range(60):
                e0, e1 = _events(torch)
                e0.record(stream)
                one.stereo_batch_device(1, dl.data_ptr() + (i % P) * fs, dr.data_ptr() + (i % P) * fs, c["width"], fs)
                e1.record(stream)
                stream.synchronize()
                dev.append(e0.elapsed_time(e1))
            one.set_stream(None)
            host = []
            ptrs = pinned_outputs(torch, nf)
            for i in range(60):
                t0 = time.perf_counter()
                one.stereo_batch_ptr(1, hl.data_ptr() + (i % P) * fs, hr.data_ptr() + (i % P) * fs, c["width"], fs, ptrs)
                host.append(1e3 * (time.perf_counter() - t0))
            tag = "graph" if graph else "stream_launches"
            row["p50_ms_device_" + tag] = float(np.median(dev[10:]))
            row["p50_ms_host_to_host_" + tag] = float(np.median(host[10:]))
        res = one.stereo_frame(l[0], r_[0])
        row["keypoints"], row["matches"] = int(len(res.kps_left)), int(res.n_matches)
        if O:
            row["check"] = oracle_flip_check(api, O, res.kps_left, res.desc_left, l[0], nf, c["n_levels"], c["scale_factor"])
        sweep[str(nf)] = row
        one.close()
    out["latency_sweep"] = {"workload": "single KITTI-shaped stereo pair per call, nFeatures in {500, 1000, 2000, 4000} (BASELINE.json configs[3])",
                            "note": "device = images and results in HBM (CUDA events); host_to_host = pinned host images in, results out (wall clock); "
                                    "graph = the call replays one captured CUDA graph, stream_launches = 8 separate launches", "n_features": sweep}
    return out


DUMP_FRAMES = 32  # frames per sampled output: about 30 MB of .npy files in all at 2000 features


def dump_outputs(out_dir, ctx, torch, d_rec, n_local, res, F):
    """Write what the last timed step returned as float32 / float64 .npy files: the per-frame records of a fixed, seeded
    sample of this rank's frames, the gathered left descriptors of a seeded sample of the sequence's frames and the gathered
    keypoint counts of every frame.  Entries past a frame's keypoint count are not part of the result and are written as 0."""
    from orb_slam2_ros2_b200 import api

    os.makedirs(out_dir, exist_ok=True)
    N = ctx.n_features
    rng = np.random.default_rng(0)
    out = {}
    idx = np.sort(rng.choice(n_local, min(n_local, DUMP_FRAMES), replace=False))
    rec = d_rec[torch.from_numpy(idx).cuda()].cpu().numpy().view(ctx.record_dtype())[:, 0]
    out["frames"] = idx.astype(np.float64)  # rank 0's block starts at frame 0
    for side in ("left", "right"):
        n = rec["n_" + side]
        keep = np.arange(N)[None, :] < n[:, None]
        kps = rec["kps_" + side]
        out["n_" + side] = n.astype(np.float64)
        out["kps_" + side] = np.where(keep[..., None], np.stack([kps[f].astype(np.float32) for f in api.KP_DTYPE.names], -1), 0)
        out["desc_" + side] = np.where(keep[..., None], rec["desc_" + side], 0).astype(np.float32)
        if side == "left":
            out["u_right"], out["depth"] = np.where(keep, rec["u_right"], 0.0), np.where(keep, rec["depth"], 0.0)
    out["n_matches"] = rec["n_matches"].astype(np.float64)
    g_n = ctx.read_device(res.gathered_n, (F,), np.int32)
    g_idx = np.sort(rng.choice(F, min(F, DUMP_FRAMES), replace=False))
    g_desc = torch.as_tensor(CudaArray(res.gathered_desc, (res.world * res.block, N, 32), "|u1"), device="cuda")
    keep = np.arange(N)[None, :] < g_n[g_idx][:, None]
    out["gathered_n"] = g_n.astype(np.float64)
    out["gathered_frames"] = g_idx.astype(np.float64)
    out["gathered_desc"] = np.where(keep[..., None], g_desc[torch.from_numpy(g_idx).cuda()].cpu().numpy(), 0).astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from orb_slam2_ros2_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL announces its version on stdout when the first communicator is created; the contract is ONE JSON line there,
        # so fd 1 points at stderr until the communicators exist
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)

    H, W, N = CFG["height"], CFG["width"], CFG["n_features"]
    B, P, F = args.batch, args.pool, args.frames
    cam = api.Camera(CFG["fx"], CFG["fy"], CFG["cx"], CFG["cy"], CFG["bl"])
    ctx = api.Context(W, H, N, CFG["n_levels"], CFG["scale_factor"], CFG["ini_th"], CFG["min_th"], camera=cam, max_batch=B, device=local_rank)
    comm = None
    try:
        if world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
            # the library's own communicator (the descriptor gather lives behind the C ABI): rank 0 makes the id, torch carries it
            ids = [api.Communicator.unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            comm = api.Communicator(ctx, rank, world, ids[0], F)
            if args.transport == "peer":
                # descriptor gather as stores into every rank's gathered array (CUDA-IPC peer pointers) from the kernel that packs the
                # records; if any rank cannot map its peers, every rank stays on the NCCL send/recv pieces
                try:
                    handle, ok = comm.ipc_handle(), 1
                except Exception:
                    handle, ok = b"", 0
                handles = [None] * world
                dist.all_gather_object(handles, (handle, ok))
                if all(h[1] for h in handles):
                    try:
                        comm.open_peers([h[0] for h in handles])
                    except Exception:
                        ok = 0
                oks = [None] * world
                dist.all_gather_object(oks, ok)
                if not all(oks):
                    raise SystemExit("bench.py: peer-memory transport could not be set up on every rank; rerun with --transport nccl")
    finally:
        if world > 1:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    # ---- the sequence: frame f = pool pair f mod P; this rank materialises its block in pinned host memory and in HBM ----
    pool_l, pool_r = synth.synth_stereo_pool(H, W, P, seed0=0)
    blk = api.frame_range(F, rank, world)
    n_local = len(blk)
    fsz = W * H
    h_left = torch.empty((max(n_local, 1), H, W), dtype=torch.uint8, pin_memory=True)
    h_right = torch.empty((max(n_local, 1), H, W), dtype=torch.uint8, pin_memory=True)
    idx = np.arange(blk.start, blk.stop) % P
    if n_local:
        np.take(pool_l, idx, axis=0, out=h_left.numpy()[:n_local])
        np.take(pool_r, idx, axis=0, out=h_right.numpy()[:n_local])
    d_left, d_right = h_left.cuda(non_blocking=True), h_right.cuda(non_blocking=True)
    rs = ctx.record_layout().record_bytes
    d_rec = torch.empty((max(n_local, 1), rs), dtype=torch.uint8, device="cuda")
    h_rec = torch.empty((max(n_local, 1), rs), dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()  # the stream every call of the timed region is issued on
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    last = {}

    def device_step():
        last["res"] = ctx.sequence_stereo_ptr(F, d_left.data_ptr(), d_right.data_ptr(), W, fsz, comm, True, d_rec.data_ptr(), rs, True)

    def host_step():
        last["res"] = ctx.sequence_stereo_ptr(F, h_left.data_ptr(), h_right.data_ptr(), W, fsz, comm, False, h_rec.data_ptr(), rs, False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (`value`): K passes over the sequence, images and records in HBM ---------------------
    sampler = ClockSampler(local_rank)
    sampler.start()  # started before the warm-up so that short timed regions still get samples under load
    sampler.wait_first_sample()
    for _ in range(args.warmup):
        device_step()
    barrier()
    launches0 = ctx.launch_count
    e0, e1 = _events(torch)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        device_step()  # returns once this rank's records and (N > 1) the gathered descriptors are complete
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, torch, d_rec, n_local, last["res"], F)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = args.steps * F / (ms_max * 1e-3)
    res = last["res"]
    cap = res.world * res.block

    # ---- verification of the timed work: records, gathered descriptors, ranks agree ---------------------------------------
    g_desc = torch.as_tensor(CudaArray(res.gathered_desc, (cap, N * 32), "|u1"), device="cuda")
    g_n = torch.as_tensor(CudaArray(res.gathered_n, (cap,), "<i4"), device="cuda")
    rec_np_dtype = ctx.record_dtype()
    check = {}
    # (a) frames f and f + P are the same pair, computed by different ranks / slots / chunks: their gathered rows must be identical
    if F > P:
        check["gathered_rows_periodic"] = bool(torch.equal(g_desc[: F - P], g_desc[P:F]) and torch.equal(g_n[: F - P], g_n[P:F]))
    # (b) one checksum of the gathered arrays per rank; all ranks must hold the same bytes (and the same as an N = 1 run of this bench)
    csum = int(g_desc[:F].view(torch.int64).sum().item()) & 0xFFFFFFFFFFFFFFFF
    csum ^= int(g_n[:F].to(torch.int64).sum().item())
    sums = [csum]
    if world > 1:
        sums = [None] * world
        dist.all_gather_object(sums, csum)
    check["gathered_checksum"] = f"{sums[0]:016x}"
    check["gathered_checksum_equal_on_all_ranks"] = bool(all(x == sums[0] for x in sums))
    check["gathered_keypoints_total"] = int(g_n[:F].sum().item())
    # (c) this rank's device records agree with its rows of the gathered array
    if n_local:
        lay = ctx.record_layout()
        mine = d_rec[:n_local, lay.off_desc_left: lay.off_desc_left + N * 32]
        ok = bool(torch.equal(mine, g_desc[blk.start:blk.stop]))
    else:
        ok = True
    oks = [ok]
    if world > 1:
        oks = [None] * world
        dist.all_gather_object(oks, ok)
    check["records_equal_gathered_rows_on_all_ranks"] = bool(all(oks))
    # (d) rank 0 recomputes sampled frames of EVERY rank's block alone (single-frame call, own context) and, for two of them, with the oracle
    if rank == 0:
        one = api.Context(W, H, N, CFG["n_levels"], CFG["scale_factor"], CFG["ini_th"], CFG["min_th"], camera=cam, max_batch=1, device=local_rank)
        sample = sorted({f for r in range(world) for b in [api.frame_range(F, r, world)] if len(b) for f in (b.start, b.stop - 1)})
        good = 0
        for f in sample:
            r1 = one.stereo_frame(pool_l[f % P], pool_r[f % P])
            row = g_desc[f].cpu().numpy().reshape(N, 32)
            n_f = int(g_n[f].item())
            good += int(n_f == len(r1.kps_left) and np.array_equal(row[:n_f], r1.desc_left) and not row[n_f:].any())
        check["sampled_frames_vs_single_frame_call"] = {"frames": sample, "identical": good}
        if not args.no_cpu_baseline:
            from oracle import oracle_py as O  # checker only

            r1 = one.stereo_frame(pool_l[0], pool_r[0])
            oc = oracle_flip_check(api, O, r1.kps_left, r1.desc_left, pool_l[0], N, CFG["n_levels"], CFG["scale_factor"])
            el, er = O.extract(pool_l[0], N, CFG["n_levels"], CFG["scale_factor"]), O.extract(pool_r[0], N, CFG["n_levels"], CFG["scale_factor"])
            nm, ur, dp, _ = O.search_by_stereo(el, er, np.float32(cam.fx), cam.bf)
            oc["stereo_matches_equal"] = bool(nm == r1.n_matches)
            oc["max_u_right_error_px"] = float(np.abs(r1.u_right - ur).max()) if len(ur) == len(r1.u_right) else None
            oc["max_depth_error"] = float(np.abs(r1.depth - dp).max()) if len(dp) == len(r1.depth) else None
            check["oracle_frame0"] = oc
        one.close()
    if n_local:
        rec0 = d_rec[0].cpu().numpy().view(rec_np_dtype)[0]
        check["first_local_frame"] = {"n_left": int(rec0["n_left"]), "n_right": int(rec0["n_right"]), "n_matches": int(rec0["n_matches"])}

    # ---- end to end (`e2e`): the same call with the block in pinned HOST memory and the records landing in pinned host memory ----
    ctx.set_stream(None)
    e2e_steps = max(2, min(args.steps, 10))
    host_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps * F / float(t.item())
    if n_local:
        check["host_records_equal_device_records"] = bool(torch.equal(h_rec[:n_local], d_rec[:n_local].cpu()))
    h2d = 2 * F * fsz
    d2h = F * rs

    # ---- platform ceiling of `e2e`: the same bytes as bare pinned-memory copies (8-frame chunks, H2D and D2H on two streams, all
    # ranks at once, no kernels).  `e2e` cannot exceed what the box moves between host and device memory.
    ceiling = None
    if n_local >= 64 or world > 1:
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        d_in = torch.empty((2, 64, fsz), dtype=torch.uint8, device="cuda")
        d_out = torch.empty((64, rs), dtype=torch.uint8, device="cuda")
        hl, hr, hrec = h_left.view(-1, fsz), h_right.view(-1, fsz), h_rec

        def bare_pass():
            for f0 in range(0, n_local, 8):
                nf = min(8, n_local - f0)
                o = (f0 // 8 % 8) * 8
                with torch.cuda.stream(s_in):
                    d_in[0, o:o + nf].copy_(hl[f0:f0 + nf], non_blocking=True)
                    d_in[1, o:o + nf].copy_(hr[f0:f0 + nf], non_blocking=True)
                with torch.cuda.stream(s_out):
                    hrec[f0:f0 + nf].copy_(d_out[o:o + nf], non_blocking=True)
            torch.cuda.synchronize()

        bare_pass()
        barrier()
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            bare_pass()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        cfps = reps * F / float(t.item())
        ceiling = {"value": cfps, "unit": UNIT, "h2d_GBps": cfps * 2 * fsz / 1e9, "d2h_GBps": cfps * rs / 1e9,
                   "what": "bare cudaMemcpyAsync of the same pinned buffers (8-frame chunks, H2D and D2H on two streams, all ranks at once, no kernels)"}
        del d_in, d_out
    ctx.set_stream(stream.cuda_stream)

    # ---- per-stage device times of one 64-frame slot batch -> roofline of the dominant kernel ------------------------------
    stage_ms = {}
    reps = 5
    nb = max(1, min(B, n_local))
    for r in range(reps):
        o = (r * nb) % max(1, n_local - nb + 1)
        sm = ctx.profile_stereo_batch_device(nb, d_left.data_ptr() + o * fsz, d_right.data_ptr() + o * fsz, W, fsz)
        if r == 0:
            continue
        for k, v in sm.items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v / (reps - 1)
    dominant = max(stage_ms, key=stage_ms.get)
    peak, peak_src = measured_peaks()
    alg_frame = ctx.algorithmic_bytes(True)
    dom_ms = stage_ms[dominant]
    achieved = alg_frame * nb / (dom_ms * 1e-3) / 1e9
    step_total = sum(stage_ms.values())
    traffic = None
    try:  # dram__bytes_read+write of the same kernel from the committed ncu --set full capture (per 64-frame launch)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[dominant]
        traffic = tj["dram_bytes_per_launch"] * nb / tj["frames_per_launch"]
    except Exception:
        pass
    roofline = {
        "bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
        "peak_source": peak_src, "algorithmic_bytes_per_frame": alg_frame, "frames_per_launch": nb, "kernel_ms": dom_ms,
        "kernel_share_of_step": dom_ms / step_total, "stage_ms": stage_ms,
        "whole_step": {"achieved": alg_frame * value / world / 1e9, "frac": alg_frame * value / world / 1e9 / peak,
                       "note": "algorithmic bytes of one frame x frames/s per GPU over the measured HBM peak"},
    }

    # ---- single-frame latency (p50), one GPU: with the CUDA graph and with plain stream launches -----------------------------
    latency = None
    if rank == 0 and n_local:
        one = api.Context(W, H, N, CFG["n_levels"], CFG["scale_factor"], CFG["ini_th"], CFG["min_th"], camera=cam, max_batch=1, device=local_rank)
        latency = {"frames": 50, "note": "one stereo pair per call; device = inputs and results in HBM, host_to_host = pinned host images in, results out"}
        np_ = min(n_local, P)
        p1 = pinned_outputs(torch, N)
        for graph in (True, False):
            one.set_graph(graph)
            one.set_stream(stream.cuda_stream)
            dev_ms, host_ms = [], []
            for i in range(60):
                a, b = _events(torch)
                a.record(stream)
                one.stereo_batch_device(1, d_left.data_ptr() + (i % np_) * fsz, d_right.data_ptr() + (i % np_) * fsz, W, fsz)
                b.record(stream)
                torch.cuda.synchronize()
                if i >= 10:
                    dev_ms.append(a.elapsed_time(b))
            one.set_stream(None)
            for i in range(60):
                t0 = time.perf_counter()
                one.stereo_batch_ptr(1, h_left.data_ptr() + (i % np_) * fsz, h_right.data_ptr() + (i % np_) * fsz, W, fsz, p1)
                if i >= 10:
                    host_ms.append(1e3 * (time.perf_counter() - t0))
            tag = "" if graph else "_stream_launches"
            latency["p50_ms_device" + tag] = float(np.median(dev_ms))
            latency["p50_ms_host_to_host" + tag] = float(np.median(host_ms))
        one.close()

    # ---- the other BASELINE configurations and the SURVEY 8(f) rows: secondary lines, one GPU --------------------------------
    configs = matchers = serialize = bow = None
    if rank == 0 and world == 1 and not args.no_configs:
        configs = bench_other_configs(args, api, torch, stream, local_rank, with_oracle=not args.no_cpu_baseline)
    if rank == 0 and world == 1 and not args.no_matchers and n_local >= B:
        matchers = bench_matchers(ctx, api, torch, stream, d_left, d_right, B, W, H, N, fsz, cpu=not args.no_cpu_baseline)
        serialize = matchers.pop("serialize", None)
        bow = matchers.pop("bow", None)

    # ---- CPU baseline beside it (rank 0, N=1 only) ---------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ncpu = os.cpu_count() or 1
        workers = max(1, ncpu // 2)
        n_frames = max(16, 8 * workers)
        cpu_reference_run(workers, workers)  # warm
        fps, cores, kind, sample = cpu_reference_run(n_frames, workers)
        cpu = {"value": fps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "opencv_primitives": opencv_primitives_timing(fps, workers)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args), "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "platform_ceiling": ceiling, "fraction_of_platform_ceiling": (e2e_value / ceiling["value"]) if ceiling else None,
                    "note": "the same orbx_sequence_stereo call with every rank's block in pinned host memory and its records landing in pinned host memory; "
                            "the gathered descriptors stay in HBM (they are consumed there)"},
            "gpu_launches": int(launches), "transport": (comm.info()["transport"] if comm else 0), "roofline": roofline, "cpu_baseline": cpu, "latency": latency,
            "configs": configs, "matchers": matchers, "serialize": serialize, "bow": bow, "check": check,
        }
        print(json.dumps(line), flush=True)
    if comm is not None:
        barrier()
        comm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=SEQ_FRAMES, help="frames of the sequence (one step = one pass over all of them, sharded over the GPUs)")
    ap.add_argument("--batch", type=int, default=64, help="device slots per GPU (frames in flight)")
    ap.add_argument("--pool", type=int, default=256, help="distinct synthetic pairs the sequence cycles through")
    ap.add_argument("--transport", default="peer", choices=["nccl", "peer"],
                    help="descriptor gather at N > 1: peer = stores through CUDA-IPC peer pointers fused into the record-packing kernel (NCCL carries the "
                         "closing barrier), nccl = grouped ncclSend/ncclRecv pieces on a side stream")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-matchers", action="store_true", help="skip the secondary tracking-matcher / serialisation / bag-of-words measurements")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary BASELINE configurations (TUM RGB-D, 1080p, latency sweep)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (a seeded sample of frames) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
