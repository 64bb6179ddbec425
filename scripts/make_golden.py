#!/usr/bin/env python
"""Generate tests/golden/*.npz from the reference's OWN code (oracle/_ref/libref.so = /root/reference sources compiled
unmodified against oracle/stub).  Run in the build container (needs /root/reference); the fixtures are committed.

Every fixture stores the generator seed + a SHA-256 of the synthetic input (so a numpy change that alters the input is
detected instead of silently failing parity) and the reference outputs: keypoints (28-byte cv::KeyPoint records),
descriptors, uRight/depth, per-level pyramid checksums.
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle_py as O  # noqa: E402
from orb_slam2_ros2_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    assert O.have_ref(), "oracle/_ref/libref.so missing: run make -C oracle in a container with /root/reference"
    os.makedirs(OUT, exist_ok=True)
    with tempfile.TemporaryDirectory() as td:
        tp = O.write_template_file(os.path.join(td, "brief_template.txt"))
        # 1. KITTI-shaped stereo pair, 2000 features (configs[0])
        c = synth.KITTI
        left, right = synth.synth_stereo_pair(c["height"], c["width"], 0, 17)
        O.ref_reset()
        O.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)
        r = O.ref_stereo(left, right, tp, 2000, 8, 1.2)
        _, _, _, info = O.ref_extract(left, tp, 2000, 8, 1.2, want_pyramid=True)
        np.savez_compressed(os.path.join(OUT, "kitti_stereo_seed0_d17.npz"), seed=0, disparity=17, left_sha=sha(left), right_sha=sha(right),
                            kl=r["kl"], dl=r["dl"], kr=r["kr"], dr=r["dr"], u_right=r["u_right"], depth=r["depth"], n_matches=r["n_matches"],
                            pyr_sha=np.array([sha(l) for l in info["levels"]]))
        # 1b. TUM-shaped stereo pair, 1000 features (test_gpu_parity.py::test_stereo_matches_the_compiled_reference)
        c = synth.TUM
        left, right = synth.synth_stereo_pair(c["height"], c["width"], 3, 17)
        O.ref_reset()
        O.ref_set_camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], None)
        r = O.ref_stereo(left, right, tp, 1000, 8, 1.2)
        np.savez_compressed(os.path.join(OUT, "tum_stereo_seed3_d17.npz"), seed=3, disparity=17, left_sha=sha(left), right_sha=sha(right),
                            kl=r["kl"], dl=r["dl"], kr=r["kr"], dr=r["dr"], u_right=r["u_right"], depth=r["depth"], n_matches=r["n_matches"])
        # 2. small stereo pair used by smoke-sized tests: 320x240, 500 features, 4 levels
        left, right = synth.synth_stereo_pair(240, 320, 0, 9)
        O.ref_reset()
        O.ref_set_camera(300.0, 300.0, 160.0, 120.0, 0.1, None)
        r = O.ref_stereo(left, right, tp, 500, 4, 1.2)
        np.savez_compressed(os.path.join(OUT, "small_stereo_seed0_d9.npz"), seed=0, disparity=9, left_sha=sha(left), right_sha=sha(right),
                            kl=r["kl"], dl=r["dl"], kr=r["kr"], dr=r["dr"], u_right=r["u_right"], depth=r["depth"], n_matches=r["n_matches"])
        # 2b. tracking-side matchers on the small frame: findFeaturesInArea + getBestMatch (+ exclusion) and verifyAngle
        kl, dl = r["kl"], r["dl"]
        sf = np.array([np.float32(np.float64(np.float32(1.2)) ** l) for l in range(4)], np.float32)
        q, qd, ex, src = synth.synth_area_queries(kl, dl, 400, 5, 320, 240, n_levels=4, th=15.0)
        bounds = (0.0, 0.0, 320.0, 240.0)
        a = O.ref_search_in_area(kl, dl, bounds, sf, q, qd, None)
        b = O.ref_search_in_area(kl, dl, bounds, sf, q, qd, ex)
        ok = a["best_idx"] >= 0
        k2 = np.zeros(len(q), O.KP_DTYPE)
        k2["angle"] = (kl["angle"][src] + np.random.default_rng(6).normal(0, 25, len(q))).astype(np.float32)
        qi, ti, di = a["best_idx"][ok], np.nonzero(ok)[0].astype(np.int32), a["best_dist"][ok].astype(np.float32)
        vq, vt, vd = O.ref_verify_angle(qi, ti, di, kl, k2)
        np.savez_compressed(os.path.join(OUT, "small_area_match_seed5.npz"), seed=5, n=400, q_sha=sha(q), qd_sha=sha(qd), k2_angle=k2["angle"],
                            best_idx=a["best_idx"], best_dist=a["best_dist"], ratio=a["ratio"], n_cand=a["n_cand"], x_best_idx=b["best_idx"],
                            x_best_dist=b["best_dist"], x_ratio=b["ratio"], x_n_cand=b["n_cand"], va_query=vq, va_train=vt, va_dist=vd)
        # 3. TUM-shaped mono extraction, 1000 features (the extractor part of configs[1]; the RGB-D ctor itself cannot be compiled in isolation)
        c = synth.TUM
        gray = synth.synth_image(c["height"], c["width"], 12)
        O.ref_reset()
        n, kps, desc, info = O.ref_extract(gray, tp, 1000, 8, 1.2, want_pyramid=True)
        np.savez_compressed(os.path.join(OUT, "tum_extract_seed12.npz"), seed=12, gray_sha=sha(gray), kps=kps, desc=desc,
                            pyr_sha=np.array([sha(l) for l in info["levels"]]))
        # 4. 1080p, 5000 features, 12 levels: hashes only (configs[4])
        c = synth.HD
        img = synth.synth_image(c["height"], c["width"], 4)
        O.ref_reset()
        n, kps, desc, info = O.ref_extract(img, tp, 5000, 12, 1.2, want_pyramid=True)
        np.savez_compressed(os.path.join(OUT, "hd_extract_seed4_hashes.npz"), seed=4, img_sha=sha(img), n=n, xy_octave_response_sha=sha(
            np.stack([kps["x"], kps["y"], kps["response"], kps["octave"].astype(np.float32)], 1)), desc_sha=sha(desc), angle=kps["angle"],
            pyr_sha=np.array([sha(l) for l in info["levels"]]))
        O.ref_reset()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
