"""GPU parity of the frame-sharded sequence entry (orbx_sequence_stereo, BASELINE.json configs[2] in miniature).

* single rank: every frame's record == the single-frame call == the oracle, whatever its position in a chunk / slot;
* two ranks in ONE process on cuda:0 (orbx_comm_create_local, peer-memory transport): ragged blocks (11 = 6 + 5), the
  gathered descriptors of BOTH ranks == the single-rank result == the oracle;
* two ranks in two processes over NCCL and over CUDA-IPC peer memory (torchrun; needs >= 2 GPUs, skipped otherwise).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

H, W, NF, NL = 240, 320, 300, 5
CAM = api.Camera(300.0, 300.0, 160.0, 120.0, 0.1)


def _pool(F, seed0=200):
    return synth.synth_stereo_pool(H, W, F, seed0=seed0, disparity=9)


def _check_record_vs_frame(rec, r):
    nl, nr = int(rec["n_left"]), int(rec["n_right"])
    assert nl == len(r.kps_left) and nr == len(r.kps_right) and int(rec["n_matches"]) == r.n_matches
    assert rec["kps_left"][:nl].tobytes() == r.kps_left.tobytes() and rec["kps_right"][:nr].tobytes() == r.kps_right.tobytes()
    assert np.array_equal(rec["desc_left"][:nl], r.desc_left) and np.array_equal(rec["desc_right"][:nr], r.desc_right)
    assert np.array_equal(rec["u_right"][:nl], r.u_right) and np.array_equal(rec["depth"][:nl], r.depth)
    # entries beyond the counts are zero, so records are deterministic
    assert not rec["desc_left"][nl:].any() and not rec["u_right"][nl:].any() and not rec["kps_right"][nr:].view(np.uint8).any()


def test_single_rank_sequence_equals_frames_and_oracle(oracle):
    F = 11
    lefts, rights = _pool(F)
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)  # 11 frames through 4 device slots
    rec, gd, gn = ctx.sequence_stereo(lefts, rights)
    assert rec.dtype.itemsize == ctx.record_layout().record_bytes and len(rec) == F
    one = api.Context(W, H, NF, NL, 1.2, camera=CAM)
    for f in range(F):
        _check_record_vs_frame(rec[f], one.stereo_frame(lefts[f], rights[f]))
        assert gn[f] == rec[f]["n_left"] and np.array_equal(gd[f], rec[f]["desc_left"])
    for f in (0, 4, 10):
        el, er = oracle.extract(lefts[f], NF, NL, 1.2), oracle.extract(rights[f], NF, NL, 1.2)
        nm, ur, dp, _ = oracle.search_by_stereo(el, er, np.float32(CAM.fx), CAM.bf)
        n = len(el.kps)
        assert rec[f]["n_left"] == n and int(np.unpackbits(rec[f]["desc_left"][:n] ^ el.desc).sum()) <= 2
        assert rec[f]["n_matches"] == nm and np.abs(rec[f]["u_right"][:n] - ur).max() <= 1e-3 and np.abs(rec[f]["depth"][:n] - dp).max() <= 1e-3
    # a second, shorter sequence on the same context reuses the gathered arrays
    rec2, gd2, gn2 = ctx.sequence_stereo(lefts[:3], rights[:3])
    assert rec2.tobytes() == rec[:3].tobytes() and np.array_equal(gd2, gd[:3])
    one.close()
    ctx.close()


def test_device_inputs_and_device_records():
    import torch

    F = 9
    lefts, rights = _pool(F, 300)
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)
    rec_h, gd, gn = ctx.sequence_stereo(lefts, rights)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    rs = ctx.record_layout().record_bytes
    d_rec = torch.zeros((F, rs), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    res = ctx.sequence_stereo_ptr(F, dl.data_ptr(), dr.data_ptr(), W, W * H, None, True, d_rec.data_ptr(), rs, True)
    assert (res.frame_lo, res.frame_hi, res.block, res.world) == (0, F, F, 1)
    assert d_rec.cpu().numpy().tobytes() == rec_h.tobytes()
    assert np.array_equal(ctx.read_device(res.gathered_desc, (F, NF, 32), np.uint8), gd)
    assert np.array_equal(ctx.read_device(res.gathered_n, (F,), np.int32), gn)
    ctx.close()


@pytest.mark.parametrize("F", [11, 2, 1])
def test_two_local_ranks_gather_equals_single_rank(oracle, F):
    """rank 0 and rank 1 are two contexts on cuda:0 driven by one thread; the pack kernel of each rank stores its left
    descriptors into BOTH ranks' gathered arrays (peer-memory transport)"""
    lefts, rights = _pool(F, 400)
    ref = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)
    rec1, gd1, gn1 = ref.sequence_stereo(lefts, rights)
    ctxs = [api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=2) for _ in range(2)]
    comms = api.Communicator.local(ctxs, F)
    assert [c.info()["transport"] for c in comms] == [api.TRANSPORT_PEER] * 2
    recs, results = [], []
    for r in range(2):
        blk = api.frame_range(F, r, 2)
        rec = np.zeros(max(len(blk), 1), ctxs[r].record_dtype())
        res = ctxs[r].sequence_stereo_ptr(F, lefts[blk.start:].ctypes.data if len(blk) else lefts.ctypes.data,
                                          rights[blk.start:].ctypes.data if len(blk) else rights.ctypes.data, W, W * H, comms[r], False,
                                          rec.ctypes.data, rec.dtype.itemsize, False)
        assert (res.frame_lo, res.frame_hi) == (blk.start, blk.stop) and res.world == 2 and res.block == -(-F // 2)
        recs.append(rec[: len(blk)])
        results.append(res)
    assert b"".join(r.tobytes() for r in recs) == rec1.tobytes()  # (np.concatenate would drop the padding bytes of the structured dtype)
    for r in range(2):
        res = results[r]
        cap = 2 * res.block
        gd = ctxs[r].read_device(res.gathered_desc, (cap, NF, 32), np.uint8)
        gn = ctxs[r].read_device(res.gathered_n, (cap,), np.int32)
        assert np.array_equal(gd[:F], gd1) and np.array_equal(gn[:F], gn1), f"rank {r}"
        assert not gn[F:].any()
    f = F - 1
    el = oracle.extract(lefts[f], NF, NL, 1.2)
    assert gn1[f] == len(el.kps) and int(np.unpackbits(gd1[f, : len(el.kps)] ^ el.desc).sum()) <= 2
    for c in comms:
        c.close()
    for c in ctxs + [ref]:
        c.close()


@pytest.mark.parametrize("transport", ["nccl", "peer"])
def test_two_processes_gather_equals_single_rank(transport):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, ORBX_TEST_TRANSPORT=transport, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29611",
           os.path.join(ROOT, "tests", "workers", "sequence_worker.py")]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("SEQUENCE_OK") == 2, r.stdout[-3000:] + r.stderr[-3000:]
