"""The host-side stereo entry points on inputs the other tests do not use: left and right rows at different strides,
pitched host batches and sequences that reuse the device slots, the per-stage profile against the device batch, and the
stride check of host batches.
"""
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

pytestmark = pytest.mark.gpu

H, W, NF, NL = 240, 320, 300, 5
CAM = api.Camera(300.0, 300.0, 160.0, 120.0, 0.1)
FIELDS = ("kps_left", "desc_left", "kps_right", "desc_right", "u_right", "depth")


def _pool(F, seed0):
    return synth.synth_stereo_pool(H, W, F, seed0=seed0, disparity=9)


def _pitched(images, stride, frame_stride):
    """images (n, H, W) copied into one host buffer: frame f at f * frame_stride, rows `stride` bytes apart"""
    n = len(images)
    buf = np.zeros((n - 1) * frame_stride + (H - 1) * stride + W, np.uint8)
    for f in range(n):
        view = np.lib.stride_tricks.as_strided(buf[f * frame_stride:], (H, W), (stride, 1))
        view[:] = images[f]
    return buf


def test_stereo_frame_with_different_row_strides(oracle):
    lefts, rights = _pool(1, 500)
    left, right = lefts[0], rights[0]
    wide = np.zeros((H, W + 37), np.uint8)
    wide[:, 5:5 + W] = left
    left_slice = wide[:, 5:5 + W]  # rows W + 37 bytes apart, wider than the staging pitch
    assert left_slice.strides[0] != right.strides[0]
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM)
    ref = ctx.stereo_frame(left, right)
    got = ctx.stereo_frame(left_slice, right)
    again = ctx.stereo_frame(left, right)
    for name in FIELDS:
        assert getattr(got, name).tobytes() == getattr(ref, name).tobytes(), name
        assert getattr(again, name).tobytes() == getattr(ref, name).tobytes(), name
    assert got.n_matches == ref.n_matches == again.n_matches
    el, er = oracle.extract(left, NF, NL, 1.2), oracle.extract(right, NF, NL, 1.2)
    nm, ur, dp, _ = oracle.search_by_stereo(el, er, np.float32(CAM.fx), CAM.bf)
    n = len(el.kps)
    assert len(got.kps_left) == n and len(got.kps_right) == len(er.kps)
    for f in ("x", "y", "response", "octave"):
        assert np.array_equal(got.kps_left[f], el.kps[f]) and np.array_equal(got.kps_right[f], er.kps[f]), f
    assert int(np.unpackbits(got.desc_left ^ el.desc).sum()) <= 2
    assert got.n_matches == nm and np.abs(got.u_right - ur).max() <= 1e-3 and np.abs(got.depth - dp).max() <= 1e-3
    ctx.close()


@pytest.mark.parametrize("n", [3, 11])
def test_pitched_host_batch_and_sequence_equal_dense(n):
    """rows wider than the staging pitch and gaps between frames; 11 frames stream through 4 device slots"""
    lefts, rights = _pool(n, 600)
    stride, frame_stride = W + 40, (W + 40) * H + 1000
    pl, pr = _pitched(lefts, stride, frame_stride), _pitched(rights, stride, frame_stride)
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)

    dense = ctx.stereo_batch(lefts, rights)
    ob = api.StereoBatchBuffers.numpy(n, NF)
    ptrs = [ob.kps_left, ob.desc_left, ob.n_left, ob.kps_right, ob.desc_right, ob.n_right, ob.u_right, ob.depth, ob.n_matches]
    ctx.stereo_batch_ptr(n, pl.ctypes.data, pr.ctypes.data, stride, frame_stride, [a.ctypes.data for a in ptrs])
    assert np.array_equal(ob.n_left, dense.n_left) and np.array_equal(ob.n_right, dense.n_right)
    assert np.array_equal(ob.n_matches, dense.n_matches) and (ob.n_matches > 0).all()
    for f in range(n):
        a, b = ob.n_left[f], ob.n_right[f]
        assert ob.kps_left[f, :a].tobytes() == dense.kps_left[f, :a].tobytes() and ob.kps_right[f, :b].tobytes() == dense.kps_right[f, :b].tobytes()
        assert np.array_equal(ob.desc_left[f, :a], dense.desc_left[f, :a]) and np.array_equal(ob.desc_right[f, :b], dense.desc_right[f, :b])
        assert np.array_equal(ob.u_right[f, :a], dense.u_right[f, :a]) and np.array_equal(ob.depth[f, :a], dense.depth[f, :a])

    rec, gd, gn = ctx.sequence_stereo(lefts, rights)
    rec2 = np.zeros(n, ctx.record_dtype())
    gd2, gn2 = np.zeros_like(gd), np.zeros_like(gn)
    ctx.sequence_stereo_ptr(n, pl.ctypes.data, pr.ctypes.data, stride, frame_stride, None, False, rec2.ctypes.data, rec2.dtype.itemsize, False,
                            gd2.ctypes.data, gn2.ctypes.data)
    assert rec2.tobytes() == rec.tobytes()
    assert np.array_equal(gd2, gd) and np.array_equal(gn2, gn)
    assert np.array_equal(rec["n_matches"], dense.n_matches)
    ctx.close()


def test_profile_equals_device_batch():
    import torch

    n = 12  # more than one 8-frame chunk: the device batch forks onto the pipeline streams, the profile does not
    lefts, rights = _pool(n, 700)
    other_l, other_r = _pool(n, 800)
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=n)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    ol, orr = torch.from_numpy(other_l).cuda(), torch.from_numpy(other_r).cuda()
    torch.cuda.synchronize()

    def read(res):
        return (ctx.read_device(res.desc, (2 * n, NF, 32), np.uint8), ctx.read_device(res.n_matches, (n,), np.int32),
                ctx.read_device(res.u_right, (n, NF), np.float64))

    res = ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), W, W * H)
    want = read(res)
    ctx.stereo_batch_device(n, ol.data_ptr(), orr.data_ptr(), W, W * H)  # other frames in the slots
    assert not np.array_equal(read(res)[0], want[0])
    before = ctx.launch_count
    ms = ctx.profile_stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), W, W * H)
    assert ctx.launch_count - before == 7
    assert len(ms) == api.N_STAGES == 7
    assert all(np.isfinite(v) and v >= 0 for v in ms.values()), ms
    got = read(res)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    ctx.close()


@pytest.mark.parametrize("n", [1, 3])
def test_host_batch_rejects_short_stride(n):
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)
    buf = np.zeros(n * W * H, np.uint8)
    with pytest.raises(ValueError, match="stride"):
        ctx.stereo_batch_ptr(n, buf.ctypes.data, buf.ctypes.data, W - 1, W * H, [0] * 9)
    # the context stays usable
    lefts, rights = _pool(1, 900)
    assert ctx.stereo_frame(lefts[0], rights[0]).n_matches > 0
    ctx.close()
