"""Colour input (orbx_set_input_format) on the device, entry point by entry point.

The pin: a colour call equals, byte for byte, the same call on a gray context fed cv2.cvtColor of the same frames.  The
gray path is held bit-exact to the reference elsewhere (test_gpu_parity, test_oracle_vs_ref), so this carries the colour
path to the reference too.  Frames are synthetic: every channel is the synth recipe with its own seed, and a stereo pair is
shifted by one common disparity, so the conversion's rounding sees every residue.  Shapes: KITTI (1241 * 3 = 3723 bytes
per row, not a multiple of 4), TUM RGB-D and an odd 517 x 333.
"""
import cv2
import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth
from test_gpu_mono_rgbd_batches import _device_buffer

pytestmark = pytest.mark.gpu

FORMATS = {"rgb8": api.FORMAT_RGB8, "bgr8": api.FORMAT_BGR8, "rgba8": api.FORMAT_RGBA8, "bgra8": api.FORMAT_BGRA8}
CVT = {api.FORMAT_RGB8: cv2.COLOR_RGB2GRAY, api.FORMAT_BGR8: cv2.COLOR_BGR2GRAY, api.FORMAT_RGBA8: cv2.COLOR_RGBA2GRAY,
       api.FORMAT_BGRA8: cv2.COLOR_BGRA2GRAY}
SHAPES = {"kitti": (1241, 376, 2000, 8), "tum": (640, 480, 1000, 8), "odd": (517, 333, 700, 6)}
KITTI_CAM = api.Camera()
TUM_CAM = api.Camera(synth.TUM["fx"], synth.TUM["fy"], synth.TUM["cx"], synth.TUM["cy"], synth.TUM["bl"], tuple(synth.TUM["dist"]), synth.TUM["depth_scale"])


def _camera(shape):
    return TUM_CAM if shape == "tum" else KITTI_CAM


def colour_pair(h, w, seed, fmt, disparity=11, alpha="random"):
    """left / right (h, w, bpp) colour views: channel c is synth_stereo_pair with seed + 101 c, all shifted by `disparity`"""
    bpp = api.FORMAT_BPP[fmt]
    chans = [synth.synth_stereo_pair(h, w, seed + 101 * c, disparity) for c in range(3)]
    left = np.stack([c[0] for c in chans], -1)
    right = np.stack([c[1] for c in chans], -1)
    if bpp == 4:
        rng = np.random.default_rng(seed + 7)
        a = {"random": lambda: rng.integers(0, 256, (h, w, 1), dtype=np.uint8), "0": lambda: np.zeros((h, w, 1), np.uint8),
             "255": lambda: np.full((h, w, 1), 255, np.uint8)}[alpha]
        left, right = np.concatenate([left, a()], -1), np.concatenate([right, a()], -1)
    return np.ascontiguousarray(left), np.ascontiguousarray(right)


def gray(img, fmt):
    return cv2.cvtColor(img, CVT[fmt])


def _contexts(shape, fmt, **kw):
    w, h, nf, nl = SHAPES[shape]
    col = api.Context(w, h, nf, nl, 1.2, camera=_camera(shape), **kw)
    col.set_input_format(fmt)
    ref = api.Context(w, h, nf, nl, 1.2, camera=_camera(shape), **kw)
    return col, ref


def _same_stereo(a: api.StereoResult, b: api.StereoResult):
    assert a.kps_left.tobytes() == b.kps_left.tobytes() and a.kps_right.tobytes() == b.kps_right.tobytes()
    assert np.array_equal(a.desc_left, b.desc_left) and np.array_equal(a.desc_right, b.desc_right)
    assert a.u_right.tobytes() == b.u_right.tobytes() and a.depth.tobytes() == b.depth.tobytes() and a.n_matches == b.n_matches


def _same_grid(ga, gb):
    assert len(ga) == len(gb)
    for ra, rb in zip(ga, gb):
        assert all(np.array_equal(x, y) for x, y in zip(ra, rb))


def _device_results(ctx, res, n_images, n_frames, stereo):
    """the valid part of every device result array of the last *_device call"""
    N = res.n_features
    nk = ctx.read_device(res.n_kps, (n_images,), np.int32)
    kps = ctx.read_device(res.kps, (n_images, N), api.KP_DTYPE)
    kund = ctx.read_device(res.kps_und, (n_images, N), api.KP_DTYPE)
    desc = ctx.read_device(res.desc, (n_images, N, 32), np.uint8)
    out = {"n_kps": nk.tobytes()}
    for i in range(n_images):
        out[f"kps{i}"] = kps[i, : nk[i]].tobytes() + kund[i, : nk[i]].tobytes()
        out[f"desc{i}"] = desc[i, : nk[i]].tobytes()
    if n_frames:
        cells = res.grid_rows * res.grid_cols + 1
        ur = ctx.read_device(res.u_right, (n_frames, N), np.float64)
        dp = ctx.read_device(res.depth, (n_frames, N), np.float64)
        gs = ctx.read_device(res.grid_start, (n_frames, cells), np.int32)
        ge = ctx.read_device(res.grid_entries, (n_frames, N), np.uint16)
        out["n_matches"] = ctx.read_device(res.n_matches, (n_frames,), np.int32).tobytes()
        for f in range(n_frames):
            n = nk[2 * f if stereo else f]
            out[f"ur{f}"], out[f"dp{f}"] = ur[f, :n].tobytes(), dp[f, :n].tobytes()
            out[f"grid{f}"] = gs[f].tobytes() + ge[f, : gs[f, -1]].tobytes()
    return out


# ---- single pair / single frame ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("graph", [True, False], ids=["graph", "plain"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_stereo_frame_equals_gray_call(fmt, shape, graph):
    fmt = FORMATS[fmt]
    w, h = SHAPES[shape][:2]
    col, ref = _contexts(shape, fmt)
    col.set_graph(graph)
    ref.set_graph(graph)
    for seed in (3, 4):  # the second pair replays the captured graph with new input pointers
        l, r = colour_pair(h, w, seed, fmt)
        _same_stereo(col.stereo_frame(l, r), ref.stereo_frame(gray(l, fmt), gray(r, fmt)))
        _same_grid(col.get_grid(0), ref.get_grid(0))
        for side, img in ((0, l), (1, r)):
            assert np.array_equal(col.get_pyramid(side)[0], gray(img, fmt)), "level 0 is cv2.cvtColor of the input"
            for a, b in zip(col.get_pyramid(side, True), ref.get_pyramid(side, True)):
                assert np.array_equal(a, b)
    col.close()
    ref.close()


@pytest.mark.parametrize("shape", ["tum", "odd"])
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_extract_and_rgbd_frame_equal_gray_calls(fmt, shape):
    fmt = FORMATS[fmt]
    w, h = SHAPES[shape][:2]
    col, ref = _contexts(shape, fmt)
    img = colour_pair(h, w, 21, fmt)[0]
    # a row stride beyond the packed row: the host copy is pitched
    padded = np.zeros((h, w * img.shape[2] + 7), np.uint8)
    padded[:, : w * img.shape[2]] = img.reshape(h, -1)
    view = np.lib.stride_tricks.as_strided(padded, img.shape, (padded.strides[0], img.shape[2], 1))
    for src in (img, view):
        k1, d1 = col.extract(src)
        k2, d2 = ref.extract(gray(img, fmt))
        assert k1.tobytes() == k2.tobytes() and np.array_equal(d1, d2)
        assert np.array_equal(col.get_pyramid(0)[0], gray(img, fmt))
    depth = synth.synth_depth_u16(h, w, 5, synth.TUM["depth_scale"])
    a, b = col.rgbd_frame(img, depth), ref.rgbd_frame(gray(img, fmt), depth)
    for f in ("kps_raw", "kps", "desc", "u_right", "depth"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    _same_grid(col.get_grid(0), ref.get_grid(0))
    col.close()
    ref.close()


@pytest.mark.parametrize("alpha", ["0", "255", "random"])
def test_alpha_is_ignored(alpha):
    w, h = SHAPES["odd"][:2]
    col, ref = _contexts("odd", api.FORMAT_BGRA8)
    l, r = colour_pair(h, w, 8, api.FORMAT_BGRA8, alpha=alpha)
    l3, r3 = colour_pair(h, w, 8, api.FORMAT_BGR8)
    assert np.array_equal(l[..., :3], l3)
    _same_stereo(col.stereo_frame(l, r), ref.stereo_frame(gray(l3, api.FORMAT_BGR8), gray(r3, api.FORMAT_BGR8)))
    col.close()
    ref.close()


def test_switching_formats_on_one_context_equals_fresh_contexts():
    w, h = SHAPES["kitti"][:2]
    g_l, g_r = synth.synth_stereo_pair(h, w, 30, 13)
    c_l, c_r = colour_pair(h, w, 31, api.FORMAT_BGR8)
    ctx = api.Context(w, h, camera=KITTI_CAM)  # graph on (the default)
    fresh_gray = api.Context(w, h, camera=KITTI_CAM)
    fresh_bgr = api.Context(w, h, camera=KITTI_CAM)
    fresh_bgr.set_input_format(api.FORMAT_BGR8)
    first = ctx.stereo_frame(g_l, g_r)
    _same_stereo(first, fresh_gray.stereo_frame(g_l, g_r))
    epoch, bytes_gray = ctx.frame_epoch, ctx.algorithmic_bytes()
    ctx.set_input_format(api.FORMAT_BGR8)
    assert ctx.frame_epoch == epoch  # the resident frame stays
    _same_grid(ctx.get_grid(0), fresh_gray.get_grid(0))
    assert ctx.algorithmic_bytes() == bytes_gray + 2 * 2 * w * h
    _same_stereo(ctx.stereo_frame(c_l, c_r), fresh_bgr.stereo_frame(c_l, c_r))
    _same_stereo(ctx.stereo_frame(c_r, c_l), fresh_bgr.stereo_frame(c_r, c_l))
    ctx.set_input_format(api.FORMAT_GRAY8)
    assert ctx.algorithmic_bytes() == bytes_gray
    _same_stereo(ctx.stereo_frame(g_r, g_l), fresh_gray.stereo_frame(g_r, g_l))
    _same_stereo(ctx.stereo_frame(g_l, g_r), first)
    for c in (ctx, fresh_gray, fresh_bgr):
        c.close()


# ---- host batches -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["linear", "pitched"])
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_stereo_batch_equals_gray_batch(fmt, layout):
    fmt = FORMATS[fmt]
    w, h = SHAPES["kitti"][:2]
    bpp = api.FORMAT_BPP[fmt]
    n = 10  # more frames than max_batch: chunks cycle through the slots on the pipeline streams
    pairs = [colour_pair(h, w, 40 + i, fmt) for i in range(n)]
    L, R = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    col, ref = _contexts("kitti", fmt, max_batch=4)
    gl = np.stack([gray(x, fmt) for x in L])
    gr = np.stack([gray(x, fmt) for x in R])
    exp = ref.stereo_batch(gl, gr)
    if layout == "linear":
        got = col.stereo_batch(L, R)
    else:
        stride = w * bpp + 5
        fs = stride * h + 3
        bl, br = np.zeros(n * fs, np.uint8), np.zeros(n * fs, np.uint8)
        for f in range(n):
            np.lib.stride_tricks.as_strided(bl[f * fs :], (h, w * bpp), (stride, 1))[:] = L[f].reshape(h, -1)
            np.lib.stride_tricks.as_strided(br[f * fs :], (h, w * bpp), (stride, 1))[:] = R[f].reshape(h, -1)
        got = api.StereoBatchBuffers.numpy(n, col.n_features)
        col.stereo_batch_ptr(n, bl.ctypes.data, br.ctypes.data, stride, fs, [getattr(got, k).ctypes.data for k in (
            "kps_left", "desc_left", "n_left", "kps_right", "desc_right", "n_right", "u_right", "depth", "n_matches")])
    for k in ("n_left", "n_right", "n_matches"):
        assert np.array_equal(getattr(got, k), getattr(exp, k)), k
    for f in range(n):
        a, b = int(exp.n_left[f]), int(exp.n_right[f])
        assert got.kps_left[f, :a].tobytes() == exp.kps_left[f, :a].tobytes() and np.array_equal(got.desc_left[f, :a], exp.desc_left[f, :a])
        assert got.kps_right[f, :b].tobytes() == exp.kps_right[f, :b].tobytes() and np.array_equal(got.desc_right[f, :b], exp.desc_right[f, :b])
        assert got.u_right[f, :a].tobytes() == exp.u_right[f, :a].tobytes() and got.depth[f, :a].tobytes() == exp.depth[f, :a].tobytes()
    col.close()
    ref.close()


# ---- device inputs ------------------------------------------------------------------------------------------------------
DEVICE_CASES = [("odd", 1, 1), ("odd", 2, 3), ("odd", 3, 3), ("kitti", 3, 1), ("tum", 1, 3)]


@pytest.mark.parametrize("case", DEVICE_CASES, ids=[f"{s}-off{o}-pad{p}" for s, o, p in DEVICE_CASES])
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_device_entry_points_equal_gray_calls(fmt, case):
    """stereo / extract / RGB-D / profile batches read the colour frames in place at byte offset `off`, rows width * bpp + pad
    bytes apart, random bytes between rows and frames"""
    fmt = FORMATS[fmt]
    shape, off, pad = case
    w, h = SHAPES[shape][:2]
    bpp = api.FORMAT_BPP[fmt]
    mb = 3
    pairs = [colour_pair(h, w, 60 + i, fmt) for i in range(mb)]
    L, R = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    stride, fs = w * bpp + pad, (w * bpp + pad) * h + 5
    bl, pl = _device_buffer(L, stride, fs, off, 1)
    br, pr = _device_buffer(R, stride, fs, off, 2)
    GL, GR = np.stack([gray(x, fmt) for x in L]), np.stack([gray(x, fmt) for x in R])
    gbl, gpl = _device_buffer(GL, w, w * h, 0, 3)
    gbr, gpr = _device_buffer(GR, w, w * h, 0, 4)
    col, ref = _contexts(shape, fmt, max_batch=mb)
    for n in (1, mb):  # one frame is the graph path
        got = _device_results(col, col.stereo_batch_device(n, pl, pr, stride, fs), 2 * n, n, True)
        assert got == _device_results(ref, ref.stereo_batch_device(n, gpl, gpr, w, w * h), 2 * n, n, True)
    n = 2 * mb
    imgs = np.concatenate([L, R])
    bi, pi = _device_buffer(imgs, stride, fs, off, 5)
    gbi, gpi = _device_buffer(np.concatenate([GL, GR]), w, w * h, 0, 6)
    assert _device_results(col, col.extract_batch_device(n, pi, stride, fs), n, 0, False) == \
        _device_results(ref, ref.extract_batch_device(n, gpi, w, w * h), n, 0, False)
    depth = np.stack([synth.synth_depth_u16(h, w, 70 + i, synth.TUM["depth_scale"]) for i in range(n)])
    bd, pd = _device_buffer(depth, 2 * w, 2 * w * h, 0, 7)
    assert _device_results(col, col.rgbd_batch_device(n, pi, stride, fs, pd, 2 * w, 2 * w * h, api.DEPTH_U16), n, n, False) == \
        _device_results(ref, ref.rgbd_batch_device(n, gpi, w, w * h, pd, 2 * w, 2 * w * h, api.DEPTH_U16), n, n, False)
    stages = col.profile_stereo_batch_device(mb, pl, pr, stride, fs)
    assert stages["pyramid_level0"] > 0
    ref.profile_stereo_batch_device(mb, gpl, gpr, w, w * h)
    for f in range(mb):
        _same_grid(col.get_grid(f), ref.get_grid(f))
    for side in range(2 * mb):
        assert np.array_equal(col.get_pyramid(side)[0], (GL, GR)[side & 1][side >> 1])
    col.close()
    ref.close()


# ---- sequences ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("on_device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_sequence_two_local_ranks_equal_gray_sequence(fmt, on_device):
    import torch

    fmt = FORMATS[fmt]
    w, h, nf, nl = SHAPES["odd"]
    bpp = api.FORMAT_BPP[fmt]
    F = 7
    pairs = [colour_pair(h, w, 80 + i, fmt) for i in range(F)]
    L, R = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    GL, GR = np.stack([gray(x, fmt) for x in L]), np.stack([gray(x, fmt) for x in R])
    ref = api.Context(w, h, nf, nl, 1.2, camera=KITTI_CAM, max_batch=4)
    rec1, gd1, gn1 = ref.sequence_stereo(GL, GR)
    ctxs = [api.Context(w, h, nf, nl, 1.2, camera=KITTI_CAM, max_batch=2) for _ in range(2)]
    for c in ctxs:
        c.set_input_format(fmt)
    comms = api.Communicator.local(ctxs, F)
    dl = torch.from_numpy(L).cuda() if on_device else None
    dr = torch.from_numpy(R).cuda() if on_device else None
    row, frame = w * bpp, w * bpp * h
    recs = []
    for r in range(2):
        blk = api.frame_range(F, r, 2)
        rec = np.zeros(max(len(blk), 1), ctxs[r].record_dtype())
        if on_device:
            lp, rp = dl.data_ptr() + blk.start * frame, dr.data_ptr() + blk.start * frame
        else:
            lp, rp = L[blk.start :].ctypes.data, R[blk.start :].ctypes.data
        res = ctxs[r].sequence_stereo_ptr(F, lp, rp, row, frame, comms[r], on_device, rec.ctypes.data, rec.dtype.itemsize, False)
        assert (res.frame_lo, res.frame_hi) == (blk.start, blk.stop)
        recs.append(rec[: len(blk)])
        gd = ctxs[r].read_device(res.gathered_desc, (2 * res.block, nf, 32), np.uint8)
        gn = ctxs[r].read_device(res.gathered_n, (2 * res.block,), np.int32)
        if r == 1:
            assert np.array_equal(gd[:F], gd1) and np.array_equal(gn[:F], gn1)
    assert b"".join(x.tobytes() for x in recs) == rec1.tobytes()
    for c in comms:
        c.close()
    # keyframe records of one rank, from colour input, against the gray sequence's
    one = api.Context(w, h, nf, nl, 1.2, camera=KITTI_CAM, max_batch=4)
    one.set_input_format(fmt)
    exp = ref.sequence_stereo_keyframes(GL, GR)
    got = one.sequence_stereo_keyframes(L, R)
    for a, b in zip(got, exp):
        assert a.tobytes() == b.tobytes()
    for c in ctxs + [ref, one]:
        c.close()


# ---- errors before anything is enqueued ---------------------------------------------------------------------------------
def test_errors_return_before_anything_is_enqueued():
    w, h = SHAPES["odd"][:2]
    ctx = api.Context(w, h, 700, 6, 1.2, camera=KITTI_CAM, max_batch=2)
    L = ctx._L
    for bad in (-1, 5, 99):
        assert L.orbx_set_input_format(ctx._h, bad) == api.ORBX_ERR_INVALID_ARG
    assert ctx.input_format == api.FORMAT_GRAY8
    assert L.orbx_set_input_format(None, api.FORMAT_RGB8) == api.ORBX_ERR_INVALID_ARG
    ctx.set_input_format(api.FORMAT_RGB8)
    l, r = colour_pair(h, w, 90, api.FORMAT_RGB8)
    ctx.stereo_frame(l, r)
    before, epoch = ctx.launch_count, ctx.frame_epoch
    buf = np.zeros(4 * (3 * w + 8) * h, np.uint8)
    outs = [0] * 9
    for stride, fs in ((3 * w - 1, (3 * w - 1) * h), (w, w * h), (3 * w, 3 * w * (h - 1) + 3 * w - 1)):
        for n in (1, 3):
            rc = L.orbx_stereo_batch(ctx._h, n, buf.ctypes.data, buf.ctypes.data, stride, fs, *outs)
            assert rc == api.ORBX_ERR_INVALID_ARG, (stride, fs, n)
        io = api.OrbxSequenceIO(buf.ctypes.data, buf.ctypes.data, stride, fs, 0, 0, None, 0, None, None)
        res = api.OrbxSequenceResult()
        assert L.orbx_sequence_stereo(ctx._h, None, 3, api.C.byref(io), api.C.byref(res)) == api.ORBX_ERR_INVALID_ARG
    assert ctx.launch_count == before and ctx.frame_epoch == epoch
    # the smallest legal layout is accepted: stride = width * 3, frame_stride = stride * (h - 1) + width * 3
    got = api.StereoBatchBuffers.numpy(3, ctx.n_features)
    packed = np.concatenate([l.reshape(-1), r.reshape(-1), l.reshape(-1)])
    ctx.stereo_batch_ptr(3, packed.ctypes.data, packed.ctypes.data, 3 * w, 3 * w * h, [getattr(got, k).ctypes.data for k in (
        "kps_left", "desc_left", "n_left", "kps_right", "desc_right", "n_right", "u_right", "depth", "n_matches")])
    assert got.n_left[0] > 0 and np.array_equal(got.desc_left[0], got.desc_left[2])
    ctx.close()


# ---- the reference-shaped classes ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("rgb", [False, True], ids=["bgr", "rgb"])
def test_reference_classes_take_colour_frames(template_path, rgb):
    w, h = SHAPES["tum"][:2]
    fmt4 = api.FORMAT_RGBA8 if rgb else api.FORMAT_BGRA8
    l, r = colour_pair(h, w, 95, fmt4)
    cam = api.Camera(rgb=rgb)
    g = lambda x: gray(x, fmt4)
    for img in (l, np.ascontiguousarray(l[..., :3])):
        k1, d1 = api.ORBExtractor(img, 1000, 8, 1.2, template_path, 20, 7, camera=cam).extract()
        k2, d2 = api.ORBExtractor(g(l), 1000, 8, 1.2, template_path, 20, 7, camera=cam).extract()
        assert k1.tobytes() == k2.tobytes() and np.array_equal(d1, d2)
    a = api.Frame.createStereo(l[..., :3].copy(), r[..., :3].copy(), 1000, template_path, 20, 7, camera=cam)
    b = api.Frame.createStereo(g(l), g(r), 1000, template_path, 20, 7, camera=cam)
    assert a.mvFeatsLeft.tobytes() == b.mvFeatsLeft.tobytes() and a.mvDepths.tobytes() == b.mvDepths.tobytes() and a.mnN == b.mnN
    depth = synth.synth_depth_u16(h, w, 5, synth.TUM["depth_scale"])
    a = api.Frame.createRGBD(l, depth, 1000, template_path, 20, 7, dScale=synth.TUM["depth_scale"], camera=cam)
    b = api.Frame.createRGBD(g(l), depth, 1000, template_path, 20, 7, dScale=synth.TUM["depth_scale"], camera=cam)
    assert a.mvFeatsLeft.tobytes() == b.mvFeatsLeft.tobytes() and a.mvDepths.tobytes() == b.mvDepths.tobytes()
    with pytest.raises(ValueError):
        api.Frame.createStereo(l[..., :2].copy(), r[..., :2].copy(), 1000, template_path, 20, 7, camera=cam)


# ---- the C++ shim -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels,rgb", [(3, 0), (3, 1), (4, 0), (4, 1)], ids=["bgr8", "rgb8", "bgra8", "rgba8"])
def test_shim_colour_frames_equal_gray_calls(template_path, tmp_path, channels, rgb):
    import subprocess
    import test_color_input

    exe = str(tmp_path / "shim_color_main")
    test_color_input.test_shim_color_driver_compiles_and_refuses_other_types(tmp_path)  # builds `exe`
    fmt = {(3, 0): api.FORMAT_BGR8, (3, 1): api.FORMAT_RGB8, (4, 0): api.FORMAT_BGRA8, (4, 1): api.FORMAT_RGBA8}[(channels, rgb)]
    w, h, nf, nl = SHAPES["kitti"]
    l, r = colour_pair(h, w, 51, fmt)
    l.tofile(tmp_path / "l.raw")
    r.tofile(tmp_path / "r.raw")
    out = tmp_path / "out.bin"
    p = subprocess.run([exe, "stereo", str(w), str(h), str(nf), str(nl), "1.2", template_path, str(tmp_path / "l.raw"), str(tmp_path / "r.raw"), str(out),
                        str(channels), str(rgb)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    b = open(out, "rb").read()
    ref = api.Context(w, h, nf, nl, 1.2, camera=KITTI_CAM, pattern=api.load_brief_template(template_path))
    k, d = ref.extract(gray(l, fmt))
    exp = ref.stereo_frame(gray(l, fmt), gray(r, fmt))
    o = 0

    def take(n):
        nonlocal o
        o += n
        return b[o - n : o]

    def kps_desc():
        n = int(np.frombuffer(take(4), np.int32)[0])
        return take(28 * n), take(32 * n)

    assert kps_desc() == (k.tobytes(), d.tobytes())
    assert take(w * h) == gray(l, fmt).tobytes()
    assert kps_desc() == (exp.kps_left.tobytes(), exp.desc_left.tobytes())
    assert kps_desc() == (exp.kps_right.tobytes(), exp.desc_right.tobytes())
    n = len(exp.kps_left)
    assert int(np.frombuffer(take(4), np.int32)[0]) == exp.n_matches
    assert take(8 * n) == exp.u_right.tobytes() and take(8 * n) == exp.depth.tobytes() and o == len(b)
    # RGB-D on the TUM shape
    w, h, nf, nl = SHAPES["tum"]
    c = colour_pair(h, w, 52, fmt)[0]
    depth = synth.synth_depth_u16(h, w, 5, synth.TUM["depth_scale"])
    c.tofile(tmp_path / "c.raw")
    depth.tofile(tmp_path / "d.raw")
    p = subprocess.run([exe, "rgbd", str(w), str(h), str(nf), str(nl), "1.2", template_path, str(tmp_path / "c.raw"), str(tmp_path / "d.raw"), str(out),
                        str(channels), str(rgb), str(synth.TUM["depth_scale"])], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    b, o = open(out, "rb").read(), 0
    ref = api.Context(w, h, nf, nl, 1.2, camera=TUM_CAM, pattern=api.load_brief_template(template_path))
    e = ref.rgbd_frame(gray(c, fmt), depth)
    assert kps_desc() == (e.kps.tobytes(), e.desc.tobytes())
    assert int(np.frombuffer(take(4), np.int32)[0]) == int((e.depth > 0).sum())
    n = len(e.kps)
    assert take(8 * n) == e.u_right.tobytes() and take(8 * n) == e.depth.tobytes() and o == len(b)
