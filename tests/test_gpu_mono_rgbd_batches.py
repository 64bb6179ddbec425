"""The mono and RGB-D device batches (orbx_extract_batch_device, orbx_rgbd_batch_device) frame by frame.

The single-frame calls reach these entry points with one dense image in the context's aligned staging buffer.  Here every
image of a full 2 * max_batch batch is read from caller memory at an odd base address, odd row stride and odd frame stride,
with random bytes between the rows and frames, and each image / frame is held to the parity bar of test_gpu_parity
against the CPU oracle and byte for byte against a max_batch = 1 context.  The RGB-D depth lookup is also checked on IEEE
edge values, the frame-level consumers (grid, area matcher, bag of words, keyframe serialiser) on frames past max_batch,
and the depth layout checks that run before anything is enqueued.  One stereo case covers odd device input for
orbx_stereo_batch_device.
"""
import types

import numpy as np
import pytest

import keyframe_bow_oracle as KB
from orb_slam2_ros2_b200 import api, synth
from test_bow import _same as _same_bow
from test_gpu_matchers import _same as _same_area
from test_gpu_parity import _cmp_kps

pytestmark = pytest.mark.gpu

TUM = synth.TUM
TUM_DIST = tuple(TUM["dist"])
NO_DIST = (0.0,) * 5
MILD_DIST = (0.231222, -0.28, -0.003257, -0.000105, 0.0)
DEPTH_TYPE = {np.uint16: api.DEPTH_U16, np.float32: api.DEPTH_F32}


def _device_buffer(images, stride, frame_stride, offset, seed):
    """images (n, H, W) of any dtype in one device buffer: image f at byte offset + f * frame_stride, rows `stride` bytes
    apart.  Every other byte is random, so a read outside the image changes the result.  -> (tensor, address of image 0)"""
    import torch

    n, h = images.shape[:2]
    rows = np.ascontiguousarray(images).view(np.uint8).reshape(n, h, -1)
    wb = rows.shape[2]
    assert stride >= wb and frame_stride >= (h - 1) * stride + wb
    buf = np.random.default_rng(seed).integers(0, 256, offset + (n - 1) * frame_stride + (h - 1) * stride + wb + 64, dtype=np.uint8)
    for f in range(n):
        np.lib.stride_tricks.as_strided(buf[offset + f * frame_stride :], (h, wb), (stride, 1))[:] = rows[f]
    t = torch.from_numpy(buf).cuda()
    torch.cuda.synchronize()
    return t, t.data_ptr() + offset


def _tum_camera(dist):
    return api.Camera(TUM["fx"], TUM["fy"], TUM["cx"], TUM["cy"], TUM["bl"], dist, TUM["depth_scale"])


def _grid_equal(got, exp, what):
    assert len(got) == len(exp) and len(got[0]) == len(exp[0]), what
    for i in range(len(exp)):
        for j in range(len(exp[0])):
            assert np.array_equal(got[i][j], exp[i][j]), f"{what}: cell ({i}, {j})"


# ---- orbx_extract_batch_device --------------------------------------------------------------------------------------
MONO = [("kitti", 1241, 376, 2000, 8, 1.2, 3), ("odd", 517, 333, 700, 6, 1.25, 2)]


@pytest.mark.parametrize("cfg", MONO, ids=[c[0] for c in MONO])
def test_extract_batch_device_every_image(oracle, cfg):
    import torch

    name, w, h, nf, nl, sc, mb = cfg
    n = 2 * mb  # the last image is the last slice of the TMA image dimension
    imgs = np.stack([synth.synth_image(h, w, 60 + i) for i in range(n)])
    imgs[1] = 128  # no corners at all: zero keypoints
    imgs[2] = (imgs[2].astype(np.float32) * 0.25 + 90).astype(np.uint8)  # low contrast: cells fall back to minThFAST
    assert oracle.fast_cells(imgs[2])[1] > 10
    stride, fs = w + 13, (w + 13) * h + 37
    buf, ptr = _device_buffer(imgs, stride, fs, 3, 1)
    ctx = api.Context(w, h, nf, nl, sc, max_batch=mb)
    before = ctx.launch_count
    res = ctx.extract_batch_device(n, ptr, stride, fs)
    assert ctx.launch_count - before == 5
    assert (res.n_images, res.n_frames) == (n, 0)
    nk = ctx.read_device(res.n_kps, (n,), np.int32)
    kps = ctx.read_device(res.kps, (n, nf), api.KP_DTYPE)
    desc = ctx.read_device(res.desc, (n, nf, 32), np.uint8)
    assert nk[1] == 0 and (np.delete(nk, 1) > 0).all()
    one = api.Context(w, h, nf, nl, sc)
    for i in range(n):  # e ends as the oracle of the last image
        k = nk[i]
        e = oracle.extract(imgs[i], nf, nl, sc)
        _cmp_kps(kps[i, :k], e.kps, desc[i, :k], e.desc, f"{name} image {i}")
        k1, d1 = one.extract(imgs[i])
        assert kps[i, :k].tobytes() == k1.tobytes() and desc[i, :k].tobytes() == d1.tobytes(), f"{name} image {i} vs max_batch=1"
    one.close()
    for blurred in (False, True):
        got = ctx.get_pyramid(n - 1, blurred)
        for l in range(nl):
            assert np.array_equal(got[l], e.pyr.blurred(l) if blurred else e.pyr.level(l)), f"{name} last image, level {l} blurred={blurred}"

    with pytest.raises(ValueError):
        ctx.extract_batch_device(n + 1, ptr, stride, fs)
    # extract-only images carry no frames: the frame-level consumers refuse them
    V = api.Vocabulary(ctx, **synth.synth_vocabulary(10, 4, 9))
    q = np.zeros(4, api.AREA_QUERY_DTYPE)
    for call in (lambda: ctx.get_grid(0), lambda: ctx.search_in_area(q, np.zeros((4, 32), np.uint8)), lambda: ctx.bow_transform(V),
                 lambda: ctx.serialize_keyframe(1)):
        with pytest.raises(ValueError, match="no frame with that index"):
            call()
    V.close()
    # and the context still runs an RGB-D batch on the same images
    depth = torch.zeros((2, h, w), dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    res = ctx.rgbd_batch_device(2, ptr, stride, fs, depth.data_ptr(), 2 * w, 2 * w * h, api.DEPTH_U16)
    assert np.array_equal(ctx.read_device(res.n_kps, (2,), np.int32), nk[:2])
    assert np.array_equal(ctx.read_device(res.desc, (2, nf, 32), np.uint8), desc[:2])
    assert np.array_equal(ctx.read_device(res.n_matches, (2,), np.int32), [0, 0])
    assert sum(len(cell) for row in ctx.get_grid(1) for cell in row) == 0
    ctx.close()


# ---- orbx_rgbd_batch_device -----------------------------------------------------------------------------------------
def _rgbd_inputs(n, seed0, dtype, uniform=2, no_depth=4):
    """n TUM frames: frame `uniform` has a uniform gray image, frame `no_depth` an all-zero depth image.  Valid depth pixels
    get (x + 3y) mod 7 added, so that reading a neighbouring pixel, row or frame changes the value."""
    h, w = TUM["height"], TUM["width"]
    gray = np.stack([synth.synth_image(h, w, seed0 + f) for f in range(n)])
    yy, xx = np.mgrid[0:h, 0:w]
    ramp = ((xx + 3 * yy) % 7).astype(np.uint16)
    depth = np.stack([synth.synth_depth_u16(h, w, seed0 + f, TUM["depth_scale"]) for f in range(n)])
    depth = np.where(depth > 0, depth + ramp, 0).astype(np.uint16)
    if uniform is not None:
        gray[uniform] = 90
    if no_depth is not None:
        depth[no_depth] = 0
    return gray, depth.astype(dtype)


def _rgbd_setup(dtype, dist, max_batch=3, seed0=200, **kw):
    """a TUM context and a 2 * max_batch frame RGB-D batch in pitched device memory: gray at +3 bytes with row stride W + 13
    and 37 bytes between frames, depth at +6 elements with row stride (W + 24) elements and 8 elements between frames"""
    h, w = TUM["height"], TUM["width"]
    n = 2 * max_batch
    gray, depth = _rgbd_inputs(n, seed0, dtype, **kw)
    esz = depth.itemsize
    s = types.SimpleNamespace(n=n, gray=gray, depth=depth, depth_type=DEPTH_TYPE[dtype], cam=_tum_camera(dist))
    s.gstride, s.gfs = w + 13, (w + 13) * h + 37
    s.dstride, s.dfs = (w + 24) * esz, (w + 24) * esz * h + 8 * esz
    s.gbuf, s.gptr = _device_buffer(gray, s.gstride, s.gfs, 3, seed0)
    s.dbuf, s.dptr = _device_buffer(depth, s.dstride, s.dfs, 6 * esz, seed0 + 1)
    s.ctx = api.Context(w, h, 1000, 8, 1.2, camera=s.cam, max_batch=max_batch)
    return s


def _rgbd_run(s):
    """the batch on s.ctx -> every device output, read back"""
    ctx, n, N = s.ctx, s.n, s.ctx.n_features
    before = ctx.launch_count
    res = ctx.rgbd_batch_device(n, s.gptr, s.gstride, s.gfs, s.dptr, s.dstride, s.dfs, s.depth_type)
    assert ctx.launch_count - before == 7  # the five extractor launches, the depth lookup, the grid
    assert (res.n_images, res.n_frames) == (n, n)
    return dict(n_kps=ctx.read_device(res.n_kps, (n,), np.int32), kps=ctx.read_device(res.kps, (n, N), api.KP_DTYPE),
                kps_und=ctx.read_device(res.kps_und, (n, N), api.KP_DTYPE), desc=ctx.read_device(res.desc, (n, N, 32), np.uint8),
                u_right=ctx.read_device(res.u_right, (n, N), np.float64), depth=ctx.read_device(res.depth, (n, N), np.float64),
                n_matches=ctx.read_device(res.n_matches, (n,), np.int32))


def _rgbd_check(oracle, s, out):
    """every frame of the batch: the oracle's keypoints and depth lookup, the max_batch = 1 context's bytes, the oracle's grid"""
    h, w = TUM["height"], TUM["width"]
    cam = s.cam
    one = api.Context(w, h, 1000, 8, 1.2, camera=cam)
    bounds = s.ctx.grid_info()[2:]
    for f in range(s.n):
        k = out["n_kps"][f]
        kr, ku, desc = out["kps"][f, :k], out["kps_und"][f, :k], out["desc"][f, :k]
        ur, dp = out["u_right"][f, :k], out["depth"][f, :k]
        e = oracle.extract(s.gray[f], 1000, 8, 1.2)
        _cmp_kps(kr, e.kps, desc, e.desc, f"frame {f}")
        xy = oracle.undistort_points(np.stack([e.kps["x"], e.kps["y"]], 1), cam.fx, cam.fy, cam.cx, cam.cy, np.array(cam.dist, np.float32))
        assert np.abs(ku["x"] - xy[:, 0]).max(initial=0.0) <= 1e-3 and np.abs(ku["y"] - xy[:, 1]).max(initial=0.0) <= 1e-3, f"frame {f}"
        # the device's undistorted x isolates the lookup: every step of it is one IEEE-rounded float operation
        e_ur, e_dp = oracle.rgbd_lookup(s.depth[f], cam.depth_scale, e.kps, ku, cam.bf)
        assert np.array_equal(dp, e_dp) and np.array_equal(ur, e_ur), f"frame {f}: depth lookup"
        assert out["n_matches"][f] == (dp > 0).sum(), f"frame {f}"
        r = one.rgbd_frame(s.gray[f], s.depth[f])
        for name, got, want in [("kps", kr, r.kps_raw), ("kps_und", ku, r.kps), ("desc", desc, r.desc), ("u_right", ur, r.u_right), ("depth", dp, r.depth)]:
            assert got.tobytes() == want.tobytes(), f"frame {f}: {name} vs max_batch=1"
        _grid_equal(s.ctx.get_grid(f), oracle.init_grid(ku, *bounds), f"frame {f} grid")
    one.close()
    assert out["n_kps"][2] == 0 and out["n_matches"][4] == 0 and out["n_kps"][4] > 0
    assert (out["n_matches"][[0, 1, 3, 5]] > 0).all()


@pytest.mark.parametrize("dist", [NO_DIST, TUM_DIST], ids=["nodist", "tumdist"])
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
def test_rgbd_batch_device_every_frame(oracle, dtype, dist):
    s = _rgbd_setup(dtype, dist)
    _rgbd_check(oracle, s, _rgbd_run(s))
    s.ctx.close()


EDGE_F32 = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, -1.0, 1e-45, 1e-38, np.finfo(np.float32).max, 1.0, 5208.0, 65535.0], np.float32)
EDGE_U16 = np.array([0, 1, 2, 5208, 40000, 65535], np.uint16)


@pytest.mark.parametrize("edge", [EDGE_F32, EDGE_U16], ids=["f32", "u16"])
def test_rgbd_depth_edge_values(oracle, edge):
    """IEEE behaviour without flush-to-zero, with depth scale 5208: +inf gives depth inf and uRight = x; 1e-38 scales to a
    subnormal depth (1.92e-42) with uRight = -inf; 1e-45 underflows to 0 (invalid); NaN, -0 and negatives are invalid"""
    h, w, n = TUM["height"], TUM["width"], 2
    yy, xx = np.mgrid[0:h, 0:w]
    depth = np.stack([edge[(xx + 5 * yy + f) % len(edge)] for f in range(n)])
    gray = np.stack([synth.synth_image(h, w, 80 + f) for f in range(n)])
    esz = depth.itemsize
    cam = _tum_camera(NO_DIST)
    ctx = api.Context(w, h, 1000, 8, 1.2, camera=cam, max_batch=1)
    gbuf, gptr = _device_buffer(gray, w, w * h, 0, 3)
    dbuf, dptr = _device_buffer(depth, w * esz, w * h * esz, 0, 4)
    res = ctx.rgbd_batch_device(n, gptr, w, w * h, dptr, w * esz, w * h * esz, DEPTH_TYPE[edge.dtype.type])
    N = ctx.n_features
    nk = ctx.read_device(res.n_kps, (n,), np.int32)
    kps, kps_und = ctx.read_device(res.kps, (n, N), api.KP_DTYPE), ctx.read_device(res.kps_und, (n, N), api.KP_DTYPE)
    ur, dp = ctx.read_device(res.u_right, (n, N), np.float64), ctx.read_device(res.depth, (n, N), np.float64)
    nm = ctx.read_device(res.n_matches, (n,), np.int32)
    hit = set()
    for f in range(n):
        k = nk[f]
        e_ur, e_dp = oracle.rgbd_lookup(depth[f], cam.depth_scale, kps[f, :k], kps_und[f, :k], cam.bf)
        assert np.array_equal(dp[f, :k], e_dp) and np.array_equal(ur[f, :k], e_ur), f"frame {f}"
        assert nm[f] == (e_dp > 0).sum()
        x, y = kps[f, :k]["x"].astype(np.int64), kps[f, :k]["y"].astype(np.int64)
        hit |= set(((x + 5 * y + f) % len(edge)).tolist())
    assert hit == set(range(len(edge))), "every edge value is under some keypoint"
    assert (dp > 0).any() and (dp[dp <= 0] == -1).all()
    if edge.dtype == np.float32:
        assert np.isposinf(dp).any() and np.isneginf(ur).any()
        assert ((dp > 0) & (dp < np.finfo(np.float32).tiny)).any()  # a subnormal depth survived
    ctx.close()


def test_frame_consumers_on_every_rgbd_frame(oracle):
    """grid, batched area matcher, batched and per-frame BoW, searchByBow and the keyframe serialisers on all 2 * max_batch
    frames of an RGB-D batch (one image per frame, so the frames past max_batch are resident too)"""
    import torch

    s = _rgbd_setup(np.uint16, MILD_DIST, seed0=300, uniform=None, no_depth=None)
    ctx, n, N = s.ctx, s.n, s.ctx.n_features
    h, w = TUM["height"], TUM["width"]
    out = _rgbd_run(s)
    nk, kps, desc = out["n_kps"], out["kps_und"], out["desc"]
    assert (nk > 0).all()
    bounds, sf = ctx.grid_info()[2:], ctx.scaled_factors()
    for f in (0, n - 1):
        _grid_equal(ctx.get_grid(f), oracle.init_grid(kps[f, : nk[f]], *bounds), f"frame {f} grid")

    # findFeaturesInArea + getBestMatch, one launch over all frames, a different query count per frame
    nq = 1200
    qs, qds, exs = np.zeros((n, nq), api.AREA_QUERY_DTYPE), np.zeros((n, nq, 32), np.uint8), np.zeros((n, N), np.uint8)
    nqs = np.array([nq, nq - 1, 700, 0, 333, nq], np.int32)
    for f in range(n):
        q, qd, ex, _ = synth.synth_area_queries(kps[f, : nk[f]], desc[f, : nk[f]], nq, 30 + f, w, h, 8, 15.0)
        qs[f], qds[f], exs[f, : len(ex)] = q, qd, ex
    t_q, t_d = torch.from_numpy(qs.view(np.uint8).reshape(n, -1)).cuda(), torch.from_numpy(qds).cuda()
    t_x, t_n = torch.from_numpy(exs).cuda(), torch.from_numpy(nqs).cuda()
    o_idx = torch.full((n, nq), -7, dtype=torch.int32, device="cuda")
    o_dist, o_nc = torch.zeros((n, nq), dtype=torch.int32, device="cuda"), torch.zeros((n, nq), dtype=torch.int32, device="cuda")
    o_ratio = torch.zeros((n, nq), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    before = ctx.launch_count
    ctx.search_in_area_batch_device(n, nq, t_q.data_ptr(), t_d.data_ptr(), t_n.data_ptr(), t_x.data_ptr(), o_idx.data_ptr(), o_dist.data_ptr(),
                                    o_ratio.data_ptr(), o_nc.data_ptr())
    assert ctx.launch_count - before == 1
    ctx.synchronize()
    for f in range(n):
        m, k = int(nqs[f]), nk[f]
        exp = oracle.search_in_area(kps[f, :k], desc[f, :k], bounds, sf, qs[f][:m], qds[f][:m], exs[f][:k])
        got = dict(best_idx=o_idx[f, :m].cpu().numpy(), best_dist=o_dist[f, :m].cpu().numpy(), ratio=o_ratio[f, :m].cpu().numpy(),
                   n_cand=o_nc[f, :m].cpu().numpy())
        _same_area(got, exp, f"frame {f}")
        assert (o_idx[f, m:] == -7).all()
        if m:
            assert (got["n_cand"] > 0).mean() > 0.5

    # the bag of words of every frame, batched and one frame at a time
    voc = synth.synth_vocabulary(10, 4, 9)
    O, V = oracle.Vocabulary(**voc), api.Vocabulary(ctx, **voc)
    before = ctx.launch_count
    d = ctx.bow_transform_batch_device(V, n, 4)
    assert ctx.launch_count - before == 2 and d.stride == N
    nb, nfv = ctx.read_device(d.n_bow, (n,), np.int32), ctx.read_device(d.n_fv_nodes, (n,), np.int32)
    ids, vals = ctx.read_device(d.bow_ids, (n, N), np.int32), ctx.read_device(d.bow_vals, (n, N), np.float64)
    fnodes, fstart = ctx.read_device(d.fv_nodes, (n, N), np.int32), ctx.read_device(d.fv_start, (n, N + 1), np.int32)
    ffeats = ctx.read_device(d.fv_feats, (n, N), np.int32)
    exp = [oracle.bow_transform(O, desc[f, : nk[f]], 4) for f in range(n)]
    for f in range(n):
        got = dict(bow_ids=ids[f, : nb[f]], bow_vals=vals[f, : nb[f]], fv_nodes=fnodes[f, : nfv[f]], fv_start=fstart[f, : nfv[f] + 1],
                   fv_feats=ffeats[f, : fstart[f, nfv[f]]])
        _same_bow(got, exp[f], f"batched frame {f}")
        assert len(got["bow_ids"]) > 100
    last = n - 1
    _same_bow(ctx.bow_transform(V, frame=last), exp[last], f"bow_transform(frame={last})")
    got = ctx.search_by_bow(exp[0], desc[0, : nk[0]], frame=last)
    e = oracle.search_by_bow(exp[last], desc[last, : nk[last]], exp[0], desc[0, : nk[0]])
    for key in e:
        assert np.array_equal(got[key], e[key], equal_nan=True), key
    assert len(got["kf_idx"]) > 100

    # the batched keyframe serialisers equal the per-frame records, with and without the bag of words
    for bow in (False, True):
        cap = ctx.serialized_capacity_bow() if bow else ctx.serialized_capacity()
        d_out = torch.zeros((n, cap), dtype=torch.uint8, device="cuda")
        d_sizes = torch.zeros(n, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        (ctx.serialize_keyframes_bow_device if bow else ctx.serialize_keyframes_device)(n, 500, d_out.data_ptr(), cap, d_sizes.data_ptr())
        ctx.synchronize()
        sizes, recs = d_sizes.cpu().numpy(), d_out.cpu().numpy()
        for f in range(n):
            assert recs[f, : sizes[f]].tobytes() == ctx.serialize_keyframe(500 + f, frame=f, bow=bow), f"frame {f} bow={bow}"
    # and the last frame's record (bag of words included) against the reference bytes
    k = nk[last]
    assert recs[last, : sizes[last]].tobytes() == KB.serialize_keyframe_bow(oracle, kps[last, :k], desc[last, :k], out["u_right"][last, :k],
                                                                             out["depth"][last, :k], 500 + last, bounds, exp[last])

    # a smaller batch afterwards leaves frames 2.. without a grid or a bag of words
    ctx.rgbd_batch_device(2, s.gptr, s.gstride, s.gfs, s.dptr, s.dstride, s.dfs, s.depth_type)
    q = np.zeros(4, api.AREA_QUERY_DTYPE)
    for call in (lambda: ctx.get_grid(2), lambda: ctx.bow_transform(V, frame=2), lambda: ctx.search_in_area(q, np.zeros((4, 32), np.uint8), frame=2)):
        with pytest.raises(ValueError, match="no frame with that index"):
            call()
    V.close()
    ctx.close()


def test_rgbd_batch_rejects_malformed_depth(oracle):
    """misaligned or short depth layouts are refused before anything is enqueued; the context then runs a valid batch"""
    s = _rgbd_setup(np.uint16, NO_DIST)
    h, w = TUM["height"], TUM["width"]
    bad = [
        (s.dptr, 2 * w + 1, s.dfs, api.DEPTH_U16),  # odd u16 row stride
        (s.dptr, 4 * w + 2, (4 * w + 2) * h, api.DEPTH_F32),  # f32 row stride not a multiple of 4
        (s.dptr + 1, s.dstride, s.dfs, api.DEPTH_U16),  # depth pointer at +1 byte
        (s.dptr, (w - 1) * 2, s.dfs, api.DEPTH_U16),  # rows shorter than the image
        (s.dptr, s.dstride, s.dstride * (h - 1) + 2 * w - 2, api.DEPTH_U16),  # frame stride one element short
    ]
    before = s.ctx.launch_count
    for ptr, stride, fs, dt in bad:
        with pytest.raises(ValueError, match="depth"):
            s.ctx.rgbd_batch_device(s.n, s.gptr, s.gstride, s.gfs, ptr, stride, fs, dt)
    assert s.ctx.launch_count == before
    _rgbd_check(oracle, s, _rgbd_run(s))
    s.ctx.close()


# ---- orbx_stereo_batch_device ---------------------------------------------------------------------------------------
def test_stereo_batch_device_odd_input():
    """left and right at odd base addresses, odd row stride and odd frame stride: the level-0 pyramid kernel's reads of
    the caller's rows must give the results of the dense host batch"""
    c = synth.KITTI
    h, w, n, N = c["height"], c["width"], 4, 2000
    lefts, rights = synth.synth_stereo_pool(h, w, n, seed0=140)
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    ctx = api.Context(w, h, N, 8, 1.2, camera=cam, max_batch=n)
    host = ctx.stereo_batch(lefts, rights)
    stride, fs = w + 13, (w + 13) * h + 37
    lbuf, lp = _device_buffer(lefts, stride, fs, 3, 11)
    rbuf, rp = _device_buffer(rights, stride, fs, 5, 12)
    before = ctx.launch_count
    res = ctx.stereo_batch_device(n, lp, rp, stride, fs)
    assert ctx.launch_count - before == 7
    nk = ctx.read_device(res.n_kps, (2 * n,), np.int32)
    kps, kps_und = ctx.read_device(res.kps, (2 * n, N), api.KP_DTYPE), ctx.read_device(res.kps_und, (2 * n, N), api.KP_DTYPE)
    desc = ctx.read_device(res.desc, (2 * n, N, 32), np.uint8)
    ur, dp = ctx.read_device(res.u_right, (n, N), np.float64), ctx.read_device(res.depth, (n, N), np.float64)
    assert np.array_equal(nk[0::2], host.n_left) and np.array_equal(nk[1::2], host.n_right)
    assert np.array_equal(ctx.read_device(res.n_matches, (n,), np.int32), host.n_matches) and (host.n_matches > 500).all()
    for f in range(n):
        a, b = host.n_left[f], host.n_right[f]
        assert kps_und[2 * f, :a].tobytes() == host.kps_left[f, :a].tobytes() and kps[2 * f + 1, :b].tobytes() == host.kps_right[f, :b].tobytes(), f
        assert np.array_equal(desc[2 * f, :a], host.desc_left[f, :a]) and np.array_equal(desc[2 * f + 1, :b], host.desc_right[f, :b]), f
        assert np.array_equal(ur[f, :a], host.u_right[f, :a]) and np.array_equal(dp[f, :a], host.depth[f, :a]), f
    ctx.close()
