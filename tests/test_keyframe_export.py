"""Offline map export: keyframe records that carry their bag of words, from single frames, device batches and sharded
sequences, framed as one orbslam2.KeyFrameList (proto/Keyframe.proto:45-70; writers src/KeyFrame.cc:553-647,585-599 and
src/Map.cc:205-224).

CPU: the reference bytes of tests/keyframe_bow_oracle.py parse to the message the protobuf runtime builds for the same content; outside field 10 they are
the runtime's deterministic bytes, inside it the same map entries (ours in ascending word id, std::map order; upb writes
them in descending order, so field 10 is compared entry by entry).  GPU: the CUDA serialiser equals the oracle; the
keyframe sequence equals the per-frame calls and leaves the raw records and the gather untouched; two ranks concatenate
to the single-rank KeyFrameList.  The BoW content itself is parity-unpinned (DESIGN section 2)."""
import io
import os

import numpy as np
import pytest

import keyframe_bow_oracle as KB
import keyframe_proto as KP
from orb_slam2_ros2_b200 import api, synth

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---- wire-format helpers ----------------------------------------------------------------------------------------------
def _varint(b: bytes, i: int):
    v, s = 0, 0
    while True:
        x = b[i]
        i += 1
        v |= (x & 0x7F) << s
        s += 7
        if x < 0x80:
            return v, i


def _fields(b: bytes):
    """top-level fields of a message -> [(number, raw bytes of the whole field, payload)]"""
    out, i = [], 0
    while i < len(b):
        j = i
        tag, i = _varint(b, i)
        wt = tag & 7
        if wt == 0:
            _, i = _varint(b, i)
            payload = b[j:i]
        elif wt == 1:
            payload, i = b[i : i + 8], i + 8
        elif wt == 5:
            payload, i = b[i : i + 4], i + 4
        else:
            assert wt == 2, wt
            n, i = _varint(b, i)
            payload, i = b[i : i + n], i + n
        out.append((tag >> 3, b[j:i], payload))
    return out


def _message(kps, desc, ur, dp, kf_id, bounds, bow, pose=None, with_map_points=True):
    """what KeyFrame::serializeToProtobuf builds for a keyframe with mBowVec / mFeatVec = bow"""
    m = KP.messages()["KeyFrameData"]()
    m.id = kf_id
    m.min_u, m.min_v, m.max_u, m.max_v = (float(b) for b in bounds)
    for i in range(len(kps)):
        k = m.keypoints.add()
        k.x, k.y, k.octave, k.angle = float(kps["x"][i]), float(kps["y"][i]), int(kps["octave"][i]), float(kps["angle"][i])
        m.right_u.append(float(np.float32(ur[i])))
        m.depths.append(float(np.float32(dp[i])))
    for i in range(len(kps)):
        m.descriptors.add().data = desc[i].tobytes()
    m.bow_vector.SetInParent()
    m.feature_vector.SetInParent()
    for w, v in zip(bow["bow_ids"], bow["bow_vals"]):
        m.bow_vector.words[int(w)] = float(v)
    for j, node in enumerate(bow["fv_nodes"]):
        nd = m.feature_vector.nodes.add()
        nd.node_id = int(node)
        nd.feature_ids.extend(int(f) for f in bow["fv_feats"][bow["fv_start"][j] : bow["fv_start"][j + 1]])
    rt = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], np.float32) if pose is None else np.asarray(pose, np.float32)
    m.pose.rotation.extend(float(v) for v in rt[:9])
    m.pose.translation.extend(float(v) for v in rt[9:])
    if with_map_points:
        m.map_points.extend([-1] * len(kps))
    return m


def _bow(ids, vals, nodes, feats):
    fs = np.concatenate([[0], np.cumsum([len(f) for f in feats])]).astype(np.int32)
    return dict(bow_ids=np.asarray(ids, np.int32), bow_vals=np.asarray(vals, np.float64), fv_nodes=np.asarray(nodes, np.int32), fv_start=fs,
                fv_feats=np.asarray([x for f in feats for x in f], np.int32))


def _cases(oracle):
    g = np.load(os.path.join(G, "small_stereo_seed0_d9.npz"))
    kps, desc, ur, dp = g["kl"], g["dl"], g["u_right"], g["depth"]
    b = (0.0, 0.0, 320.0, 240.0)
    for k, L, levelsup in [(10, 3, 2), (6, 4, 4), (10, 2, 4)]:  # the last: levelsup >= L, every feature under node 0
        V = oracle.Vocabulary(**synth.synth_vocabulary(k, L, 5))
        yield f"golden k{k} L{L} up{levelsup}", kps, desc, ur, dp, 9, b, oracle.bow_transform(V, desc, levelsup), None, True
    # ids with 1- to 5-byte varints (word 0, node 0, >= 2^21), features >= 128 and >= 16384, a node without node_id
    big = _bow([0, 1, 127, 128, 16383, 16384, (1 << 21) - 1, 1 << 21, (1 << 28) + 3, (1 << 31) - 1],
               [0.5, 1e-300, 0.0, 1.0, 0.25, 3.0, 1e300, 2.5e-5, 0.125, 7.0],
               [0, 5, 200, 1 << 21, (1 << 28) + 1], [[0, 3], [1], [127, 128, 300, 16383, 16384, 40000], list(range(130)), [65535]])
    pose = np.arange(12, dtype=np.float32) * 0.25 - 1.0
    yield "wide ids", kps[:40], desc[:40], ur[:40], dp[:40], (1 << 40) + 5, b, big, pose, False
    yield "empty bow", kps[:7], desc[:7], ur[:7], dp[:7], 0, b, _bow([], [], [], []), None, True
    yield "empty frame", kps[:0], desc[:0], ur[:0], dp[:0], 3, b, _bow([0], [1.0], [0], [[]]), None, True


def _check_against_runtime(got: bytes, m, name):
    back = KP.messages()["KeyFrameData"]()
    back.ParseFromString(got)
    assert back == m, name
    exp = m.SerializeToString(deterministic=True)
    fg, fe = _fields(got), _fields(exp)
    assert [(n, raw) for n, raw, _ in fg if n != 10] == [(n, raw) for n, raw, _ in fe if n != 10], name
    (bg,), (be,) = [p for n, _, p in fg if n == 10], [p for n, _, p in fe if n == 10]
    eg, ee = [raw for _, raw, _ in _fields(bg)], [raw for _, raw, _ in _fields(be)]
    assert sorted(eg) == sorted(ee), name
    keys = [_entry_key(p) for _, _, p in _fields(bg)]
    assert keys == sorted(keys) and len(set(keys)) == len(keys), name


def _entry_key(entry: bytes) -> int:
    key = [p for n, _, p in _fields(entry) if n == 1]
    return _varint(key[0], 1)[0] if key else 0  # payload of a varint field = tag byte + value


def test_oracle_bow_record_equals_protobuf_runtime(oracle):
    for name, kps, desc, ur, dp, kf_id, bounds, bow, pose, wmp in _cases(oracle):
        got = KB.serialize_keyframe_bow(oracle, kps, desc, ur, dp, kf_id, bounds, bow, pose, wmp)
        m = _message(kps, desc, ur, dp, kf_id, bounds, bow, pose, wmp)
        _check_against_runtime(got, m, name)
        assert len(m.bow_vector.words) == len(bow["bow_ids"]) and len(m.feature_vector.nodes) == len(bow["fv_nodes"])
        if len(bow["bow_ids"]) == 0 and len(bow["fv_nodes"]) == 0:  # no BoW: the record of a fresh frame
            assert got == oracle.serialize_keyframe(kps, desc, ur, dp, kf_id, bounds, pose, wmp)


def test_keyframe_list_of_bow_records(oracle):
    """KeyFrameList framing: head (next_id, packed scale factors) + length-delimited records == the runtime's list"""
    cases = list(_cases(oracle))
    recs = [KB.serialize_keyframe_bow(oracle, *c[1:7], c[7], c[8], c[9]) for c in cases]
    scales = oracle.scale_factors(1.2, 8)
    lst = KP.messages()["KeyFrameList"]()
    lst.next_id = 12
    lst.scale_factors.extend(float(s) for s in scales)
    for r in recs:
        lst.keyframes.add().ParseFromString(r)
    raw = lst.SerializeToString(deterministic=True)
    head = bytes([0x08, 12, 0x12, 32]) + np.asarray(scales, np.float32).tobytes()
    assert raw.startswith(head)
    back = KP.messages()["KeyFrameList"]()
    back.ParseFromString(head + b"".join(bytes([0x1A]) + KB.varint(len(r)) + r for r in recs))
    assert back == lst


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _kitti_ctx(max_batch=1):
    c = synth.KITTI
    return api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=max_batch)


@pytest.mark.gpu
def test_cuda_bow_serializer_equals_oracle(oracle):
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 2, 17)
    ctx = _kitti_ctx()
    r = ctx.stereo_frame(left, right)
    assert len(r.kps_left) == 2000
    b = ctx.grid_info()[2:]
    cap = ctx.serialized_capacity_bow()
    assert cap % 16 == 0 and cap > ctx.serialized_capacity()
    with pytest.raises(ValueError, match="bow_transform"):
        ctx.serialize_keyframe(1, bow=True)  # ORBX_ERR_STATE: no BoW resident
    pose = (np.arange(12, dtype=np.float32) - 3.0) / 7.0
    for (k, L, seed), levelsup in [((10, 6, 1), 4), ((10, 3, 2), 4), ((6, 4, 3), 2)]:  # ORBvoc.txt's shape; everything under node 0; nodes at level 2
        V = api.Vocabulary(ctx, **synth.synth_vocabulary(k, L, seed))
        bow = ctx.bow_transform(V, levelsup=levelsup)
        for kf_id, ps, wmp in [(11, None, True), (0, pose, True), ((1 << 35) + 9, pose, False)]:
            got = ctx.serialize_keyframe(kf_id, pose_rt=ps, with_map_points=wmp, bow=True)
            exp = KB.serialize_keyframe_bow(oracle, r.kps_left, r.desc_left, r.u_right, r.depth, kf_id, b, bow, ps, wmp)
            assert got == exp, (k, L, levelsup, kf_id, len(got), len(exp))
            assert len(got) <= cap
        m = KP.messages()["KeyFrameData"]()
        m.ParseFromString(got)
        assert len(m.bow_vector.words) == len(bow["bow_ids"]) > 0 and len(m.feature_vector.nodes) == len(bow["fv_nodes"])
        if k == 10 and L == 6:
            assert bow["bow_ids"].max() >= 1 << 14  # 3-byte word ids
        V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_bow_serializer_rgbd_distortion(oracle):
    c = synth.TUM
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], (0.231222, -0.28, -0.003257, -0.000105, 0.0), c["depth_scale"])
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam)
    gray = synth.synth_image(c["height"], c["width"], 12)
    r = ctx.rgbd_frame(gray, synth.synth_depth_u16(c["height"], c["width"], 12, c["depth_scale"]))
    V = api.Vocabulary(ctx, **synth.synth_vocabulary(10, 5, 4))
    bow = ctx.bow_transform(V)
    got = ctx.serialize_keyframe(3, bow=True)
    assert got == KB.serialize_keyframe_bow(oracle, r.kps, r.desc, r.u_right, r.depth, 3, ctx.grid_info()[2:], bow, None, True)
    assert len(got) <= ctx.serialized_capacity_bow()
    V.close()
    ctx.close()


@pytest.mark.gpu
def test_cuda_bow_serializer_batch_device_equals_per_frame(oracle):
    import torch

    c = synth.KITTI
    n = 3
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=90)
    ctx = _kitti_ctx(max_batch=n)
    V = api.Vocabulary(ctx, **synth.synth_vocabulary(10, 6, 1))
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    torch.cuda.synchronize()
    ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    cap = ctx.serialized_capacity_bow()
    out = torch.zeros((n, cap), dtype=torch.uint8, device="cuda")
    sizes = torch.zeros(n, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError, match="bow_transform"):
        ctx.serialize_keyframes_bow_device(n, 100, out.data_ptr(), cap, sizes.data_ptr())
    ctx.bow_transform_batch_device(V, n)
    with pytest.raises(ValueError, match="capacity"):
        ctx.serialize_keyframes_bow_device(n, 100, out.data_ptr(), ctx.serialized_capacity(), sizes.data_ptr())
    before = ctx.launch_count
    ctx.serialize_keyframes_bow_device(n, 100, out.data_ptr(), cap, sizes.data_ptr())
    assert ctx.launch_count - before == 1
    ctx.synchronize()
    dev = [bytes(out[f, : int(sizes[f])].cpu().numpy()) for f in range(n)]
    per_frame = [ctx.serialize_keyframe(100 + f, frame=f, bow=True) for f in range(n)]
    assert dev == per_frame and max(len(x) for x in dev) <= cap
    host = ctx.stereo_batch(lefts, rights)  # the same frames again, for the oracle's inputs
    b = ctx.grid_info()[2:]
    for f in range(n):
        bow = ctx.bow_transform(V, frame=f)
        assert dev[f] == KB.serialize_keyframe_bow(oracle, host.kps_left[f], host.desc_left[f], host.u_right[f], host.depth[f], 100 + f, b, bow, None, True), f
    V.close()
    ctx.close()


H, W, NF, NL = 240, 320, 300, 5
CAM = api.Camera(300.0, 300.0, 160.0, 120.0, 0.1)
VOC = dict(k=10, L=5, seed=7)  # levelsup 4: FeatureVector nodes at level 1


def _pool(F, seed0):
    return synth.synth_stereo_pool(H, W, F, seed0=seed0, disparity=9)


def _per_frame_records(lefts, rights, id0, poses, with_vocab, with_map_points=True):
    one = api.Context(W, H, NF, NL, 1.2, camera=CAM)
    V = api.Vocabulary(one, **synth.synth_vocabulary(**VOC)) if with_vocab else None
    out = []
    for f in range(len(lefts)):
        one.stereo_frame(lefts[f], rights[f])
        if V is not None:
            one.bow_transform(V)
        out.append(one.serialize_keyframe(id0 + f, pose_rt=None if poses is None else poses[f], with_map_points=with_map_points, bow=V is not None))
    if V is not None:
        V.close()
    one.close()
    return out


@pytest.mark.gpu
def test_single_rank_keyframe_sequence():
    import torch

    F, ID0 = 11, 1000
    lefts, rights = _pool(F, 500)
    poses = (np.arange(F * 12, dtype=np.float32).reshape(F, 12) - 40.0) / 13.0
    ctx = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)  # 11 frames through 4 device slots (chunks of 4, 4, 3)
    V = api.Vocabulary(ctx, **synth.synth_vocabulary(**VOC))
    l0 = ctx.launch_count
    rec0, gd0, gn0 = ctx.sequence_stereo(lefts, rights)
    plain = ctx.launch_count - l0
    l0 = ctx.launch_count
    rec, gd, gn, kf, sizes = ctx.sequence_stereo_keyframes(lefts, rights, vocab=V, id0=ID0, poses=poses)
    assert ctx.launch_count - l0 == plain + 3 * 3  # BoW descent, assembly and serialiser per chunk
    assert rec.tobytes() == rec0.tobytes() and np.array_equal(gd, gd0) and np.array_equal(gn, gn0)
    exp = _per_frame_records(lefts, rights, ID0, poses, True)
    assert [kf[f, : sizes[f]].tobytes() for f in range(F)] == exp
    assert sizes.max() <= kf.shape[1] == ctx.serialized_capacity_bow()
    kfd = KP.messages()["KeyFrameData"]()
    kfd.ParseFromString(exp[4])
    assert kfd.id == ID0 + 4 and len(kfd.bow_vector.words) > 0 and list(kfd.pose.rotation) == [float(x) for x in poses[4, :9]]
    # the BoW results of a sequence are not kept resident
    one = api.Context(W, H, NF, NL, 1.2, camera=CAM)
    one.stereo_frame(lefts[0], rights[0])
    V1 = api.Vocabulary(one, **synth.synth_vocabulary(**VOC))
    kb = one.bow_transform(V1)
    r1 = one.stereo_frame(lefts[0], rights[0])
    with pytest.raises(ValueError, match="bow_transform"):
        ctx.search_by_bow(kb, r1.desc_left)
    # without a vocabulary: the plain records of orbx_serialize_keyframe
    _, _, _, kf2, sizes2 = ctx.sequence_stereo_keyframes(lefts, rights, id0=ID0, poses=poses, with_map_points=False)
    assert kf2.shape[1] == ctx.serialized_capacity()
    assert [kf2[f, : sizes2[f]].tobytes() for f in range(F)] == _per_frame_records(lefts, rights, ID0, poses, False, False)
    # device inputs and device outputs (records, keyframes, sizes, poses)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    rs, ks = ctx.record_layout().record_bytes, ctx.serialized_capacity_bow()
    d_rec = torch.zeros((F, rs), dtype=torch.uint8, device="cuda")
    d_kf = torch.zeros((F, ks), dtype=torch.uint8, device="cuda")
    d_sz = torch.zeros(F, dtype=torch.int64, device="cuda")
    d_pose = torch.from_numpy(poses).cuda()
    torch.cuda.synchronize()
    ctx.sequence_stereo_keyframes_ptr(F, dl.data_ptr(), dr.data_ptr(), W, W * H, d_kf.data_ptr(), ks, d_sz.data_ptr(), V, 4, ID0, True, d_pose.data_ptr(),
                                      True, None, True, d_rec.data_ptr(), rs, True)
    assert d_rec.cpu().numpy().tobytes() == rec0.tobytes()
    szh = d_sz.cpu().numpy()
    assert np.array_equal(szh, sizes) and [bytes(d_kf[f, : szh[f]].cpu().numpy()) for f in range(F)] == exp
    # input checks
    kfh, szb = api._aligned_zeros((F, ks)), np.zeros(F, np.int64)
    args = (F, lefts.ctypes.data, rights.ctypes.data, W, W * H)
    with pytest.raises(ValueError, match="capacity"):
        ctx.sequence_stereo_keyframes_ptr(*args, kfh.ctypes.data, ks - 16, szb.ctypes.data, V)
    with pytest.raises(ValueError, match="16"):
        ctx.sequence_stereo_keyframes_ptr(*args, kfh.ctypes.data, ks + 8, szb.ctypes.data, V)
    with pytest.raises(ValueError, match="another context"):
        ctx.sequence_stereo_keyframes_ptr(*args, kfh.ctypes.data, ks, szb.ctypes.data, V1)
    for o in (V1, one, V, ctx):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("F", [11, 2, 1])
def test_two_local_ranks_form_one_keyframe_list(F):
    ID0 = 7
    lefts, rights = _pool(F, 600)
    ref = api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=4)
    Vr = api.Vocabulary(ref, **synth.synth_vocabulary(**VOC))
    _, gd1, gn1, kf1, sz1 = ref.sequence_stereo_keyframes(lefts, rights, vocab=Vr, id0=ID0)
    single = io.BytesIO()
    api.write_keyframe_list(single, ref, kf1, sz1, ID0 + F)
    ctxs = [api.Context(W, H, NF, NL, 1.2, camera=CAM, max_batch=2) for _ in range(2)]
    vocs = [api.Vocabulary(c, **synth.synth_vocabulary(**VOC)) for c in ctxs]
    comms = api.Communicator.local(ctxs, F)
    parts = []
    for r in range(2):
        blk = api.frame_range(F, r, 2)
        _, gd, gn, kf, sz = ctxs[r].sequence_stereo_keyframes(lefts[blk.start : blk.stop], rights[blk.start : blk.stop], vocab=vocs[r], id0=ID0, comm=comms[r],
                                                             n_frames_total=F)
        if r == 1:  # the gathered arrays are complete once every rank's call has returned
            assert np.array_equal(gd, gd1) and np.array_equal(gn, gn1)
        buf = io.BytesIO()
        api.write_keyframe_list(buf, ctxs[r], kf, sz, ID0 + F, head=r == 0)
        parts.append(buf.getvalue())
    whole = b"".join(parts)
    assert whole == single.getvalue()
    lst = KP.messages()["KeyFrameList"]()
    lst.ParseFromString(whole)
    assert lst.next_id == ID0 + F and [k.id for k in lst.keyframes] == list(range(ID0, ID0 + F))
    assert np.array_equal(np.asarray(lst.scale_factors, np.float32), ref.scaled_factors())
    assert all(len(k.bow_vector.words) > 0 for k in lst.keyframes)
    for o in comms + vocs + ctxs + [Vr, ref]:
        o.close()
