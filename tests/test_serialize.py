"""Result serialisation (SURVEY.md section 8(f) rank 4): orbslam2.KeyFrameData wire format.

CPU: the restated schema equals the reference's proto/Keyframe.proto; the oracle's bytes equal what the protobuf runtime's
own serializer writes for the same content, and parse back to it.  GPU: the CUDA serializer's bytes equal the oracle's."""
import hashlib
import json
import os

import numpy as np
import pytest

import keyframe_proto as KP
from orb_slam2_ros2_b200 import api, synth

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# SHA-256 of the reference's proto/Keyframe.proto as KP.parse_proto_text reads it (JSON, sorted keys); the reference
# sources are not part of this repository
REF_SCHEMA_SHA256 = "2bf4cca03594e6ebdaf4b7788dda960faea2b09748354440ad399d9569f88448"


def test_restated_schema_matches_reference_proto():
    assert hashlib.sha256(json.dumps(KP.SCHEMA, sort_keys=True).encode()).hexdigest() == REF_SCHEMA_SHA256


def _message(kps, desc, ur, dp, kf_id, bounds, pose=None, with_map_points=True):
    """what KeyFrame::serializeToProtobuf (src/KeyFrame.cc:553-647) builds for a keyframe made from a fresh frame"""
    M = KP.messages()
    m = M["KeyFrameData"]()
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
    rt = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], np.float32) if pose is None else np.asarray(pose, np.float32)
    m.pose.rotation.extend(float(v) for v in rt[:9])
    m.pose.translation.extend(float(v) for v in rt[9:])
    if with_map_points:
        m.map_points.extend([-1] * len(kps))
    return m


def _cases():
    g = np.load(os.path.join(G, "small_stereo_seed0_d9.npz"))
    kps, desc, ur, dp = g["kl"], g["dl"], g["u_right"], g["depth"]
    yield "small frame", kps, desc, ur, dp, 7, (0.0, 0.0, 320.0, 240.0), None, True
    k2 = kps[:5].copy()
    k2["x"][0], k2["y"][1], k2["angle"][2], k2["octave"][3] = 0.0, 0.0, 0.0, 0  # proto3: zero scalars are not written
    k2["angle"][4], k2["octave"][4] = -0.0, -3                                   # -0.0 has a non-zero bit pattern; negative int32 takes 10 bytes
    pose = np.arange(12, dtype=np.float32) * 0.25 - 1.0
    yield "zeros", k2, desc[:5], np.array([0.0, -1, 3.5, 1e-3, 2]), np.array([-1, 0.0, 2, 7.25, 1e6]), 0, (-3.5, 0.0, 640.0, -0.0), pose, True
    yield "empty", kps[:0], desc[:0], ur[:0], dp[:0], 300, (0.0, 0.0, 1241.0, 376.0), None, True
    yield "no map points, big id", kps[:40], desc[:40], ur[:40], dp[:40], (1 << 40) + 5, (0.0, 0.0, 320.0, 240.0), None, False


def test_oracle_bytes_equal_protobuf_runtime(oracle):
    for name, kps, desc, ur, dp, kf_id, bounds, pose, wmp in _cases():
        got = oracle.serialize_keyframe(kps, desc, ur, dp, kf_id, bounds, pose, wmp)
        m = _message(kps, desc, ur, dp, kf_id, bounds, pose, wmp)
        assert got == m.SerializeToString(deterministic=True), name
        back = KP.messages()["KeyFrameData"]()
        back.ParseFromString(got)
        assert back == m and len(back.keypoints) == len(kps), name
        if len(kps):
            assert back.descriptors[len(kps) - 1].data == desc[len(kps) - 1].tobytes()
            assert back.keypoints[0].octave == int(kps["octave"][0])


def test_keyframe_list_wrapping(oracle):
    """KeyFrameList { next_id, scale_factors, repeated KeyFrameData keyframes = 3 }: records are length-delimited field 3"""
    name, kps, desc, ur, dp, kf_id, bounds, pose, wmp = next(_cases())
    rec = oracle.serialize_keyframe(kps, desc, ur, dp, kf_id, bounds, pose, wmp)
    M = KP.messages()
    lst = M["KeyFrameList"]()
    lst.next_id = 8
    lst.scale_factors.extend([1.0, 1.2])
    lst.keyframes.add().ParseFromString(rec)
    lst.keyframes.add().ParseFromString(rec)
    raw = lst.SerializeToString(deterministic=True)
    assert raw.count(rec) == 2


@pytest.mark.gpu
def test_cuda_serializer_equals_oracle(oracle):
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 2, 17)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]))
    r = ctx.stereo_frame(left, right)
    b = ctx.grid_info()[2:]
    pose = (np.arange(12, dtype=np.float32) - 3.0) / 7.0
    for kf_id, ps, wmp in [(11, None, True), (0, pose, True), ((1 << 35) + 9, pose, False)]:
        got = ctx.serialize_keyframe(kf_id, pose_rt=ps, with_map_points=wmp)
        exp = oracle.serialize_keyframe(r.kps_left, r.desc_left, r.u_right, r.depth, kf_id, b, ps, wmp)
        assert got == exp, (kf_id, len(got), len(exp))
    m = KP.messages()["KeyFrameData"]()
    m.ParseFromString(got)
    assert len(m.keypoints) == 2000 and m.id == (1 << 35) + 9 and m.descriptors[1999].data == r.desc_left[1999].tobytes()
    ctx.close()


@pytest.mark.gpu
def test_cuda_serializer_rgbd_distortion_and_small_frames(oracle):
    c = synth.TUM
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"], (0.231222, -0.28, -0.003257, -0.000105, 0.0), c["depth_scale"])
    ctx = api.Context(c["width"], c["height"], 1000, 8, 1.2, camera=cam)
    gray = synth.synth_image(c["height"], c["width"], 12)
    r = ctx.rgbd_frame(gray, synth.synth_depth_u16(c["height"], c["width"], 12, c["depth_scale"]))
    got = ctx.serialize_keyframe(3)
    exp = oracle.serialize_keyframe(r.kps, r.desc, r.u_right, r.depth, 3, ctx.grid_info()[2:], None, True)
    assert got == exp
    # an image without corners: n = 0
    r0 = ctx.rgbd_frame(np.full((c["height"], c["width"]), 90, np.uint8), np.zeros((c["height"], c["width"]), np.uint16))
    assert len(r0.kps) == 0
    assert ctx.serialize_keyframe(5) == oracle.serialize_keyframe(r0.kps, r0.desc, r0.u_right, r0.depth, 5, ctx.grid_info()[2:], None, True)
    ctx.close()


@pytest.mark.gpu
def test_cuda_serializer_batch_device(oracle):
    import torch

    c = synth.KITTI
    n = 3
    lefts, rights = synth.synth_stereo_pool(c["height"], c["width"], n, seed0=90)
    ctx = api.Context(c["width"], c["height"], 2000, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]), max_batch=n)
    host = ctx.stereo_batch(lefts, rights)
    dl, dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.stereo_batch_device(n, dl.data_ptr(), dr.data_ptr(), c["width"], c["width"] * c["height"])
    cap = ctx.serialized_capacity()
    with torch.cuda.stream(stream):
        out = torch.zeros((n, cap), dtype=torch.uint8, device="cuda")
        sizes = torch.zeros(n, dtype=torch.int64, device="cuda")
        before = ctx.launch_count
        ctx.serialize_keyframes_device(n, 100, out.data_ptr(), cap, sizes.data_ptr())
        assert ctx.launch_count - before == 1
    stream.synchronize()
    b = ctx.grid_info()[2:]
    for f in range(n):
        exp = oracle.serialize_keyframe(host.kps_left[f], host.desc_left[f], host.u_right[f], host.depth[f], 100 + f, b, None, True)
        assert bytes(out[f, : int(sizes[f])].cpu().numpy()) == exp, f
    ctx.set_stream(None)
    ctx.close()


# ---- text variant (operator<<(std::ostream &, KeyFrame &), src/KeyFrame.cc:423-533) -----------------------------------------
def _g(v) -> str:
    """std::ostream << float / double in the classic locale: printf("%g"), 6 significant digits"""
    return "%g" % float(v)


def _expected_text(kps, desc, u_right, depth, kf_id, bounds, pose, with_map_points, scales=None, next_id=None) -> bytes:
    min_u, min_v, max_u, max_v = bounds  # Context.grid_info()[2:]
    t = []
    if scales is not None:
        t.append(f"{next_id} " + "".join(_g(s) + " " for s in scales) + "\n")
    t.append(f"{kf_id} {_g(max_u)} {_g(max_v)} {_g(min_u)} {_g(min_v)}\n")
    t.append("".join(f"{_g(k['x'])} {_g(k['y'])} {int(k['octave'])} {_g(k['angle'])} {_g(u)} {_g(d)} " for k, u, d in zip(kps, u_right, depth)) + "\n")
    t.append("".join(f"{int(b)} " for b in np.asarray(desc, np.uint8).reshape(-1)) + "\n")
    t.append("\n\n")
    p = np.asarray([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], np.float32) if pose is None else np.asarray(pose, np.float32)
    t.append("".join(_g(v) + " " for v in p) + "\n")
    t.append("\n\n\n")
    t.append(("-1 " * len(kps) if with_map_points else "") + "\n")
    return "".join(t).encode()


def test_stream_formatting_rule_is_percent_g(tmp_path):
    """pins the formatting rule the text record relies on against the real thing: a C++ ostream printing floats and doubles"""
    import shutil
    import subprocess

    if not shutil.which("g++"):
        pytest.skip("no g++")
    vals = [0.0, -1.0, 1.0, 0.5, 123.456, 1241.0, 607.1928, 1e-5, 9.99999e-5, 123456.7, 999999.5, 1e6, 3.4e7, 386.1457, 359.99997, 0.1, 2.0736, 1e-7]
    src = tmp_path / "fmt.cpp"
    src.write_text("#include <iostream>\nint main(){ float f; double d; while (std::cin >> d) { f = (float)d; std::cout << f << ' ' << (double)f << '\\n'; } }\n")
    exe = tmp_path / "fmt"
    subprocess.run(["g++", "-O1", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], input="\n".join(repr(v) for v in vals), capture_output=True, text=True, check=True).stdout.split("\n")
    for v, line in zip(vals, out):
        f = np.float32(v)
        assert line == f"{_g(f)} {_g(float(f))}", (v, line)


@pytest.mark.gpu
def test_text_record_equals_stream_formatting():
    c = synth.KITTI
    left, right = synth.synth_stereo_pair(c["height"], c["width"], 4, 17)
    ctx = api.Context(c["width"], c["height"], 1500, 8, 1.2, camera=api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"]))
    r = ctx.stereo_frame(left, right)
    b = ctx.grid_info()[2:]
    pose = (np.arange(12, dtype=np.float32) - 3.0) / 7.0
    scales = [np.float32(1.2) ** 0] + [np.float32(np.float64(1.2) ** l) for l in range(1, 8)]
    got = ctx.serialize_keyframe_text(7, pose_rt=pose, with_map_points=True, scale_header_next_id=8)
    assert got == _expected_text(r.kps_left, r.desc_left, r.u_right, r.depth, 7, b, pose, True, scales, 8)
    got = ctx.serialize_keyframe_text(9)
    assert got == _expected_text(r.kps_left, r.desc_left, r.u_right, r.depth, 9, b, None, True)
    assert got.count(b"\n") == 10 and len(got.split(b"\n")[1].split()) == 6 * len(r.kps_left)
    assert ctx.serialize_keyframe_text(9, with_map_points=False).endswith(b"\n\n\n\n\n")
    ctx.close()
