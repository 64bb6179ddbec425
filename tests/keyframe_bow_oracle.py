"""Reference bytes of an orbslam2.KeyFrameData record whose bag of words is known, for tests/test_keyframe_export.py.

KeyFrame::serializeToProtobuf fills bow_vector = 10 from mBowVec and feature_vector = 11 from mFeatVec
(src/KeyFrame.cc:585-599).  The record is the plain oracle's (oracle_serialize_keyframe: fields 10 / 11 present but empty)
with those two empty fields -- the four bytes 52 00 5A 00 in front of the 54-byte pose and the map points -- replaced by:
  BowVector { map<uint32, double> words = 1 }: one entry per word in ascending word id (std::map iteration order), key and
    value always written: 0A len 08 varint(id) 11 <little-endian double>;
  FeatureVector { repeated FeatureNode nodes = 1 }, FeatureNode { uint32 node_id = 1; repeated uint32 feature_ids = 2 }:
    nodes in ascending id; node_id left out when 0 and feature_ids (packed) when empty, as proto3 does.
A plain sequential restatement written independently of the CUDA serialiser; BoW inputs in the layout of bow_transform()."""
import struct

import numpy as np


def varint(v: int) -> bytes:
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def _delimited(tag: int, payload: bytes) -> bytes:
    return bytes([tag]) + varint(len(payload)) + payload


def bow_fields(bow: dict) -> bytes:
    """fields 10 and 11 of the record, from bow_ids / bow_vals / fv_nodes / fv_start / fv_feats"""
    words = b"".join(_delimited(0x0A, b"\x08" + varint(int(w) & 0xFFFFFFFF) + b"\x11" + struct.pack("<d", float(v)))
                     for w, v in zip(bow["bow_ids"], bow["bow_vals"]))
    nodes = []
    for j, node in enumerate(bow["fv_nodes"]):
        node = int(node) & 0xFFFFFFFF
        feats = bow["fv_feats"][bow["fv_start"][j] : bow["fv_start"][j + 1]]
        body = (b"\x08" + varint(node) if node else b"")
        if len(feats):
            body += _delimited(0x12, b"".join(varint(int(f) & 0xFFFFFFFF) for f in feats))
        nodes.append(_delimited(0x0A, body))
    return _delimited(0x52, words) + _delimited(0x5A, b"".join(nodes))


def serialize_keyframe_bow(oracle, kps, desc, u_right, depth, kf_id, bounds, bow: dict, pose_rt=None, with_map_points=True) -> bytes:
    """oracle.serialize_keyframe() with bow_vector / feature_vector filled.  bounds = (min_u, min_v, max_u, max_v)"""
    rec = oracle.serialize_keyframe(kps, desc, u_right, depth, kf_id, bounds, pose_rt, with_map_points)
    n = len(np.asarray(kps))
    tail = 54 + ((2 + len(varint(10 * n)) + 10 * n) if with_map_points and n else 0)  # pose, map points
    at = len(rec) - tail - 4
    assert rec[at : at + 4] == b"\x52\x00\x5a\x00"
    return rec[:at] + bow_fields(bow) + rec[at + 4 :]
