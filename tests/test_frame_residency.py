"""The residency rule of the frame-level consumers, entry point by entry point.

Every consumer of what a call leaves in the context's device slots is run against seven states of one KITTI-shaped context
(max_batch = 3): fresh, after a mono extract-only batch, a stereo batch, a bag-of-words transform of part of it, a second
stereo batch, a keyframe sequence with a vocabulary, and a debug quadtree run.  The consumers read by image (pyramid, FAST
corners, quadtree survivors), by frame (grid, area matchers, keyframe serialisers, BoW transform) or by the frame's bag of
words (BoW serialisers, searchByBow).  In every state each index at or past the resident end is refused with
ORBX_ERR_STATE (ValueError) and the message of the rule that refuses it, with no launch and no change of the frame epoch;
the last resident index is accepted.
"""
import types

import numpy as np
import pytest

from orb_slam2_ros2_b200 import api, synth

pytestmark = pytest.mark.gpu

MAX_BATCH = 3
CAP = 2 * MAX_BATCH  # images of the device slots; also the most frames a mono / RGB-D batch leaves
BIG = 2**31 - 2  # a per-frame index far past the slots; batched calls ask for BIG + 1 = INT_MAX frames
MSG = {"images": "no image with that index", "frames": "no frame with that index", "bow": "orbx_bow_transform"}
QS = 4  # area queries per frame


def _dev_area(e, n):
    return (n, QS, e.d_q.data_ptr(), e.d_qd.data_ptr(), 0, 0, e.d_idx.data_ptr(), e.d_dist.data_ptr(), e.d_ratio.data_ptr(), e.d_nc.data_ptr())


# (name, the rules the entry point checks in order, call(env, i)): i = the image / frame index, or n_frames - 1 for the
# batched calls
CONSUMERS = [
    ("get_pyramid", ("images",), lambda e, i: e.ctx.get_pyramid(i)),
    ("level_corners", ("images",), lambda e, i: e.ctx.level_corners(i, 0)),
    ("level_selected", ("images",), lambda e, i: e.ctx.level_selected(i, 0)),
    ("get_grid", ("frames",), lambda e, i: e.ctx.get_grid(i)),
    ("search_in_area", ("frames",), lambda e, i: e.ctx.search_in_area(e.q, e.qd, frame=i)),
    ("search_in_area_batch_device", ("frames",), lambda e, i: e.ctx.search_in_area_batch_device(*_dev_area(e, i + 1))),
    ("serialize_keyframe", ("frames",), lambda e, i: e.ctx.serialize_keyframe(7, frame=i)),
    ("serialize_keyframe_text", ("frames",), lambda e, i: e.ctx.serialize_keyframe_text(7, frame=i)),
    ("serialize_keyframes_device", ("frames",), lambda e, i: e.ctx.serialize_keyframes_device(i + 1, 7, e.d_out.data_ptr(), e.cap, e.d_sizes.data_ptr())),
    ("bow_transform", ("frames",), lambda e, i: e.ctx.bow_transform(e.V, frame=i)),
    ("bow_transform_batch_device", ("frames",), lambda e, i: e.ctx.bow_transform_batch_device(e.V, i + 1)),
    ("serialize_keyframe_bow", ("frames", "bow"), lambda e, i: e.ctx.serialize_keyframe(7, frame=i, bow=True)),
    ("serialize_keyframes_bow_device", ("frames", "bow"),
     lambda e, i: e.ctx.serialize_keyframes_bow_device(i + 1, 7, e.d_out.data_ptr(), e.cap, e.d_sizes.data_ptr())),
    ("search_by_bow", ("bow",), lambda e, i: e.ctx.search_by_bow(e.kf_bow, e.kf_desc, frame=i)),
]


@pytest.fixture(scope="module")
def frames():
    c = synth.KITTI
    return synth.synth_stereo_pool(c["height"], c["width"], 5, seed0=40)


def _env(lefts, rights):
    import torch

    c = synth.KITTI
    h, w = c["height"], c["width"]
    cam = api.Camera(c["fx"], c["fy"], c["cx"], c["cy"], c["bl"])
    e = types.SimpleNamespace(ctx=api.Context(w, h, 2000, 8, 1.2, camera=cam, max_batch=MAX_BATCH), w=w, h=h)
    e.V = api.Vocabulary(e.ctx, **synth.synth_vocabulary(10, 4, 9))
    e.dl, e.dr = torch.from_numpy(lefts).cuda(), torch.from_numpy(rights).cuda()
    e.images = torch.from_numpy(np.concatenate([lefts, rights])).cuda()
    rng = np.random.default_rng(5)
    e.q = np.zeros(QS, api.AREA_QUERY_DTYPE)
    e.q["x"], e.q["y"], e.q["radius"], e.q["max_level"] = rng.uniform(100, w - 100, QS), rng.uniform(50, h - 50, QS), 15.0, 7
    e.qd = rng.integers(0, 256, (QS, 32), dtype=np.uint8)
    e.d_q = torch.from_numpy(np.tile(e.q, CAP).view(np.uint8)).cuda()
    e.d_qd = torch.from_numpy(np.tile(e.qd, (CAP, 1))).cuda()
    e.d_idx, e.d_dist, e.d_nc = (torch.zeros((CAP, QS), dtype=torch.int32, device="cuda") for _ in range(3))
    e.d_ratio = torch.zeros((CAP, QS), dtype=torch.float32, device="cuda")
    e.cap = e.ctx.serialized_capacity_bow()
    e.d_out = torch.zeros((CAP, e.cap), dtype=torch.uint8, device="cuda")
    e.d_sizes = torch.zeros(CAP, dtype=torch.int64, device="cuda")
    # a keyframe FeatureVector of two nodes over three features
    e.kf_bow = dict(fv_nodes=np.array([1, 5], np.int32), fv_start=np.array([0, 2, 3], np.int32), fv_feats=np.array([0, 2, 1], np.int32))
    e.kf_desc = rng.integers(0, 256, (3, 32), dtype=np.uint8)
    # a corner list for the debug quadtree run on level 0 (ROI coordinates, distinct x)
    e.qt = (rng.choice(w - 43, 50, replace=False) + 3, rng.integers(3, h - 40, 50), rng.integers(1, 256, 50))
    torch.cuda.synchronize()
    return e


def _states(e, lefts, rights):
    """(state, the call that leads to it, resident end per rule after it)"""
    ctx, w, h = e.ctx, e.w, e.h
    return [
        ("fresh", lambda: None, dict(images=0, frames=0, bow=0)),
        ("extract-only batch", lambda: ctx.extract_batch_device(5, e.images.data_ptr(), w, w * h), dict(images=5, frames=0, bow=0)),
        ("stereo batch", lambda: ctx.stereo_batch_device(3, e.dl.data_ptr(), e.dr.data_ptr(), w, w * h), dict(images=6, frames=3, bow=0)),
        ("BoW of 2 of 3 frames", lambda: ctx.bow_transform_batch_device(e.V, 2), dict(images=6, frames=3, bow=2)),
        ("second stereo batch", lambda: ctx.stereo_batch_device(2, e.dl.data_ptr(), e.dr.data_ptr(), w, w * h), dict(images=4, frames=2, bow=0)),
        # 5 frames in chunks of 3 through one group of slots: the last pass over the slots stays resident, without a BoW
        ("keyframe sequence", lambda: ctx.sequence_stereo_keyframes(lefts, rights, vocab=e.V), dict(images=6, frames=3, bow=0)),
        ("debug quadtree", lambda: ctx.run_quadtree(0, *e.qt), dict(images=6, frames=0, bow=0)),
    ]


@pytest.mark.parametrize("name,rules,call", CONSUMERS, ids=[c[0] for c in CONSUMERS])
def test_consumer_refuses_what_is_not_resident(frames, name, rules, call):
    lefts, rights = frames
    e = _env(lefts, rights)
    for state, enter, resident in _states(e, lefts, rights):
        enter()
        end = min(resident[r] for r in rules)
        for i in list(range(end, CAP + 1)) + [BIG]:
            rule = next(r for r in rules if i >= resident[r])
            launches, epoch = e.ctx.launch_count, e.ctx.frame_epoch
            with pytest.raises(ValueError, match=MSG[rule]) as err:
                call(e, i)
            assert "invalid state" in str(err.value), (state, i)
            assert (e.ctx.launch_count, e.ctx.frame_epoch) == (launches, epoch), (state, i)
        if end > 0:
            call(e, end - 1)
            e.ctx.synchronize()
    e.V.close()
    e.ctx.close()
