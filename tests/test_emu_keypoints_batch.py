"""CPU (`-m "not gpu"`): opb_keypoints_detect_batch -- N face / hand crops of different sizes in one upload, one
resize launch, one forward and one launch per post-process stage -- under the CUDA-on-CPU emulator
(tests/cuda_emu), and the host-only whole-body helper that feeds it.

The network runs at a reduced size (emulation speed, see test_emu_conv.py) and in fast precision; every stage around
it is compared bit for bit with the oracle applied to what the device itself produced: the resized network inputs of
every slot, the upsampled maps of every crop and the keypoints (mirror flag included)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import pkg
from oracle import restate as R

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "cuda_emu"))
from test_emu_conv import emu_lib, emu_native  # noqa: E402,F401  (fixtures: the emulated library, bound to _native)

THRESH = 0.1


def _hand_engine(native, wd=None):
    nm = pkg("models.HandNet")
    wd = wd if wd is not None else pkg("synthetic").he_weights(0, layers=nm.LAYERS)
    net = nm.HandNet()
    net.load_npz(wd)
    eng = native.Engine(0, pkg("pose_detector").make_opb_params(), native.PRECISION_FAST)
    eng.load_model(net)
    return eng, wd


def _device_array(ptr, dtype, shape):
    count = int(np.prod(shape))
    buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr)   # emulated device memory is host memory
    return np.frombuffer(buf, dtype).reshape(shape).copy()


def _crops(sizes, seed):
    syn = pkg("synthetic")
    return [np.ascontiguousarray(syn.procedural_image(h, w, seed=seed + i)) for i, (h, w) in enumerate(sizes)]


def test_ragged_resize_bit_exact_vs_cv2(emu_native):
    """One launch resizes crops smaller and larger than the network input, exactly its size (the identity), very wide,
    very tall and odd-sized, from one packed buffer, into the slots of the bucket-4 chain input.  (176 is the smallest
    network size the 7x7 TMA boxes admit; each emulated HandNet forward at 176 takes ~20 s.)"""
    net = 176
    eng, _ = _hand_engine(emu_native)
    crops = _crops([(37, 53), (net, net), (24, 410), (391, 17)], seed=40)
    eng.keypoints_detect_batch(crops, net, THRESH, False)
    slots = _device_array(eng.device_buffer(7), np.uint8, (4, net, net, 3))
    for i, crop in enumerate(crops):
        assert np.array_equal(slots[i], R.cv2_resize_linear_u8(crop, (net, net))), "slot %d (%dx%d)" % ((i,) + crop.shape[:2])
    assert np.array_equal(slots[1], crops[1])


def test_batch_end_to_end_vs_oracle(emu_native):
    """3 crops of different sizes (bucket 4), the middle one mirrored, through the HandNet chain at 176: maps within the
    fp16 tolerance of the oracle's forward; each crop's maps are exactly F.resize_images of its own slot of the device's
    low-resolution maps; keypoints exactly the oracle's peak finder on the returned maps, mirror applied."""
    net = 176
    eng, wd = _hand_engine(emu_native)
    crops = _crops([(120, 140), (97, 61), (190, 233)], seed=50)
    mirrors = [False, True, False]
    kps, maps = eng.keypoints_detect_batch(crops, net, THRESH, mirrors, return_maps=True)
    assert len(kps) == len(maps) == 3
    planes, kc, lo_n = eng.kp_channels - 1, eng.kp_channels, net // 8
    slots = _device_array(eng.device_buffer(7), np.uint8, (4, net, net, 3))
    lo_dev = _device_array(eng.device_buffer(1), np.float32, (4, kc, lo_n, lo_n))
    weights = {n: (wd[n + "/W"], wd[n + "/b"]) for n, _, _, _ in pkg("models.HandNet").LAYERS}
    resized = [R.cv2_resize_linear_u8(c, (net, net)) for c in crops]
    lo_ref = R.keypoint_forward(weights, np.concatenate([R.keypoint_preprocess(r) for r in resized]))
    n_valid = 0
    for i, (crop, m) in enumerate(zip(crops, mirrors)):
        h, w = crop.shape[:2]
        assert np.array_equal(slots[i], resized[i])
        assert not slots[3].any(), "the padding slot holds zeros"
        assert maps[i].shape == (planes, h, w)
        assert np.abs(maps[i] - R.resize_bilinear_align_corners(lo_ref[i:i + 1], (h, w))[0][:-1]).max() <= 1e-2
        assert np.array_equal(maps[i], R.resize_bilinear_align_corners(lo_dev[i:i + 1, :planes], (h, w))[0])
        full = np.concatenate([maps[i], np.zeros((1, h, w), np.float32)])
        ref = R.keypoints_from_heatmaps(np.ascontiguousarray(full[:, :, ::-1]) if m else full, THRESH)
        assert len(kps[i]) == planes
        for a, b in zip(kps[i], ref):
            assert (a is None) == (b is None)
            if a is not None:
                n_valid += 1
                assert (a[0], a[1]) == (b[0], b[1]) and np.float32(a[2]) == np.float32(b[2])
    assert n_valid > 0, "random-weight maps give some keypoints above the threshold; none tests nothing"


def test_argument_errors_leave_the_engine_usable(emu_native):
    native = emu_native
    eng, _ = _hand_engine(native)
    lib, ctx = eng.lib, eng.ctx
    planes = eng.kp_channels - 1
    out = np.empty((2, planes, 3), np.float64)
    valid = np.empty((2, planes), np.int32)
    dims = np.array([[20, 30], [0, 12]], np.int32)
    mirror = np.zeros(2, np.int32)
    img = np.zeros(20 * 30 * 3, np.uint8)
    p = native._ptr
    before = eng.launch_count()
    # n = 0: nothing to do, nothing launched
    assert lib.opb_keypoints_detect_batch(ctx, p(img), native.OPB_HOST, 0, p(dims), p(mirror), 128, THRESH,
                                          p(out), p(valid), None) == 0
    assert eng.keypoints_detect_batch([], 128, THRESH, False) == []
    # n < 0, a zero-size crop (named in the message), NULL arrays
    assert lib.opb_keypoints_detect_batch(ctx, p(img), native.OPB_HOST, -1, p(dims), p(mirror), 128, THRESH,
                                          p(out), p(valid), None) == native.ERR_ARG
    assert lib.opb_keypoints_detect_batch(ctx, p(img), native.OPB_HOST, 2, p(dims), p(mirror), 128, THRESH,
                                          p(out), p(valid), None) == native.ERR_ARG
    assert b"crop 1" in lib.opb_last_error(ctx)
    for args in ((None, p(dims), p(mirror)), (p(img), None, p(mirror)), (p(img), p(dims), None)):
        assert lib.opb_keypoints_detect_batch(ctx, args[0], native.OPB_HOST, 1, args[1], args[2], 128, THRESH,
                                              p(out), p(valid), None) == native.ERR_ARG
    with pytest.raises(native.OpbError, match="crop 0 has size 0x5"):
        eng.keypoints_detect_batch([np.zeros((0, 5, 3), np.uint8)], 128, THRESH, False)
    assert eng.launch_count() == before, "argument errors are found before anything is launched"
    # a pose-net context refuses the call
    pose = native.Engine(0, pkg("pose_detector").make_opb_params(), native.PRECISION_FAST)
    assert pose.lib.opb_keypoints_detect_batch(pose.ctx, p(img), native.OPB_HOST, 1, p(dims), p(mirror), 128, THRESH,
                                               p(out), p(valid), None) == native.ERR_STATE
    # the engine still works: the post-process alone, then a batch of one through the network
    maps = np.random.RandomState(3).uniform(0, 1, (planes, 23, 31)).astype(np.float32)
    full = np.concatenate([maps, np.zeros((1, 23, 31), np.float32)])
    got = eng.keypoints_from_heatmaps(maps, THRESH)
    assert [None if k is None else (k[0], k[1], np.float32(k[2])) for k in got] == \
           [None if k is None else (k[0], k[1], np.float32(k[2])) for k in R.keypoints_from_heatmaps(full, THRESH)]
    crop = _crops([(45, 38)], seed=60)[0]
    kps, m = eng.keypoints_detect_batch([crop], 176, THRESH, False, return_maps=True)
    assert len(kps) == 1 and m[0].shape == (planes, 45, 38) and np.isfinite(m[0]).all()


# ---- the whole-body helper (host only) ----------------------------------------------------------------------------
class _Recorder(object):
    def __init__(self, n_kp):
        self.calls, self.n_kp = [], n_kp

    def _result(self, img):
        return [[int(img.shape[1]), int(img.shape[0]), np.float32(0.5)]] + [None] * (self.n_kp - 1)


class _FakeFace(_Recorder):
    def __call__(self, img):
        self.calls.append(("single", img.copy(), None))
        return self._result(img)

    def detect_batch(self, imgs):
        self.calls.append(("batch", [a.copy() for a in imgs], None))
        return [self._result(a) for a in imgs]


class _FakeHand(_Recorder):
    def __call__(self, img, hand_type="right"):
        self.calls.append(("single", img.copy(), hand_type))
        return self._result(img)

    def detect_batch(self, imgs, hand_types):
        self.calls.append(("batch", [a.copy() for a in imgs], list(hand_types)))
        return [self._result(a) for a in imgs]


def _demo_loop(img, person_pose_array, pose_detector, face_detector, hand_detector):
    """The per-person loop of the reference demo.py (:30-57), drawing left out: what each detector receives."""
    faces, hands = [], []
    for person_pose in person_pose_array:
        unit_length = pose_detector.get_unit_length(person_pose)
        cropped_face_img, bbox = pose_detector.crop_face(img, person_pose, unit_length)
        if cropped_face_img is not None:
            faces.append((face_detector(cropped_face_img), bbox))
        hands_ = pose_detector.crop_hands(img, person_pose, unit_length)
        if hands_["left"] is not None:
            hands.append((hand_detector(hands_["left"]["img"], hand_type="left"), hands_["left"]["bbox"], "left"))
        if hands_["right"] is not None:
            hands.append((hand_detector(hands_["right"]["img"], hand_type="right"), hands_["right"]["bbox"], "right"))
    return faces, hands


def _poses():
    J = pkg("entity").JointType
    P = np.zeros((4, 18, 3))

    def put(p, j, x, y):
        P[p, j] = (x, y, 2)
    # 0: a full upper body in the middle of the frame
    for j, (x, y) in {J.Nose: (160, 60), J.Neck: (160, 95), J.RightShoulder: (130, 95), J.RightElbow: (120, 140),
                      J.RightHand: (118, 180), J.LeftShoulder: (190, 95), J.LeftElbow: (200, 140),
                      J.LeftHand: (205, 181), J.RightEye: (153, 53), J.LeftEye: (167, 53), J.RightEar: (145, 58),
                      J.LeftEar: (175, 58), J.RightWaist: (140, 190), J.LeftWaist: (180, 190)}.items():
        put(0, j, x, y)
    # 1: no nose (no face crop); a left hand without its elbow (crop centred on the hand itself)
    for j, (x, y) in {J.Neck: (60, 110), J.RightShoulder: (40, 110), J.LeftShoulder: (80, 110), J.LeftHand: (95, 170),
                      J.RightElbow: (33, 150), J.RightHand: (31, 187), J.RightWaist: (48, 200)}.items():
        put(1, j, x, y)
    # 2: at the top-left corner: face and hand crops off the image edge
    for j, (x, y) in {J.Nose: (6, 4), J.Neck: (8, 30), J.RightShoulder: (1, 31), J.LeftShoulder: (25, 30),
                      J.RightElbow: (2, 60), J.RightHand: (1, 89), J.LeftEar: (14, 2)}.items():
        put(2, j, x, y)
    # 3: at the bottom-right corner, both hands with elbows (hand joints move towards the elbow direction)
    for j, (x, y) in {J.Nose: (315, 235), J.Neck: (312, 215), J.RightShoulder: (300, 214), J.LeftShoulder: (318, 216),
                      J.RightElbow: (296, 228), J.RightHand: (305, 238), J.LeftElbow: (319, 232),
                      J.LeftHand: (318, 239)}.items():
        put(3, j, x, y)
    return P


def test_whole_body_helper_feeds_the_detectors_what_the_demo_loop_does():
    wb = pkg("whole_body")
    PD = pkg("pose_detector").PoseDetector
    det = PD.__new__(PD)                 # crop helpers only: no engine
    img = pkg("synthetic").procedural_image(240, 320, seed=70)
    poses_demo, poses_batch = _poses(), _poses()
    face_a, hand_a = _FakeFace(70), _FakeHand(21)
    faces, hands = _demo_loop(img, poses_demo, det, face_a, hand_a)
    face_b, hand_b = _FakeFace(70), _FakeHand(21)
    people = wb.detect_face_and_hands(img, poses_batch, det, face_b, hand_b)

    assert np.array_equal(poses_batch, poses_demo) and not np.array_equal(poses_demo, _poses()), \
        "the hand joints are moved in place exactly as the demo loop moves them"
    assert [c[0] for c in face_b.calls] == ["batch"] and [c[0] for c in hand_b.calls] == ["batch"]
    demo_faces = [c[1] for c in face_a.calls]
    assert len(face_b.calls[0][1]) == len(demo_faces) == 3
    assert all(a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b)
               for a, b in zip(face_b.calls[0][1], demo_faces))
    demo_hands, demo_types = [c[1] for c in hand_a.calls], [c[2] for c in hand_a.calls]
    assert hand_b.calls[0][2] == demo_types == ["left", "right", "left", "right", "right", "left", "right"]
    assert len(hand_b.calls[0][1]) == len(demo_hands) == 7
    assert all(a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b)
               for a, b in zip(hand_b.calls[0][1], demo_hands))
    # per person: (keypoints, bbox) in the demo loop's order, None where the loop calls nothing
    assert len(people) == 4 and people[1]["face"] is None
    got_faces = [p["face"] for p in people if p["face"] is not None]
    assert [(k, tuple(b)) for k, b in got_faces] == [(k, tuple(b)) for k, b in faces]
    got_hands = [(p[s][0], tuple(p[s][1]), s) for p in people for s in ("left", "right") if p[s] is not None]
    assert got_hands == [(k, tuple(b), s) for k, b, s in hands]
    # crops off the edge: zero-filled outside the image, bboxes reaching past it
    assert min(b[0] for _, b in faces) < 0 and max(b[3] for _, b, _ in hands) > img.shape[0]
