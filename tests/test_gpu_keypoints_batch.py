"""`-m gpu`: FaceDetector.detect_batch / HandDetector.detect_batch (opb_keypoints_detect_batch) and the whole-body
helper on a B200, against the goldens of test_gpu_keypoints.py (the reference's own face_detector.py / hand_detector.py
on seeded weights): both faces in one face batch, the right and the left hand in one hand batch, at parity and at the
default comp precision.  Besides the goldens, every crop's result must not depend on its neighbours in the batch, on
the order of the batch or on chunking, and a batch of one is today's single-crop call bit for bit."""
import numpy as np
import pytest

from conftest import load_golden, pkg
from oracle import restate as R
from test_gpu_keypoints import CASES, MAP_TOL, TIE_FACTOR, _golden_list, detectors, detectors_comp  # noqa: F401

pytestmark = pytest.mark.gpu

FACES = [c for c in CASES if c[1] == "face"]
HANDS = [c for c in CASES if c[1] == "hand"]


def _img(g):
    h, w, seed = (int(v) for v in g["img_hw_seed"])
    return pkg("synthetic").procedural_image(h, w, seed=seed)


def _dets(detectors, detectors_comp, precision):
    return detectors if precision == "parity" else detectors_comp


def _engine_batch(det, kind, imgs, hand_types=None):
    """(keypoints, maps) of detect_batch's own call: maps of the (for left hands: flipped) crops the net sees."""
    import cv2
    P = pkg("entity").params
    if kind == "face":
        return det.engine.keypoints_detect_batch(imgs, P["face_inference_img_size"], P["face_heatmap_peak_thresh"],
                                                 False, return_maps=True)
    left = [t == "left" for t in hand_types]
    crops = [cv2.flip(a, 1) if lf else a for a, lf in zip(imgs, left)]
    return det.engine.keypoints_detect_batch(crops, P["hand_inference_img_size"], P["hand_heatmap_peak_thresh"], left,
                                             return_maps=True)


def _tie_check(got, ref, maps, mirror, err, what):
    """got == ref except channels whose decision is a near-tie in the maps `ref` came from (threshold margin or
    runner-up margin below TIE_FACTOR x the map error); returns the number of such flips."""
    oriented = np.ascontiguousarray(maps[:, :, ::-1]) if mirror else maps
    sm = R.gaussian_smooth(np.ascontiguousarray(oriented, np.float32))
    eps = TIE_FACTOR * max(err, 1e-6)
    flips = 0
    for c, (a, b) in enumerate(zip(got, ref)):
        mx = float(sm[c].max())
        if (a is None) != (b is None):
            assert abs(mx - np.float32(0.1)) < eps, "%s channel %d validity differs with margin %.3e" % (what, c, mx - 0.1)
            flips += 1
            continue
        if a is None:
            continue
        assert abs(float(a[2]) - float(b[2])) <= max(MAP_TOL, eps)
        if (a[0], a[1]) != (b[0], b[1]):
            assert mx - float(sm[c][a[1], a[0]]) < eps, "%s channel %d argmax differs beyond the near-tie margin" % (what, c)
            flips += 1
    return flips


def _same(a, b):
    return [None if k is None else (k[0], k[1], np.float32(k[2])) for k in a] == \
           [None if k is None else (k[0], k[1], np.float32(k[2])) for k in b]


def _cases(kind):
    return FACES if kind == "face" else HANDS


@pytest.mark.parametrize("precision", ["parity", "comp"])
@pytest.mark.parametrize("kind", ["face", "hand"])
def test_batch_against_goldens(detectors, detectors_comp, kind, precision):
    det = _dets(detectors, detectors_comp, precision)[kind]
    cases = _cases(kind)
    gs = [load_golden(name) for name, _, _ in cases]
    imgs = [_img(g) for g in gs]
    types = [t for _, _, t in cases]
    kps, maps = _engine_batch(det, kind, imgs, types)
    public = det.detect_batch(imgs) if kind == "face" else det.detect_batch(imgs, types)
    assert all(_same(a, b) for a, b in zip(public, kps))
    for (name, _, hand_type), g, img, k, m in zip(cases, gs, imgs, kps, maps):
        h, w = img.shape[:2]
        ref_maps = R.resize_bilinear_align_corners(g["heat_lo"][None], (h, w))[0][:-1]
        err = float(np.abs(m - ref_maps).max())
        print("%s %s-precision batch max abs map err %.3e" % (name, precision, err))
        assert err <= MAP_TOL
        # keypoints against the golden, near-ties allowed as in test_detector_end_to_end_parity
        flips = _tie_check(k, _golden_list(g), ref_maps, hand_type == "left", err, name)
        assert flips <= (3 if precision == "parity" else 6)
        # keypoints on the device's own maps: the oracle's peak finder, bit for bit
        full = np.concatenate([m, np.zeros((1, h, w), np.float32)])
        own = R.keypoints_from_heatmaps(np.ascontiguousarray(full[:, :, ::-1]) if hand_type == "left" else full)
        assert _same(k, own), name


@pytest.mark.parametrize("precision", ["parity", "comp"])
@pytest.mark.parametrize("name,kind,hand_type", CASES)
def test_batch_of_one_is_the_single_crop_call(detectors, detectors_comp, name, kind, hand_type, precision):
    import cv2
    det = _dets(detectors, detectors_comp, precision)[kind]
    img = _img(load_golden(name))
    if kind == "face":
        assert _same(det.detect_batch([img])[0], det(img))
    else:
        assert _same(det.detect_batch([img], hand_type)[0], det(img, hand_type=hand_type))
    kb, mb = _engine_batch(det, kind, [img], [hand_type])
    src = cv2.flip(img, 1) if hand_type == "left" else img
    P = pkg("entity").params
    ks, ms = det.engine.keypoints_detect(src, P["%s_inference_img_size" % kind], P["%s_heatmap_peak_thresh" % kind],
                                         mirror=hand_type == "left", return_maps=True)
    assert _same(kb[0], ks) and np.array_equal(mb[0], ms)


@pytest.mark.parametrize("precision", ["parity", "comp"])
def test_slots_do_not_depend_on_their_neighbours(detectors, detectors_comp, precision):
    """Within one bucket (4), a batch and its reverse give bit-identical per-crop results, and 4 copies of one crop give
    4 identical results: every image of the batch is computed on its own."""
    det = _dets(detectors, detectors_comp, precision)["face"]
    syn = pkg("synthetic")
    imgs = [_img(load_golden(n)) for n, _, _ in FACES] + [syn.procedural_image(133, 97, seed=81),
                                                           syn.procedural_image(64, 250, seed=82)]
    kf, mf = _engine_batch(det, "face", imgs)
    kr, mr = _engine_batch(det, "face", imgs[::-1])
    for i in range(4):
        assert _same(kf[i], kr[3 - i]) and np.array_equal(mf[i], mr[3 - i]), "crop %d" % i
    kc, mc = _engine_batch(det, "face", [imgs[2]] * 4)
    for i in range(1, 4):
        assert _same(kc[i], kc[0]) and np.array_equal(mc[i], mc[0]), "copy %d" % i


def test_chunking_and_launch_count(detectors_comp):
    """n = 3 and 5 fill buckets 4 and 8; n = 33 runs as a chunk of 32 and a chunk of 1, each crop giving what the batch
    of its own chunk gives.  Two n in the same bucket launch the same kernels: no per-crop launches."""
    det = detectors_comp["hand"]
    syn = pkg("synthetic")
    rs = np.random.RandomState(5)
    imgs = [syn.procedural_image(int(rs.randint(60, 200)), int(rs.randint(60, 200)), seed=100 + i) for i in range(33)]
    types = ["left" if i % 3 == 0 else "right" for i in range(33)]
    eng = det.engine

    def delta(n):
        before = eng.launch_count()
        out = det.detect_batch(imgs[:n], types[:n])
        assert len(out) == n and all(len(k) == 21 for k in out)
        return eng.launch_count() - before

    for n in (3, 5):                                   # warm buckets 4 and 8
        delta(n)
    assert delta(3) == delta(4)
    assert delta(5) == delta(8) == delta(7)
    k33, m33 = _engine_batch(det, "hand", imgs, types)
    k32, m32 = _engine_batch(det, "hand", imgs[:32], types[:32])
    k1, m1 = _engine_batch(det, "hand", imgs[32:], types[32:])
    assert len(k33) == 33
    for i in range(32):
        assert _same(k33[i], k32[i]) and np.array_equal(m33[i], m32[i]), "crop %d" % i
    assert _same(k33[32], k1[0]) and np.array_equal(m33[32], m1[0])


def _frame_and_poses():
    J = pkg("entity").JointType
    img = pkg("synthetic").procedural_image(480, 640, seed=90)
    people = [
        {J.Nose: (200, 110), J.Neck: (200, 170), J.RightShoulder: (150, 170), J.RightElbow: (130, 250),
         J.RightHand: (125, 320), J.LeftShoulder: (250, 170), J.LeftElbow: (270, 250), J.LeftHand: (280, 322),
         J.RightEye: (188, 100), J.LeftEye: (212, 100), J.RightEar: (175, 108), J.LeftEar: (225, 108),
         J.RightWaist: (170, 330), J.LeftWaist: (230, 330)},
        {J.Neck: (450, 200), J.RightShoulder: (415, 200), J.LeftShoulder: (485, 200), J.LeftHand: (510, 300),
         J.RightElbow: (405, 260), J.RightHand: (400, 315), J.RightWaist: (430, 360), J.LeftWaist: (470, 360)},
        {J.Nose: (610, 20), J.Neck: (612, 70), J.RightShoulder: (585, 72), J.LeftShoulder: (636, 70),
         J.RightElbow: (580, 130), J.RightHand: (585, 185), J.LeftEar: (625, 15)},
    ]
    P = np.zeros((len(people), 18, 3))
    for p, joints in enumerate(people):
        for j, (x, y) in joints.items():
            P[p, j] = (x, y, 2)
    return img, P


def test_whole_body_helper(detectors_comp):
    """detect_face_and_hands on hand-made poses over a procedural frame: the bboxes are those of demo.py's per-crop loop,
    the keypoints those of the per-crop calls except at near-ties (margin from the batch-vs-single map difference)."""
    import cv2
    wb = pkg("whole_body")
    PD = pkg("pose_detector").PoseDetector
    pose_det = PD.__new__(PD)                             # crop helpers only
    face, hand = detectors_comp["face"], detectors_comp["hand"]
    img, poses = _frame_and_poses()
    poses_loop = poses.copy()
    people = wb.detect_face_and_hands(img, poses, pose_det, face, hand)
    faces, hands = [], []
    for p, person_pose in enumerate(poses_loop):          # demo.py:30-57
        unit_length = pose_det.get_unit_length(person_pose)
        crop, bbox = pose_det.crop_face(img, person_pose, unit_length)
        if crop is not None:
            faces.append((p, "face", crop, bbox))
        crops = pose_det.crop_hands(img, person_pose, unit_length)
        hands += [(p, s, crops[s]["img"], crops[s]["bbox"]) for s in ("left", "right") if crops[s] is not None]
    assert np.array_equal(poses, poses_loop), "the helper moves the hand joints exactly as the loop does"
    assert len(faces) == 2 and len(hands) == 5
    assert sum(people[p][s] is not None for p in range(len(people)) for s in ("face", "left", "right")) == 7
    P = pkg("entity").params
    for kind, det, jobs in (("face", face, faces), ("hand", hand, hands)):
        types = [s for _, s, _, _ in jobs]
        kb, mb = _engine_batch(det, kind, [c for _, _, c, _ in jobs], types)
        for (p, slot, crop, bbox), k_b, m_b in zip(jobs, kb, mb):
            kps, got_bbox = people[p][slot]
            assert tuple(got_bbox) == tuple(bbox)
            assert _same(kps, k_b)
            mirror = slot == "left"
            ref, ref_maps = det.engine.keypoints_detect(cv2.flip(crop, 1) if mirror else crop,
                                                        P["%s_inference_img_size" % kind],
                                                        P["%s_heatmap_peak_thresh" % kind], mirror=mirror,
                                                        return_maps=True)
            assert _same(ref, det(crop) if kind == "face" else det(crop, hand_type=slot))
            err = float(np.abs(m_b - ref_maps).max())
            print("person %d %s: batch vs single max abs map diff %.3e" % (p, slot, err))
            _tie_check(kps, ref, ref_maps, mirror, err, "person %d %s" % (p, slot))
