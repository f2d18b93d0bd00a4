"""`not gpu`: the C-ABI library loads and exports every symbol include/opb.h declares; the
POD structs of the Python binding have the sizes the header documents; constructing the
product without a GPU fails loudly (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, pkg


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "opb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(opb_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    native = pkg("_native")
    if not os.path.isfile(native.LIB_PATH):
        pkg("_build").build_native()
    lib = native.load_library()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), "libopb.so does not export " + name
    assert sorted(native.exported_symbols()) == declared
    assert lib.opb_version() == 1


def test_struct_sizes_match_header():
    native = pkg("_native")
    assert native.PERSON_DTYPE.itemsize == 240
    assert native.HEADER_DTYPE.itemsize == 16
    # limbs 152 + 6 doubles 48 + 4 ints 16 + taps 512 + 4 ints 16
    assert ctypes.sizeof(native.OpbParams) == 19 * 2 * 4 + 6 * 8 + 4 * 4 + 64 * 8 + 4 * 4


def test_params_struct_matches_entity_and_scipy_taps():
    from scipy.ndimage._filters import _gaussian_kernel1d
    p = pkg("pose_detector").make_opb_params()
    ent = pkg("entity")
    assert [[p.limbs[i][0], p.limbs[i][1]] for i in range(19)] == [[int(a), int(b)] for a, b in ent.params["limbs_point"]]
    assert p.gauss_radius == 10
    assert np.array_equal(np.array(p.gauss_taps[:21]), _gaussian_kernel1d(2.5, 0, 10))
    assert (p.heatmap_peak_thresh, p.inner_product_thresh, p.n_integ_points, p.n_integ_points_thresh) == (0.05, 0.05, 10, 8)


def test_entity_matches_reference_values():
    """entity.params / JointType carry the reference's values (entity.py:9-46,71-105)."""
    from oracle import restate as R
    ent = pkg("entity")
    assert tuple((int(a), int(b)) for a, b in ent.params["limbs_point"]) == R.LIMBS
    assert len(ent.JointType) == 18 and ent.JointType.Nose == 0 and ent.JointType.LeftEar == 17
    for k, v in dict(inference_img_size=368, heatmap_size=320, gaussian_sigma=2.5, n_integ_points=10,
                     n_integ_points_thresh=8, heatmap_peak_thresh=0.05, inner_product_thresh=0.05,
                     limb_length_ratio=1.0, length_penalty_value=1, n_subset_limbs_thresh=3,
                     subset_score_thresh=0.2, downscale=8).items():
        assert ent.params[k] == v
    assert ent.params["inference_scales"] == [0.5, 1, 1.5, 2]


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CPU fallback|no CUDA device"):
        pkg("pose_detector").PoseDetector("posenet", None)


def test_host_helpers_match_oracle():
    """compute_optimal_size / pad_image / preprocess are host NumPy in both worlds."""
    from oracle import restate as R
    PD = pkg("pose_detector").PoseDetector
    det = PD.__new__(PD)          # no engine needed for the host helpers
    rs = np.random.RandomState(0)
    for h, w in ((368, 656), (480, 640), (584, 584), (640, 480), (333, 517), (1080, 1920), (100, 37)):
        img = rs.randint(0, 255, (h, w, 3)).astype(np.uint8)
        for size in (368, 320):
            assert det.compute_optimal_size(img, size) == R.compute_optimal_size(img, size)
        a, pa = det.pad_image(img, 8, (104, 117, 123))
        b, pb = R.pad_image(img, 8, (104, 117, 123))
        assert np.array_equal(a, b) and list(pa) == list(pb)
        assert np.array_equal(det.preprocess(img), R.preprocess(img))


def test_pose_array_and_unit_length_helpers():
    from oracle import restate as R
    PD = pkg("pose_detector").PoseDetector
    det = PD.__new__(PD)
    peaks = np.zeros((40, 5)); peaks[:, 1] = np.arange(40) * 3.5; peaks[:, 2] = np.arange(40) * 2.0 + 1
    subsets = -np.ones((2, 20)); subsets[0, :5] = [3, 7, 9, 11, 30]; subsets[1, 10:14] = [1, 2, 4, 39]
    assert np.array_equal(det.subsets_to_pose_array(subsets, peaks), R.subsets_to_pose_array(subsets, peaks))
    assert det.subsets_to_pose_array(subsets[:0], peaks).shape == (0,)
    pose = det.subsets_to_pose_array(subsets, peaks)[0]
    joints = [j if j[2] > 0 else None for j in pose]
    lens, limbs = det.compute_limbs_length(joints)
    assert lens.shape == (19,) and det.compute_unit_length(lens) > 0


def test_camera_demo_import_flow_and_drawing():
    """What camera_pose_demo.py does before its capture loop (reference :1-14), flat imports:
    `import chainer`, `from pose_detector import PoseDetector, draw_person_pose`, then the
    drawing helper on a poses array (no GPU needed up to the constructor)."""
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import chainer\n"
        "from pose_detector import PoseDetector, draw_person_pose\n"
        "chainer.using_config('enable_backprop', False)\n"
        "img = np.zeros((120, 160, 3), np.uint8)\n"
        "poses = np.zeros((1, 18, 3)); poses[0, :, 0] = np.linspace(10, 150, 18); poses[0, :, 1] = 60; poses[0, :, 2] = 2\n"
        "out = draw_person_pose(img, poses)\n"
        "assert out.shape == img.shape and out.any() and not img.any()\n"
        "assert draw_person_pose(img, np.empty((0, 18, 3))) is img\n"
        "print('ok')\n") % (os.path.join(ROOT, "chainer_realtime_multi-person_pose_estimation_b200"),
                             os.path.join(ROOT, "chainer_realtime_multi-person_pose_estimation_b200", "compat"))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout


def test_demo_import_flow_face_hand_modules():
    """What demo.py does before inference (reference demo.py:1-20), flat imports: the three detector modules and
    their drawing helpers; host-only helpers (draw_*, crop_face) checked against the reference's own functions
    (their digest in tests/golden/host_helpers_ref.json)."""
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import chainer\n"
        "from entity import params\n"
        "from pose_detector import PoseDetector, draw_person_pose\n"
        "from face_detector import FaceDetector, draw_face_keypoints, crop_face\n"
        "from hand_detector import HandDetector, draw_hand_keypoints\n"
        "assert set(params['archs']) == {'posenet', 'facenet', 'handnet'}\n"
        "assert len(params['archs']['facenet'].LAYERS) == 52 and len(params['archs']['handnet'].LAYERS) == 52\n"
        "img = np.zeros((100, 120, 3), np.uint8)\n"
        "face = [[10 + i, 20 + (i %% 7), np.float32(0.5)] if i %% 5 else None for i in range(70)]\n"
        "hand = [[15 + 3 * i, 30 + (i %% 4), np.float32(0.5)] if i %% 6 else None for i in range(21)]\n"
        "a = draw_face_keypoints(img, face, (3, 4)); b = draw_hand_keypoints(img, hand, (3, 4))\n"
        "assert a.any() and b.any() and not img.any()\n"
        "pf, lt = crop_face(np.arange(100 * 120 * 3, dtype=np.uint8).reshape(100, 120, 3), (30, 20, 40, 50))\n"
        "assert pf.shape[0] == pf.shape[1] and lt == (20, 7)\n"
        "np.save(sys.argv[1], np.concatenate([a.ravel(), b.ravel(), pf.ravel()]))\n"
        "print('ok')\n") % (os.path.join(ROOT, "chainer_realtime_multi-person_pose_estimation_b200"),
                             os.path.join(ROOT, "chainer_realtime_multi-person_pose_estimation_b200", "compat"))
    import tempfile
    out = os.path.join(tempfile.mkdtemp(), "draw.npy")
    r = subprocess.run([sys.executable, "-c", code, out], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout
    import json
    from conftest import GOLDEN
    from oracle import make_goldens as MG
    with open(os.path.join(GOLDEN, "host_helpers_ref.json")) as f:
        assert MG.digest(np.load(out)) == json.load(f)["demo_face_hand_drawing"]



@pytest.mark.parametrize("name,hw", [("fast_584_he0.npz", (584, 584)), ("fast_480x640_he0.npz", (480, 640)),
                                      ("fast_368x656_he0_img0.npz", (368, 656))])
def test_pose_records_to_pose_array_reproduces_reference_rescale(name, hw):
    """Host half of __call__: the device returns integer peak coordinates at map resolution; the float64 rescale of
    pose_detector.py:513-515 (`x *= orig_w / map_w` in place, then subsets_to_pose_array) is redone on the host and
    must give the golden poses / scores bit for bit."""
    from conftest import load_golden
    from oracle import restate as R
    native = pkg("_native")
    PD = pkg("pose_detector").PoseDetector
    det = PD.__new__(PD)

    class _Eng(object):
        def raise_for_status(self, s):
            assert s == 0
    det.engine = _Eng()
    g = load_golden(name)
    oh, ow = hw
    map_w, map_h = R.compute_optimal_size(np.zeros((oh, ow, 3), np.uint8), 320)
    subsets, peaks = g["subsets"], g["all_peaks"]
    n = len(subsets)
    header = np.zeros(1, native.HEADER_DTYPE)
    header["n_peaks"], header["n_persons"] = len(peaks), n
    persons = np.zeros(max(n, 1), native.PERSON_DTYPE)
    ids = subsets[:, :18].astype(np.int64)
    persons["peak_id"][:n] = ids
    safe = np.where(ids >= 0, ids, 0)
    persons["x"][:n] = np.where(ids >= 0, peaks[safe, 1].astype(np.int64), 0)
    persons["y"][:n] = np.where(ids >= 0, peaks[safe, 2].astype(np.int64), 0)
    persons["score"][:n] = subsets[:, 18]
    persons["count"][:n] = subsets[:, 19]
    poses, scores = det._poses_from_records(header[0], persons, ow / map_w, oh / map_h)
    assert poses.shape == g["poses"].shape and np.array_equal(poses, g["poses"])
    assert np.array_equal(scores, g["scores"])
