"""`not gpu`: pins oracle/restate.py against the committed goldens, which were produced by
the reference's own files executed verbatim (oracle/make_goldens.py), and against the
third-party routines it restates (scipy gaussian_filter)."""
import numpy as np
import pytest

from conftest import load_golden, pkg, split_conns
from oracle import make_goldens
from oracle import restate as R


@pytest.fixture(autouse=True)
def golden_torch_threads():
    """The torch-CPU convolutions run with the thread count the goldens were made with (their last bits depend on it)."""
    import torch
    saved = torch.get_num_threads()
    torch.set_num_threads(make_goldens.TORCH_THREADS)
    yield
    torch.set_num_threads(saved)


def test_layer_table_matches_package():
    assert tuple(R.layer_table()) == pkg("models.CocoPoseNet").LAYERS
    assert pkg("models.CocoPoseNet").conv_flops_per_image(368, 656) == 484634285056


def test_gaussian_bit_exact_vs_scipy():
    from scipy.ndimage import gaussian_filter
    rs = np.random.RandomState(0)
    for t in range(6):
        a = (rs.standard_normal((3, 40 + 7 * t, 33 + 11 * t)) * rs.uniform(0.01, 3)).astype(np.float32)
        mine = R.gaussian_smooth(a)
        for c in range(3):
            assert np.array_equal(mine[c], gaussian_filter(a[c], sigma=2.5))
    # tiny maps: reflect extension longer than the image
    a = rs.standard_normal((1, 12, 15)).astype(np.float32)
    assert np.array_equal(R.gaussian_smooth(a)[0], gaussian_filter(a[0], sigma=2.5))


def test_resize_matches_torch_align_corners():
    import torch
    rs = np.random.RandomState(1)
    x = rs.standard_normal((1, 5, 46, 82)).astype(np.float32)
    y = R.resize_bilinear_align_corners(x, (320, 576))
    t = torch.nn.functional.interpolate(torch.from_numpy(x), size=(320, 576), mode="bilinear", align_corners=True)
    assert np.abs(y - t.numpy()).max() < 1e-4   # torch uses an fp32 scale; sanity only
    assert np.array_equal(y[..., 0, 0], x[..., 0, 0]) and np.array_equal(y[..., -1, -1], x[..., -1, -1])


@pytest.mark.parametrize("seed", [0, 1])
def test_postprocess_synth8(seed):
    g = load_golden("synth8_post_seed%d.npz" % seed)
    paf, heat, joints = pkg("synthetic").eight_person_maps(seed=seed)
    assert np.array_equal(joints, g["joints"])
    peaks = R.compute_peaks_from_heatmaps(heat)
    assert np.array_equal(peaks, g["all_peaks"])
    conns = R.compute_connections(paf, peaks, 576)
    ref = split_conns(g["conn_lens"], g["conn_flat"])
    for a, b in zip(conns, ref):
        assert np.array_equal(a, b)
    subsets = R.grouping_key_points(conns, peaks)
    assert np.array_equal(subsets, g["subsets"])
    assert np.array_equal(R.subsets_to_pose_array(subsets, peaks), g["poses"])
    assert len(subsets) == 8


def _check_fast(name, img, weights):
    g = load_golden(name)
    poses, scores, parts = R.detect_fast(weights, img, return_parts=True)
    assert np.array_equal(parts["paf_lo"], g["paf_lo_0"])
    assert np.array_equal(parts["heat_lo"], g["heat_lo_0"])
    if g["all_peaks"].shape[0] == 0:
        assert poses.shape == (0, 18, 3) and scores.shape == (0,)
        return
    assert np.array_equal(parts["all_peaks"], g["all_peaks"])
    for a, b in zip(parts["connections"], split_conns(g["conn_lens"], g["conn_flat"])):
        assert np.array_equal(a, b)
    assert np.array_equal(parts["subsets"], g["subsets"])
    assert np.array_equal(poses, g["poses"]) and np.array_equal(scores, g["scores"])


def test_fast_path_584(he_weights):
    _check_fast("fast_584_he0.npz", pkg("synthetic").procedural_image(584, 584, seed=1), he_weights)


def test_fast_path_webcam_shape(he_weights):
    _check_fast("fast_480x640_he0.npz", pkg("synthetic").procedural_image(480, 640, seed=2), he_weights)


def test_fast_path_noise_frame_dense_candidates(he_weights):
    # ~5 800 peaks, ~2 M candidate pairs: the dense stress case
    _check_fast("fast_368x656_he0_img0.npz", pkg("synthetic").random_images(2, 368, 656, seed=0)[0], he_weights)


def test_fast_path_default_init_empty():
    d = pkg("synthetic").he_weights(0, bias_scale=0.0, gain=1.0)
    w = {k[:-2]: (d[k], d[k[:-2] + "/b"]) for k in d if k.endswith("/W")}
    _check_fast("fast_584_lecun0.npz", pkg("synthetic").procedural_image(584, 584, seed=1), w)


def test_precise_path_480(he_weights):
    g = load_golden("precise_480_he0.npz")
    img = pkg("synthetic").procedural_image(480, 480, seed=3)
    poses, scores, parts = R.detect_precise(he_weights, img, return_parts=True)
    assert np.array_equal(parts["pafs"][:, ::9, ::9], g["pafs_sample"])
    assert np.array_equal(parts["heatmaps"][:, ::9, ::9], g["heatmaps_sample"])
    assert np.array_equal(parts["all_peaks"], g["all_peaks"])
    assert np.array_equal(parts["subsets"], g["subsets"])
    assert np.array_equal(poses, g["poses"]) and np.array_equal(scores, g["scores"])


def test_precise_path_padded_200x300(he_weights):
    # scales 0.5 and 1.5 need right-padding to a multiple of 8: pad_image / crop of :445,:462,:466
    g = load_golden("precise_200x300_he0.npz")
    img = pkg("synthetic").procedural_image(200, 300, seed=4)
    poses, scores, parts = R.detect_precise(he_weights, img, return_parts=True)
    assert np.array_equal(parts["pafs"][:, ::5, ::5], g["pafs_sample"])
    assert np.array_equal(parts["heatmaps"][:, ::5, ::5], g["heatmaps_sample"])
    assert np.array_equal(parts["all_peaks"], g["all_peaks"])
    assert np.array_equal(parts["subsets"], g["subsets"])
    assert np.array_equal(poses, g["poses"]) and np.array_equal(scores, g["scores"])


def test_cv2_linear_u8_restatement_bit_exact():
    import cv2
    rs = np.random.RandomState(0)
    shapes = [((480, 640), (496, 368)), ((584, 584), (368, 368)), ((1080, 1920), (656, 368)), ((100, 37), (368, 1000)),
              ((240, 320), (496, 368)), ((736, 1312), (656, 368)), ((368, 656), (656, 368)), ((333, 517), (576, 368))]
    for _ in range(10):
        shapes.append(((rs.randint(40, 600), rs.randint(40, 600)), (rs.randint(40, 500), rs.randint(40, 500))))
    for (h0, w0), (W, H) in shapes:
        img = rs.randint(0, 256, (h0, w0, 3)).astype(np.uint8)
        assert np.array_equal(R.cv2_resize_linear_u8(img, (W, H)), cv2.resize(img, (W, H))), ((h0, w0), (W, H))


def test_cv2_cubic_u8_restatement_bit_exact():
    """OpenCV's own 8-bit INTER_CUBIC path (pose_detector.py:443), i.e. cv2 with IPP dispatch off; with IPP on (this
    image's default) ippiResizeCubic differs by 1 LSB on a few per cent of the pixels -- bounded here, not matched."""
    import cv2
    rs = np.random.RandomState(0)
    shapes = [((480, 480), (184, 184)), ((480, 480), (368, 368)), ((480, 480), (552, 552)), ((480, 480), (736, 736)),
              ((200, 300), (276, 184)), ((200, 300), (1104, 736)), ((3000, 54), (27, 1500)), ((2000, 10), (5, 1000)),
              ((360, 640), (321, 181)), ((97, 131), (131, 97))]
    for _ in range(8):
        shapes.append(((rs.randint(20, 400), rs.randint(20, 400)), (rs.randint(5, 500), rs.randint(5, 500))))
    was = cv2.ipp.useIPP()
    try:
        for (h0, w0), (W, H) in shapes:
            img = rs.randint(0, 256, (h0, w0, 3)).astype(np.uint8)
            got = R.cv2_resize_cubic_u8(img, (W, H))
            cv2.ipp.setUseIPP(False)
            assert np.array_equal(got, cv2.resize(img, (W, H), interpolation=cv2.INTER_CUBIC)), ((h0, w0), (W, H))
            cv2.ipp.setUseIPP(True)
            d = np.abs(got.astype(int) - cv2.resize(img, (W, H), interpolation=cv2.INTER_CUBIC).astype(int))
            assert d.max() <= 1 and (d != 0).mean() < 0.15, ((h0, w0), (W, H), d.max(), (d != 0).mean())
    finally:
        cv2.ipp.setUseIPP(was)


def test_optimal_size_rule():
    z = np.zeros
    assert R.compute_optimal_size(z((368, 656, 3)), 368) == (656, 368)
    assert R.compute_optimal_size(z((368, 656, 3)), 320) == (576, 320)
    assert R.compute_optimal_size(z((480, 640, 3)), 368) == (496, 368)
    assert R.compute_optimal_size(z((584, 584, 3)), 368) == (368, 368)
    assert R.compute_optimal_size(z((640, 480, 3)), 368) == (368, 496)


def test_grouping_third_match_raises_index_error():
    # three subsets matching one connection: the reference raises IndexError (:193-198)
    peaks = np.zeros((12, 5)); peaks[:, 4] = np.arange(12); peaks[:, 3] = 1.0
    conns = [np.zeros((0, 3)) for _ in range(19)]
    conns[0] = np.array([[0., 1., 1.], [2., 3., 1.]])
    conns[3] = np.array([[4., 5., 1.]])
    conns[6] = np.array([[0., 6., 1.], [2., 6., 0.9], [4., 6., 0.8]])
    with pytest.raises(IndexError):
        R.grouping_key_points(conns, peaks)


@pytest.mark.parametrize("name,kind,hand_type", [("face_150x170_he0.npz", "face", None),
                                                  ("hand_120x131_he0_right.npz", "hand", "right"),
                                                  ("hand_120x131_he0_left.npz", "hand", "left")])
def test_keypoint_restatement_matches_reference_goldens(name, kind, hand_type):
    """FaceDetector / HandDetector run verbatim (oracle/make_goldens.py keypoint_goldens) vs the restatement."""
    g = load_golden(name)
    h, w, seed = (int(v) for v in g["img_hw_seed"])
    mod = pkg("models.FaceNet" if kind == "face" else "models.HandNet")
    wd = pkg("synthetic").he_weights(0, layers=mod.LAYERS)
    weights = {n: (wd[n + "/W"], wd[n + "/b"]) for n, _, _, _ in mod.LAYERS}
    assert [tuple(t) for t in R.keypoint_layer_table(mod.N_OUT)] == [tuple(t) for t in mod.LAYERS]
    kps, lo, _ = R.detect_keypoints(weights, pkg("synthetic").procedural_image(h, w, seed=seed), hand_type)
    assert np.array_equal(lo, g["heat_lo"])
    assert [k is not None for k in kps] == g["valid"].tolist()
    for k, xy, c in zip(kps, g["xy"], g["conf"]):
        if k is not None:
            assert (k[0], k[1]) == (xy[0], xy[1]) and np.float32(k[2]) == c

