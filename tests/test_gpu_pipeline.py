"""`-m gpu`: end-to-end parity of the device pipeline against the committed goldens (outputs of
the reference's own files run verbatim, oracle/make_goldens.py) on identical seeded weights, in the two
precisions that claim parity ("parity": split fp16, ~2e-5; "comp": fp16 + 8-bit-float rounding corrections, ~1e-4).

Every end-to-end case asserts, UNCONDITIONALLY:
  (1) float maps: |device - reference golden| <= 1e-3 (north_star tolerance);
  (2) bit-exact keypoints given the maps: peaks, connections (ids and float64 scores), subsets, poses and scores
      returned by the device equal the oracle post-process (oracle/restate.py, pinned to the reference) run on the
      DEVICE's own maps;
  (3) against the golden: every peak that differs is a provable near-tie (its decision margin in the reference maps is
      below TIE_FACTOR x the measured map error) and their number stays inside _max_flips().
When (3) finds no flipped peak and no flipped connection threshold the "strong" branch additionally asserts poses
identical to the reference golden (OKS = 1.0); the branch each case took is recorded (gpurun_out/r2_e2e_branches.json
when that directory exists) and REQUIRED to be the strong one for the cases in STRONG_REQUIRED.
Kernel-level bit-exactness on identical inputs is in test_gpu_postprocess.py."""
import json
import os
import numpy as np
import pytest

from conftest import load_golden, pkg, split_conns
from oracle import restate as R

pytestmark = pytest.mark.gpu

MAP_TOL = 1e-3
TIE_FACTOR = 4.0      # a peak may flip only if its oracle margin is below TIE_FACTOR x the measured map error
# (precision, golden) pairs whose poses must be IDENTICAL to the reference golden (measured on a B200, round 2)
STRONG_REQUIRED = {("parity", "fast_584_he0.npz"), ("parity", "precise_480_he0.npz"), ("parity", "precise_200x300_he0.npz")}


def _max_flips(n_ref, map_err):
    """Sanity bound on top of the per-peak margin check: these goldens are dense noise maps (thousands of peaks at noise
    level), so the number of peaks whose margin lies inside the error band grows with the map error; measured on a B200:
    parity (2e-5) 0 / 3 / 2 flips of 1758 / 2190 / 5829 peaks, i.e. a flipped fraction of up to ~60 x map_err."""
    return max(2, int(np.ceil(80.0 * map_err * n_ref)))
_BRANCHES = {}


def _record_branch(precision, name, info):
    _BRANCHES["%s/%s" % (precision, name)] = info
    out_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out_dir):
        with open(os.path.join(out_dir, "r2_e2e_branches.json"), "w") as f:
            json.dump(_BRANCHES, f, indent=1, sort_keys=True)
    if (precision, name) in STRONG_REQUIRED:
        assert info["strong"], "%s/%s must reproduce the reference golden exactly: %s" % (precision, name, info)


@pytest.fixture(scope="module")
def weights_model():
    m = pkg("models.CocoPoseNet").CocoPoseNet()
    m.load_npz(pkg("synthetic").he_weights(0))
    return m


@pytest.fixture(scope="module")
def det_parity(weights_model):
    return pkg("pose_detector").PoseDetector(model=weights_model, device=0, precision="parity",
                                             max_candidates=131072, max_persons=4096)


@pytest.fixture(scope="module")
def det_comp(weights_model):
    return pkg("pose_detector").PoseDetector(model=weights_model, device=0, precision="comp",
                                             max_candidates=131072, max_persons=4096)


@pytest.fixture(params=["parity", "comp"])
def det_any(request, det_parity, det_comp):
    d = det_parity if request.param == "parity" else det_comp
    d._test_precision = request.param
    return d


def _oracle_margins(heat):
    """Per-pixel decision margin of the oracle's peak test on the smoothed maps."""
    g = R.gaussian_smooth(heat[:-1].astype(np.float32)).astype(np.float64)
    pad = np.pad(g, ((0, 0), (1, 1), (1, 1)))
    nb = np.maximum.reduce([pad[:, :-2, 1:-1], pad[:, 2:, 1:-1], pad[:, 1:-1, :-2], pad[:, 1:-1, 2:]])
    return np.minimum(g - R.HEATMAP_PEAK_THRESH, g - nb)


def _peak_sets_match(got_peaks, ref_peaks, heat_oracle, tie_eps):
    margin = _oracle_margins(heat_oracle)
    key = lambda p: set(map(tuple, p[:, :3].astype(int))) if len(p) else set()
    G, Rf = key(got_peaks), key(ref_peaks)
    sym = G ^ Rf
    for (c, x, y) in sym:
        assert abs(margin[c, y, x]) < tie_eps, "peak (%d,%d,%d) differs with oracle margin %.3e (eps %.1e)" % (
            c, x, y, margin[c, y, x], tie_eps)
    return len(sym)


def test_forward_maps_parity_mode(det_any):
    det_parity = det_any
    g = load_golden("fast_584_he0.npz")
    img = pkg("synthetic").procedural_image(584, 584, seed=1)
    import cv2
    x = det_parity.preprocess(cv2.resize(img, (368, 368)))
    paf, heat = det_parity.engine.forward(x)
    e1, e2 = np.abs(paf[0] - g["paf_lo_0"]).max(), np.abs(heat[0] - g["heat_lo_0"]).max()
    print("%s-precision max abs err: paf %.3e heat %.3e" % (det_any._test_precision, e1, e2))
    assert e1 <= MAP_TOL and e2 <= MAP_TOL
    assert max(e1, e2) <= (1e-4 if det_any._test_precision == "parity" else 5e-4)   # measured: ~2e-5 / ~1.5e-4
    # uint8 entry (preprocess fused into the exact tensor-core conv1_1) vs the float32 entry (fp32 CUDA-core conv1_1): the
    # two first layers agree to ~1e-7; compensated precision amplifies that through its 8-bit correction bytes
    paf_u8, heat_u8 = det_parity.engine.forward(cv2.resize(img, (368, 368))[None])
    tol_entry = 1e-5 if det_any._test_precision == "parity" else 2e-4
    assert np.abs(paf_u8 - paf).max() <= tol_entry and np.abs(heat_u8 - heat).max() <= tol_entry
    e3 = max(np.abs(paf_u8[0] - g["paf_lo_0"]).max(), np.abs(heat_u8[0] - g["heat_lo_0"]).max())
    assert e3 <= (1e-4 if det_any._test_precision == "parity" else 5e-4)


def test_fast_mode_uint8_entry_matches_float_entry(weights_model):
    """conv1_1 on tensor cores (uint8 frames, im2col built per thread) vs the CUDA-core conv1_1 fed the preprocessed
    float32 image: same network, so the maps may differ only by fp16 rounding of the first layer's operands (which the
    other 91 layers amplify to ~1e-2 on a white-noise frame whose maps are O(10); a misplaced tap would give O(1)).
    The bound is relative to the map magnitude."""
    det = pkg("pose_detector").PoseDetector(model=weights_model, device=0, precision="fast")
    imgs = pkg("synthetic").random_images(2, 368, 496, seed=4)
    imgs[1, :, :, :] = pkg("synthetic").procedural_image(368, 496, seed=9)
    paf_u8, heat_u8 = det.engine.forward(imgs)
    x = np.concatenate([det.preprocess(im) for im in imgs])
    paf_f, heat_f = det.engine.forward(x)
    for i in range(2):
        e = max(float(np.abs(paf_u8[i] - paf_f[i]).max()), float(np.abs(heat_u8[i] - heat_f[i]).max()))
        mag = max(float(np.abs(paf_f[i]).max()), float(np.abs(heat_f[i]).max()))
        print("fast mode, uint8 (tensor-core conv1_1) vs float32 entry, image %d: max abs diff %.3e (maps up to %.2f)"
              % (i, e, mag))
        assert e < 4e-3 * max(mag, 1.0)


@pytest.mark.parametrize("precision", ["fast", "comp"])
def test_fused_1x1_pair_is_bit_identical_to_two_launches(weights_model, monkeypatch, precision):
    """Mconv6 + Mconv7 fused into one kernel (csrc/conv_mlp2.cuh, the 128-channel intermediate stays in shared memory)
    vs the two separate 1x1 launches: same MMA shapes and accumulation order, so the maps must be bit-identical --
    batch 2 (throughput tile shapes), batch 1 (small-batch shapes) and HandNet (single branch); fp16 and compensated
    precision (there the fused kernel also writes the intermediate's 8-bit correction bytes into the operand tile)."""
    syn = pkg("synthetic")
    imgs = syn.random_images(2, 368, 496, seed=4)
    hn = pkg("models.HandNet")
    hand = hn.HandNet()
    hand.load_npz(syn.he_weights(0, layers=hn.LAYERS))
    crop = syn.procedural_image(368, 368, seed=5)[None]
    out = []
    monkeypatch.setenv("OPB_MLP2_COMP", "1")   # the compensated variant is opt-in (slower than the two launches at batch 32)
    for no_fuse in ("0", "1"):
        monkeypatch.setenv("OPB_NO_MLP2", no_fuse)
        det = pkg("pose_detector").PoseDetector(model=weights_model, device=0, precision=precision)
        hd = pkg("hand_detector").HandDetector(model=hand, device=0, precision=precision)
        out.append((det.engine.forward(imgs), det.engine.forward(imgs[:1]), hd.engine.forward_keypoint_maps(crop)))
        del det, hd
    (a2, a1, ah), (b2, b1, bh) = out
    for x, y in ((a2[0], b2[0]), (a2[1], b2[1]), (a1[0], b1[0]), (a1[1], b1[1]), (ah, bh)):
        assert np.isfinite(x).all() and np.array_equal(x, y), float(np.abs(x - y).max())


def test_forward_maps_fast_mode(weights_model):
    """fp16 operands ("fast"): OUTSIDE the 1e-3 tolerance by design (BASELINE.json configs[1] names fp16 for the roofline
    measurement); SURVEY 8d(ii) prescribes reporting its max-abs map error and the symmetric difference of the peak sets
    on the fast goldens instead of claiming parity -- both are bounded here so that a regression shows."""
    import cv2
    det = pkg("pose_detector").PoseDetector(model=weights_model, device=0, precision="fast", max_candidates=131072,
                                            max_persons=4096)
    syn = pkg("synthetic")
    report = {}
    for name, img in (("fast_584_he0.npz", syn.procedural_image(584, 584, seed=1)),
                      ("fast_480x640_he0.npz", syn.procedural_image(480, 640, seed=2)),
                      ("fast_368x656_he0_img0.npz", syn.random_images(2, 368, 656, seed=0)[0])):
        g = load_golden(name)
        in_w, in_h = R.compute_optimal_size(img, 368)
        paf, heat = det.engine.forward(cv2.resize(img, (in_w, in_h))[None])
        err = max(float(np.abs(paf[0] - g["paf_lo_0"]).max()), float(np.abs(heat[0] - g["heat_lo_0"]).max()))
        det(img)
        peaks = det.engine.image_detail(0)[0]
        key = lambda p: set(map(tuple, p[:, :3].astype(int))) if len(p) else set()
        sym, n_ref = len(key(peaks) ^ key(g["all_peaks"])), len(g["all_peaks"])
        report[name] = dict(map_err=err, peak_symdiff=sym, ref_peaks=n_ref)
        print("fast (fp16) %s: max abs map err %.3e, peak-set symmetric difference %d of %d" % (name, err, sym, n_ref))
        assert err <= 2e-2                  # ~3e-3 on the O(1) procedural maps, ~1e-2 on the O(10) white-noise frame
        assert sym <= max(4, n_ref // 4)    # SURVEY probe: ~10 % of the noise peaks flip at fp16
    _record_branch("fast", "peak_symdiff_report", dict(strong=False, report=report))


def _check_call(det, name, img):
    precision = det._test_precision
    g = load_golden(name)
    poses, scores = det(img)
    if g["all_peaks"].shape[0] == 0:
        assert poses.shape == (0, 18, 3) and scores.shape == (0,)
        return
    oh, ow = img.shape[:2]
    in_w, in_h = R.compute_optimal_size(img, 368)
    map_w, map_h = R.compute_optimal_size(img, 320)
    peaks, conns, subsets = det.engine.image_detail(0)
    import cv2
    paf_lo, heat_lo = det.engine.forward(cv2.resize(img, (in_w, in_h))[None])
    # (1) maps within the tolerance of the reference
    map_err = max(np.abs(paf_lo[0] - g["paf_lo_0"]).max(), np.abs(heat_lo[0] - g["heat_lo_0"]).max())
    assert map_err <= MAP_TOL
    # (2) given the device's maps, everything downstream is bit-exact: oracle post-process of the device's own maps
    d_pafs = R.resize_bilinear_align_corners(paf_lo, (map_h, map_w))[0]
    d_heat = R.resize_bilinear_align_corners(heat_lo, (map_h, map_w))[0]
    o_poses, o_scores, parts = R.postprocess_fast(d_pafs, d_heat, map_w, ow, oh, map_h, return_parts=True)
    assert np.array_equal(peaks, parts["all_peaks"])
    assert len(conns) == len(parts["connections"]) and all(np.array_equal(a, b) for a, b in zip(conns, parts["connections"]))
    assert np.array_equal(subsets, parts["subsets"])
    assert poses.shape == o_poses.shape and np.array_equal(poses, o_poses) and np.array_equal(scores, o_scores)
    # (3) against the reference golden: only provable near-ties may differ
    heat_or = R.resize_bilinear_align_corners(g["heat_lo_0"][None], (map_h, map_w))[0]
    n_ties = _peak_sets_match(peaks, g["all_peaks"], heat_or, max(TIE_FACTOR * map_err, 1e-4))
    assert n_ties <= _max_flips(len(g["all_peaks"]), map_err)
    ref_conns = split_conns(g["conn_lens"], g["conn_flat"])
    n_conn_diff = -1
    if n_ties == 0:
        assert np.array_equal(peaks[:, :3], g["all_peaks"][:, :3])
        assert np.abs(peaks[:, 3] - g["all_peaks"][:, 3]).max() <= MAP_TOL
        # connection acceptance thresholds (ip > 0.05, score > 0) have their own measure-zero ties
        n_conn_diff = sum(0 if (a.shape == b.shape and np.array_equal(a[:, :2], b[:, :2])) else 1
                          for a, b in zip(conns, ref_conns))
        assert n_conn_diff <= 2
    strong = n_ties == 0 and n_conn_diff == 0
    if strong:
        assert subsets.shape == g["subsets"].shape
        assert np.array_equal(subsets[:, :18], g["subsets"][:, :18])
        assert np.abs(subsets[:, 18:] - g["subsets"][:, 18:]).max() <= 1e-2
        assert poses.shape == g["poses"].shape and np.array_equal(poses, g["poses"])      # OKS = 1.0
        assert np.abs(scores - g["scores"]).max() <= 1e-2
    info = dict(strong=bool(strong), map_err=float(map_err), peaks=int(len(peaks)), ref_peaks=int(len(g["all_peaks"])),
                near_tie_peak_flips=int(n_ties), limbs_with_flipped_connections=int(n_conn_diff),
                persons=int(len(poses)), ref_persons=int(len(g["poses"])))
    print(precision, name, info)
    _record_branch(precision, name, info)


def test_call_fast_path_584(det_any):
    _check_call(det_any, "fast_584_he0.npz", pkg("synthetic").procedural_image(584, 584, seed=1))


def test_call_fast_path_webcam_shape(det_any):
    _check_call(det_any, "fast_480x640_he0.npz", pkg("synthetic").procedural_image(480, 640, seed=2))


def test_call_fast_path_dense_noise(det_any):
    _check_call(det_any, "fast_368x656_he0_img0.npz", pkg("synthetic").random_images(2, 368, 656, seed=0)[0])


def test_call_default_init_returns_empty():
    m = pkg("models.CocoPoseNet").CocoPoseNet()
    m.load_npz(pkg("synthetic").he_weights(0, bias_scale=0.0, gain=1.0))
    det = pkg("pose_detector").PoseDetector(model=m, device=0)
    poses, scores = det(pkg("synthetic").procedural_image(584, 584, seed=1))
    assert poses.shape == (0, 18, 3) and scores.shape == (0,)


def test_detect_batch_matches_single_calls(det_parity):
    imgs = pkg("synthetic").random_images(2, 368, 656, seed=0)
    res = det_parity.detect_batch(imgs)
    for i in range(2):
        g = load_golden("fast_368x656_he0_img%d.npz" % i)
        poses, scores = res[i]
        single = det_parity(imgs[i])
        assert poses.shape == single[0].shape and np.array_equal(poses, single[0])
        assert abs(len(poses) - len(g["poses"])) <= 3


def test_stream_mode_matches_single_calls(det_parity):
    """Pipelined submit/collect (two slots, copy stream, device resize) returns, in order, exactly what the
    synchronous __call__ returns for every frame -- frames of different sizes, single frames and batches."""
    syn = pkg("synthetic")
    frames = [syn.procedural_image(480, 640, seed=3), syn.procedural_image(584, 584, seed=1),
              syn.random_images(2, 368, 656, seed=0), syn.procedural_image(240, 320, seed=7),
              syn.procedural_image(480, 640, seed=4)]
    got = list(det_parity.detect_stream(iter(frames)))
    assert len(got) == len(frames)
    for f, g in zip(frames, got):
        if f.ndim == 4:
            for i in range(len(f)):
                p, sc = det_parity(f[i])
                assert g[i][0].shape == p.shape and np.array_equal(g[i][0], p) and np.array_equal(g[i][1], sc)
        else:
            p, sc = det_parity(f)
            assert g[0].shape == p.shape and np.array_equal(g[0], p) and np.array_equal(g[1], sc)
    # same shape submitted repeatedly: from the second submit per slot the launch sequence is captured into a CUDA
    # graph and replayed -- results must not change (8 frames = 4 per slot: eager, capture, replay, replay)
    same = [syn.procedural_image(480, 640, seed=30 + i) for i in range(8)]
    got = list(det_parity.detect_stream(iter(same)))
    for f, g in zip(same, got):
        p, sc = det_parity(f)
        assert g[0].shape == p.shape and np.array_equal(g[0], p) and np.array_equal(g[1], sc)
    # protocol errors are reported, not silently overwritten
    eng = det_parity.engine
    eng.stream_submit(frames[0], 368, 496, 320, 432, slot=0)
    with pytest.raises(RuntimeError):
        eng.stream_submit(frames[0], 368, 496, 320, 432, slot=0)
    eng.stream_collect(0)
    with pytest.raises(RuntimeError):
        eng.stream_collect(0)


def test_injected_synthetic_eight_person_maps(det_parity):
    """Config #3: synthetic 8-person maps injected as the network output (the conv chain still
    runs); 8 persons must come out for every image of the batch, identical to the oracle run
    on the same low-resolution maps."""
    import torch
    syn = pkg("synthetic")
    paf_lo, heat_lo = syn.eight_person_lowres(46, 82, seed=0)
    imgs = syn.random_images(2, 368, 656, seed=5)
    n = len(imgs)
    d_paf = torch.from_numpy(np.repeat(paf_lo[None], n, 0)).cuda()
    d_heat = torch.from_numpy(np.repeat(heat_lo[None], n, 0)).cuda()
    torch.cuda.synchronize()
    headers, persons = det_parity.engine.detect_batch(imgs, 320, 576, inject_paf=d_paf.data_ptr(),
                                                      inject_heat=d_heat.data_ptr())
    pafs = R.resize_bilinear_align_corners(paf_lo[None], (320, 576))[0]
    heat = R.resize_bilinear_align_corners(heat_lo[None], (320, 576))[0]
    ref_poses, ref_scores, parts = R.postprocess_fast(pafs, heat, 576, 576, 320, 320, return_parts=True)
    for i in range(n):
        assert headers[i]["status"] == 0 and headers[i]["n_persons"] == len(ref_scores) == 8
        peaks, conns, subsets = det_parity.engine.image_detail(i)
        assert np.array_equal(peaks, parts["all_peaks"])
        assert np.array_equal(subsets, parts["subsets"])


def _check_precise(weights_model, precision, name, img, stride):
    det = pkg("pose_detector").PoseDetector(model=weights_model, device=0, precise=True, precision=precision,
                                            max_candidates=131072, max_persons=4096)
    g = load_golden(name)
    oh, ow = img.shape[:2]
    poses, scores = det(img)
    # (1) maps
    e1 = np.abs(det.pafs[:, ::stride, ::stride] - g["pafs_sample"]).max()
    e2 = np.abs(det.heatmaps[:, ::stride, ::stride] - g["heatmaps_sample"]).max()
    assert e1 <= MAP_TOL and e2 <= MAP_TOL
    # (2) bit-exact post-process of the device's own averaged maps (pose_detector.py:476-482, img_len = original width)
    o_peaks = R.compute_peaks_from_heatmaps(det.heatmaps)
    assert np.array_equal(det.all_peaks, o_peaks)
    o_conns = R.compute_connections(det.pafs, o_peaks, ow)
    o_subsets = R.grouping_key_points(o_conns, o_peaks)
    o_poses = R.subsets_to_pose_array(o_subsets, o_peaks)
    assert poses.shape == o_poses.shape and np.array_equal(poses, o_poses) and np.array_equal(scores, o_subsets[:, -2])
    # (3) against the reference golden
    G = set(map(tuple, det.all_peaks[:, :3].astype(int)))
    Rf = set(map(tuple, g["all_peaks"][:, :3].astype(int)))
    assert len(G ^ Rf) <= _max_flips(len(Rf), max(e1, e2))
    strong = (G == Rf) and poses.shape == g["poses"].shape and np.array_equal(poses, g["poses"])   # OKS = 1.0 vs the reference
    info = dict(strong=bool(strong), map_err=float(max(e1, e2)), peaks=len(G), ref_peaks=len(Rf), peak_symdiff=len(G ^ Rf),
                persons=int(len(poses)), ref_persons=int(len(g["poses"])))
    print(precision, name, info)
    _record_branch(precision, name, info)


def test_precise_path_device_cubic_ingest(weights_model):
    """detect_precise with the per-scale uint8 INTER_CUBIC resize (:443) on the device as well (OpenCV's own 8-bit cubic
    arithmetic).  The committed goldens were produced with this image's IPP-dispatching cv2 (input pixels 1 LSB apart on a
    few per cent of the frame, which a random-weight net amplifies to ~2e-3 on the maps), so the oracle is re-run here with
    IPP dispatch off -- the cv2 code path the device kernel reproduces bit for bit: maps inside the tolerance,
    post-process bit-exact on the device's maps, peak flips only at near-ties."""
    import cv2
    syn = pkg("synthetic")
    wd = syn.he_weights(0)
    weights = {k[:-2]: (wd[k], wd[k[:-2] + "/b"]) for k in wd if k.endswith("/W")}
    img = syn.procedural_image(200, 300, seed=4)
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        ref_pafs, ref_heat = R.precise_maps(weights, img)
    finally:
        cv2.ipp.setUseIPP(was)
    for precision in ("parity", "comp"):
        det = pkg("pose_detector").PoseDetector(model=weights_model, device=0, precise=True, precision=precision,
                                                max_candidates=131072, max_persons=4096, device_cubic=True)
        poses, scores = det(img)
        e1, e2 = float(np.abs(det.pafs - ref_pafs).max()), float(np.abs(det.heatmaps - ref_heat).max())
        assert e1 <= MAP_TOL and e2 <= MAP_TOL, (precision, e1, e2)
        o_peaks = R.compute_peaks_from_heatmaps(det.heatmaps)
        assert np.array_equal(det.all_peaks, o_peaks)
        o_conns = R.compute_connections(det.pafs, o_peaks, img.shape[1])
        o_subsets = R.grouping_key_points(o_conns, o_peaks)
        o_poses = R.subsets_to_pose_array(o_subsets, o_peaks)
        assert poses.shape == o_poses.shape and np.array_equal(poses, o_poses) and np.array_equal(scores, o_subsets[:, -2])
        r_peaks = R.compute_peaks_from_heatmaps(ref_heat)
        G, Rf = set(map(tuple, det.all_peaks[:, :3].astype(int))), set(map(tuple, r_peaks[:, :3].astype(int)))
        assert len(G ^ Rf) <= _max_flips(len(Rf), max(e1, e2))
        _record_branch(precision + "+device_cubic", "precise_200x300_ipp_off", dict(strong=bool(G == Rf), map_err=max(e1, e2), peaks=len(G),
                                                                                    ref_peaks=len(Rf), peak_symdiff=len(G ^ Rf)))


@pytest.mark.parametrize("precision", ["parity", "comp"])
def test_precise_path_480(weights_model, precision):
    _check_precise(weights_model, precision, "precise_480_he0.npz", pkg("synthetic").procedural_image(480, 480, seed=3), 9)


@pytest.mark.parametrize("precision", ["parity", "comp"])
def test_precise_path_padded_200x300(weights_model, precision):
    """Precise path with padding: the scaled inputs 184x276 and 552x828 are padded to 280 / 832 columns
    (pad_image, :445) and the x8 maps cropped again (:462,:466)."""
    _check_precise(weights_model, precision, "precise_200x300_he0.npz", pkg("synthetic").procedural_image(200, 300, seed=4), 5)


def test_overlay_from_device_records_matches_cv2(det_parity):
    """draw_person_pose (pose_detector.py:520-553) for the frame just passed to __call__, rasterised on the device from the
    device-resident person records (opb_draw_last_result: float64 rescale + rint as :513-514 / :539), against the host cv2
    loop on the returned poses: dense random-weight "persons" (hundreds of overlapping limbs and joints), so the overwrite
    order matters on most covered pixels."""
    pd = pkg("pose_detector")
    for seed, (h, w) in ((2, (480, 640)), (7, (368, 656))):
        img = pkg("synthetic").procedural_image(h, w, seed=seed)
        poses, scores = det_parity(img)
        assert len(scores) > 0
        assert np.array_equal(det_parity.draw_last_result(img), pd.draw_person_pose(img, poses))
        assert np.array_equal(pd.draw_person_pose(img, poses, engine=det_parity.engine), pd.draw_person_pose(img, poses))
