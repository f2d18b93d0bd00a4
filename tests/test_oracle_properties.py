"""Property tests (CPU) pinning pieces of oracle/restate.py against the third-party arithmetic the reference calls
(SciPy gaussian_filter, OpenCV resize) and against the reference's own helper on many random shapes -- the oracle is
only as good as these restatements (SURVEY.md 8c: "parity unpinned" boundaries)."""
import numpy as np
from hypothesis import given, settings, strategies as st

from conftest import load_golden
from oracle import restate as R


@settings(max_examples=40, deadline=None)
@given(st.integers(1, 70), st.integers(1, 90), st.integers(0, 2 ** 31 - 1))
def test_gaussian_smooth_is_scipy_bit_for_bit(h, w, seed):
    """Includes maps smaller than the 10-pixel radius (multiple reflections)."""
    from scipy.ndimage import gaussian_filter
    a = np.random.RandomState(seed).standard_normal((h, w)).astype(np.float32)
    assert np.array_equal(R.gaussian_smooth(a), gaussian_filter(a, sigma=R.GAUSSIAN_SIGMA))


@settings(max_examples=60, deadline=None)
@given(st.integers(2, 300), st.integers(2, 300), st.integers(1, 400), st.integers(1, 400), st.integers(0, 2 ** 31 - 1))
def test_cv2_linear_u8_restatement_random_shapes(h0, w0, h, w, seed):
    import cv2
    img = np.random.RandomState(seed).randint(0, 256, (h0, w0, 3)).astype(np.uint8)
    assert np.array_equal(R.cv2_resize_linear_u8(img, (w, h)), cv2.resize(img, (w, h)))


def test_compute_optimal_size_matches_reference():
    """The reference's own compute_optimal_size on the corners of the 16..2000 range and 4 000 seeded random
    (h, w, size) triples (tests/golden/optimal_size_ref.npz, oracle/make_goldens.py host_helper_goldens)."""
    g = load_golden("optimal_size_ref.npz")
    for (h, w, size), want in zip(g["h_w_size"], g["optimal_size"]):
        img = np.zeros((int(h), int(w), 3), np.uint8)
        assert tuple(R.compute_optimal_size(img, int(size))) == tuple(want), (h, w, size)


@settings(max_examples=25, deadline=None)
@given(st.integers(2, 40), st.integers(2, 40), st.integers(2, 150), st.integers(2, 150), st.integers(0, 2 ** 31 - 1))
def test_resize_bilinear_align_corners_matches_stub_resize(h, w, H, W, seed):
    """The restatement vs the Chainer-style resize_images of the stub the reference files run on."""
    import sys, os
    stub = os.path.join(os.path.dirname(os.path.abspath(R.__file__)), "chainer_stub")
    x = np.random.RandomState(seed).standard_normal((1, 3, h, w)).astype(np.float32)
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "chainer" or k.startswith("chainer.")}
    sys.path.insert(0, stub)
    try:
        import chainer.functions as F
        want = np.asarray(F.resize_images(x, (H, W)).data)
    finally:
        sys.path.remove(stub)
        for k in list(sys.modules):
            if k == "chainer" or k.startswith("chainer."):
                del sys.modules[k]
        sys.modules.update(saved)
    assert np.array_equal(R.resize_bilinear_align_corners(x, (H, W)), want)


@settings(max_examples=30, deadline=None)
@given(st.integers(3, 30), st.integers(3, 30), st.integers(0, 2 ** 31 - 1), st.booleans())
def test_keypoints_from_heatmaps_matches_reference_logic(h, w, seed, plateau):
    """The CPU branch of face/hand compute_peaks_from_heatmaps restated literally, incl. exact ties."""
    from scipy.ndimage import gaussian_filter
    rs = np.random.RandomState(seed)
    maps = rs.uniform(0, 0.3, (4, h, w)).astype(np.float32)
    if plateau:
        maps[1] = 0.25
    got = R.keypoints_from_heatmaps(maps)
    for i in range(3):
        g = gaussian_filter(maps[i], sigma=2.5)
        mx = g.max()
        if mx > 0.1:
            coords = np.array(np.where(g == mx)).flatten().tolist()
            assert got[i] is not None and got[i][0] == coords[1] and got[i][1] == coords[0] and got[i][2] == mx
        else:
            assert got[i] is None
