"""B200-native drop-in for the reference module `hand_detector` (reference hand_detector.py).

Same surface: `HandDetector(arch, weights_file, model, device)`, `__call__(hand_img, fast_mode=False, hand_type="right")`,
`compute_peaks_from_heatmaps`, `create_gaussian_kernel`, `draw_hand_keypoints`.  The whole numeric path --
cv2.resize of the crop to 368x368 (bit-exact uint8 INTER_LINEAR on the device), HandNet forward (tcgen05 conv chain),
F.resize_images back to the crop size, scipy gaussian_filter and the per-channel maximum -- runs as sm_100a CUDA
behind include/opb.h (opb_keypoints_detect).  `device < 0` selects GPU 0: there is no CPU path.
Unlike the reference (:13-16), `weights_file=None` keeps the seeded random init and `model=` is honoured."""
import os

import cv2
import numpy as np

try:
    from . import _native
    from .entity import params
    from .pose_detector import make_opb_params, _PRECISIONS
except ImportError:  # flat import, like the reference
    import _native
    from entity import params
    from pose_detector import make_opb_params, _PRECISIONS


class HandDetector(object):
    def __init__(self, arch=None, weights_file=None, model=None, device=-1, precision=None):
        print('Loading HandNet...')
        if model is not None:
            self.model = model
        else:
            self.model = params['archs'][arch]()
            if weights_file:
                self.model.load_npz(weights_file)
        self.device = device
        precision = precision if precision is not None else os.environ.get("OPB_PRECISION", "comp")
        self.engine = _native.Engine(max(int(device), 0), make_opb_params(params), _PRECISIONS[precision])
        self.engine.load_model(self.model)
        self.model._engine = self.engine
        self.gaussian_kernel = self.create_gaussian_kernel(sigma=params['gaussian_sigma'], ksize=params['ksize'])

    def __call__(self, hand_img, fast_mode=False, hand_type="right"):
        """hand_detector.py:28-51: list of 21 entries, [x, y, conf] in crop coordinates or None.  A left hand is
        mirrored into the network (:29-30) and its maps mirrored back (:46-47)."""
        left = hand_type == "left"
        if left:
            hand_img = cv2.flip(hand_img, 1)
        return self.engine.keypoints_detect(hand_img, params["hand_inference_img_size"],
                                            params['hand_heatmap_peak_thresh'], mirror=left)

    def detect_batch(self, hand_imgs, hand_types="right"):
        """[self(img, hand_type=t) for img, t in zip(hand_imgs, hand_types)], computed as one batch
        (opb_keypoints_detect_batch).  hand_types: one string for every crop, or one per crop; left crops are flipped
        here and reported in the flipped maps' coordinates, as __call__ does."""
        types = [hand_types] * len(hand_imgs) if isinstance(hand_types, str) else list(hand_types)
        if len(types) != len(hand_imgs):
            raise ValueError("%d hand types for %d crops" % (len(types), len(hand_imgs)))
        left = [t == "left" for t in types]
        crops = [cv2.flip(img, 1) if lf else img for img, lf in zip(hand_imgs, left)]
        return self.engine.keypoints_detect_batch(crops, params["hand_inference_img_size"],
                                                  params['hand_heatmap_peak_thresh'], left)

    def create_gaussian_kernel(self, sigma=1, ksize=5):
        """The 2-D kernel of the reference's GPU branch (hand_detector.py:44-52); kept for API compatibility --
        peak extraction here follows the CPU branch (scipy gaussian_filter) exactly."""
        ax = np.abs(np.arange(ksize) - int(ksize / 2))
        d2 = ax[None, :] ** 2 + ax[:, None] ** 2
        return (1 / (sigma ** 2 * 2 * np.pi) * np.exp(-d2 / (2 * sigma ** 2))).astype(np.float32)[None, None]

    def compute_peaks_from_heatmaps(self, heatmaps):
        """[C+1,H,W] maps (last = background) -> per keypoint [x, y, conf] or None (hand_detector.py:65-77)."""
        return self.engine.keypoints_from_heatmaps(np.asarray(heatmaps)[:-1], params['hand_heatmap_peak_thresh'])

_FINGER_COLORS = [(0, 0, 255), (0, 255, 255), (0, 255, 0), (255, 0, 0), (255, 0, 255)]


def draw_hand_keypoints(orig_img, hand_keypoints, left_top):
    """Finger polylines then joints, one colour per finger (hand_detector.py:79-111)."""
    img = orig_img.copy()
    left, top = left_top
    for i, finger in enumerate(params["fingers_indices"]):
        for a, b in finger:
            ka, kb = hand_keypoints[a], hand_keypoints[b]
            if ka:
                cv2.circle(img, (ka[0] + left, ka[1] + top), 3, _FINGER_COLORS[i], -1)
            if kb:
                cv2.circle(img, (kb[0] + left, kb[1] + top), 3, _FINGER_COLORS[i], -1)
            if ka and kb:
                cv2.line(img, (ka[0] + left, ka[1] + top), (kb[0] + left, kb[1] + top), _FINGER_COLORS[i], 1)
    return img
