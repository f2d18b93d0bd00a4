"""B200-native drop-in for the reference module `face_detector` (reference face_detector.py).

Same surface: `FaceDetector(arch, weights_file, model, device)`, `__call__(face_img, fast_mode=False)`,
`compute_peaks_from_heatmaps`, `create_gaussian_kernel`, `draw_face_keypoints`, `crop_face`.  The whole numeric path --
cv2.resize of the crop to 368x368 (bit-exact uint8 INTER_LINEAR on the device), FaceNet forward (tcgen05 conv chain),
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


class FaceDetector(object):
    def __init__(self, arch=None, weights_file=None, model=None, device=-1, precision=None):
        print('Loading FaceNet...')
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

    def __call__(self, face_img, fast_mode=False):
        """face_detector.py:28-41: list of 70 entries, [x, y, conf] in crop coordinates or None."""
        return self.engine.keypoints_detect(face_img, params["face_inference_img_size"],
                                            params['face_heatmap_peak_thresh'])

    def detect_batch(self, face_imgs):
        """[self(img) for img in face_imgs], computed as one batch (opb_keypoints_detect_batch)."""
        return self.engine.keypoints_detect_batch(face_imgs, params["face_inference_img_size"],
                                                  params['face_heatmap_peak_thresh'], False)

    def create_gaussian_kernel(self, sigma=1, ksize=5):
        """The 2-D kernel of the reference's GPU branch (face_detector.py:44-52); kept for API compatibility --
        peak extraction here follows the CPU branch (scipy gaussian_filter) exactly."""
        ax = np.abs(np.arange(ksize) - int(ksize / 2))
        d2 = ax[None, :] ** 2 + ax[:, None] ** 2
        return (1 / (sigma ** 2 * 2 * np.pi) * np.exp(-d2 / (2 * sigma ** 2))).astype(np.float32)[None, None]

    def compute_peaks_from_heatmaps(self, heatmaps):
        """[C+1,H,W] maps (last = background) -> per keypoint [x, y, conf] or None (face_detector.py:55-67)."""
        return self.engine.keypoints_from_heatmaps(np.asarray(heatmaps)[:-1], params['face_heatmap_peak_thresh'])

def draw_face_keypoints(orig_img, face_keypoints, left_top):
    """Dots and the 63 contour segments of entity.params['face_line_indices'] (face_detector.py:69-88)."""
    img = orig_img.copy()
    left, top = left_top
    for kp in face_keypoints:
        if kp:
            cv2.circle(img, (kp[0] + left, kp[1] + top), 2, (255, 255, 0), -1)
    for a, b in params["face_line_indices"]:
        ka, kb = face_keypoints[a], face_keypoints[b]
        if ka and kb:
            cv2.line(img, (ka[0] + left, ka[1] + top), (kb[0] + left, kb[1] + top), (255, 255, 0), 1)
    return img


def crop_face(img, rect):
    """Square, zero-padded crop around rect = (x, y, w, h) scaled by face_crop_scale (face_detector.py:90-105).
    Returns (padded_face, (crop_left, crop_top))."""
    h, w, _ = img.shape
    cx, cy = rect[0] + rect[2] / 2, rect[1] + rect[3] / 2
    cw, chh = rect[2] * params['face_crop_scale'], rect[3] * params['face_crop_scale']
    left, top = max(0, int(cx - cw / 2)), max(0, int(cy - chh / 2))
    right, bottom = min(w - 1, int(cx + cw / 2)), min(h - 1, int(cy + chh / 2))
    face = img[top:bottom, left:right]
    edge = np.max(face.shape[:-1])
    padded = np.zeros((edge, edge, face.shape[-1]), dtype=np.uint8)
    padded[0:face.shape[0], 0:face.shape[1]] = face
    return padded, (left, top)
