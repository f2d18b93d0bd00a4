"""ctypes binding of libopb.so (C ABI: include/opb.h).  Fails loudly when the CUDA library
is missing or no B200 is present -- there is no CPU fallback in this package."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OPB_LIB_PATH", os.path.join(HERE, "libopb.so"))   # OPB_LIB_PATH: A/B builds only

OPB_HOST, OPB_DEVICE = 0, 1
F32_NCHW, U8_NHWC_BGR = 0, 1
PRECISION_FAST, PRECISION_PARITY, PRECISION_COMP = 0, 1, 2
UPSAMPLE_BILINEAR_AC, UPSAMPLE_BICUBIC = 0, 1
ERR_CUDA, ERR_ARG, ERR_STATE, ERR_CAPACITY, ERR_INDEX, ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
N_JOINTS, N_LIMBS, MAX_TAPS = 18, 19, 64


class OpbParams(C.Structure):
    _fields_ = [("limbs", (C.c_int32 * 2) * N_LIMBS),
                ("heatmap_peak_thresh", C.c_double), ("inner_product_thresh", C.c_double),
                ("limb_length_ratio", C.c_double), ("length_penalty_value", C.c_double),
                ("n_subset_limbs_thresh", C.c_double), ("subset_score_thresh", C.c_double),
                ("n_integ_points", C.c_int32), ("n_integ_points_thresh", C.c_int32),
                ("gauss_radius", C.c_int32), ("reserved0", C.c_int32),
                ("gauss_taps", C.c_double * MAX_TAPS),
                ("max_peaks", C.c_int32), ("max_candidates", C.c_int32), ("max_persons", C.c_int32),
                ("reserved1", C.c_int32)]


PERSON_DTYPE = np.dtype([("score", "<f8"), ("count", "<f8"), ("peak_id", "<i4", (N_JOINTS,)),
                         ("x", "<i4", (N_JOINTS,)), ("y", "<i4", (N_JOINTS,)), ("pad", "<i4", (2,))])
HEADER_DTYPE = np.dtype([("n_peaks", "<i4"), ("n_persons", "<i4"), ("status", "<i4"), ("n_connections", "<i4")])
assert PERSON_DTYPE.itemsize == 240 and HEADER_DTYPE.itemsize == 16

_SIGNATURES = {
    "opb_version": (C.c_int, []),
    "opb_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(OpbParams)]),
    "opb_destroy": (None, [C.c_void_p]),
    "opb_last_error": (C.c_char_p, [C.c_void_p]),
    "opb_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "opb_synchronize": (C.c_int, [C.c_void_p]),
    "opb_load_weights": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "opb_finalize_weights": (C.c_int, [C.c_void_p, C.c_int]),
    "opb_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                              C.c_void_p, C.c_int]),
    "opb_upsample": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                               C.c_int, C.c_int, C.c_int]),
    "opb_peaks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                            C.POINTER(C.c_int)]),
    "opb_connections": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                  C.c_double, C.c_void_p, C.c_int, C.c_void_p]),
    "opb_candidates": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                 C.c_double, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "opb_group": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                            C.POINTER(C.c_int)]),
    "opb_detect_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_postprocess_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_resize_linear_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                       C.c_int, C.c_int]),
    "opb_resize_cubic_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                      C.c_int, C.c_int]),
    "opb_precise_add_scale_orig": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_int, C.c_int]),
    "opb_detect_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_double, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_draw_person_pose": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                       C.c_int]),
    "opb_draw_last_result": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                       C.c_void_p, C.c_int]),
    "opb_stream_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_stream_collect": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "opb_stream_join": (C.c_int, [C.c_void_p]),
    "opb_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "opb_nccl_comm_init": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p]),
    "opb_nccl_comm_destroy": (C.c_int, [C.c_void_p]),
    "opb_record_block_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "opb_allgather_results": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "opb_keypoints_detect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "opb_keypoints_from_heatmaps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_double, C.c_void_p, C.c_void_p]),
    "opb_keypoints_detect_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                             C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "opb_precise_add_scale_unpadded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                 C.c_int, C.c_int]),
    "opb_get_image_detail": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "opb_precise_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "opb_precise_add_scale": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int]),
    "opb_precise_finish": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_download_maps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "opb_device_buffer": (C.c_void_p, [C.c_void_p, C.c_int]),
    "opb_launch_count": (C.c_int64, [C.c_void_p]),
    "opb_time_stage": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_float)]),
    "opb_test_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


def load_library():
    """dlopen libopb.so and declare every symbol of include/opb.h (no GPU needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError("libopb.so is missing (%s). Build it with `python __graft_entry__.py build` "
                           "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else int(a))


class OpbError(RuntimeError):
    pass


class Engine(object):
    """One device context (opb_ctx) + the weights of one CocoPoseNet."""

    def __init__(self, device, params, precision=PRECISION_COMP):
        self.lib = load_library()
        self.ctx = C.c_void_p()
        self.params = params
        self.max_peaks, self.max_persons = params.max_peaks, params.max_persons
        rc = self.lib.opb_create(C.byref(self.ctx), int(device), C.byref(params))
        if rc != 0:
            msg = self.lib.opb_last_error(None)
            self.ctx = None
            raise OpbError("opb_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.precision = precision
        self._weights_ready = False

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.opb_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    def _check(self, rc):
        if rc == 0:
            return
        msg = self.lib.opb_last_error(self.ctx)
        msg = msg.decode() if msg else ""
        if rc == ERR_INDEX:
            raise IndexError(msg or "list assignment index out of range")   # pose_detector.py:197
        raise OpbError("libopb error %d: %s" % (rc, msg))

    def raise_for_status(self, status):
        if status == 0:
            return
        if status == ERR_INDEX:
            raise IndexError("list assignment index out of range")
        raise OpbError("device post-process status %d (capacity exceeded: raise max_peaks / max_candidates / "
                       "max_persons)" % status)

    # -- weights ---------------------------------------------------------------------------
    def load_model(self, model, precision=None):
        """model: object with children_items() -> (name, link with .W.data/.b.data)."""
        if precision is not None:
            self.precision = precision
        for name, link in model.children_items():
            W = np.ascontiguousarray(link.W.data, np.float32)
            b = np.ascontiguousarray(link.b.data, np.float32)
            shape = (C.c_int64 * 4)(*W.shape)
            self._check(self.lib.opb_load_weights(self.ctx, name.encode(), _ptr(W), shape, _ptr(b)))
        self._check(self.lib.opb_finalize_weights(self.ctx, int(self.precision)))
        self._weights_ready = True
        last = dict(model.children_items()).get("conv6_2_CPM")      # FaceNet / HandNet: channels of the final maps
        self.kp_channels = int(last.W.data.shape[0]) if last is not None else 0

    def set_stream(self, stream_handle):
        self._check(self.lib.opb_set_stream(self.ctx, C.c_void_p(int(stream_handle) if stream_handle else 0)))

    def synchronize(self):
        self._check(self.lib.opb_synchronize(self.ctx))

    # -- forward ----------------------------------------------------------------------------
    def forward(self, x):
        """x: [N,3,H,W] float32 (preprocessed) or [N,H,W,3] uint8 BGR.  Returns numpy
        (paf [N,38,h,w], heat [N,19,h,w])."""
        x = np.ascontiguousarray(x)
        if x.dtype == np.uint8:
            n, h, w, _ = x.shape
            fmt = U8_NHWC_BGR
        else:
            x = np.ascontiguousarray(x, np.float32)
            n, _, h, w = x.shape
            fmt = F32_NCHW
        paf = np.empty((n, 38, h // 8, w // 8), np.float32)
        heat = np.empty((n, 19, h // 8, w // 8), np.float32)
        self._check(self.lib.opb_forward(self.ctx, _ptr(x), fmt, OPB_HOST, n, h, w, _ptr(paf), _ptr(heat), OPB_HOST))
        return paf, heat

    def upsample(self, maps, out_h, out_w, mode=UPSAMPLE_BILINEAR_AC):
        maps = np.ascontiguousarray(maps, np.float32)
        lead = maps.shape[:-2]
        h, w = maps.shape[-2:]
        planes = int(np.prod(lead)) if lead else 1
        out = np.empty(lead + (out_h, out_w), np.float32)
        self._check(self.lib.opb_upsample(self.ctx, mode, _ptr(maps), OPB_HOST, planes, h, w, _ptr(out), OPB_HOST,
                                          out_h, out_w))
        return out

    # -- stage methods ------------------------------------------------------------------------
    def peaks(self, heatmaps):
        hm = np.ascontiguousarray(heatmaps, np.float32)
        c1, h, w = hm.shape
        out = np.empty((self.max_peaks, 5), np.float64)
        n = C.c_int(0)
        self._check(self.lib.opb_peaks(self.ctx, _ptr(hm), OPB_HOST, c1, h, w, _ptr(out), self.max_peaks, C.byref(n)))
        return out[:n.value].copy()

    def connections(self, pafs, all_peaks, img_len):
        pafs = np.ascontiguousarray(pafs, np.float32)
        _, h, w = pafs.shape
        pk = np.ascontiguousarray(all_peaks, np.float64).reshape(-1, 5)
        cap = max(len(pk), 1) * 2
        out = np.empty((cap, 3), np.float64)
        counts = np.zeros(N_LIMBS, np.int32)
        self._check(self.lib.opb_connections(self.ctx, _ptr(pafs), OPB_HOST, h, w, _ptr(pk), len(pk), float(img_len),
                                             _ptr(out), cap, _ptr(counts)))
        res, o = [], 0
        for c in counts:
            res.append(out[o:o + c].copy() if c else np.zeros((0, 3)))
            o += int(c)
        return res

    def candidates(self, paf, cand_a, cand_b, img_len):
        paf = np.ascontiguousarray(paf, np.float32)
        _, h, w = paf.shape
        a = np.ascontiguousarray(cand_a, np.float64).reshape(-1, 4)
        b = np.ascontiguousarray(cand_b, np.float64).reshape(-1, 4)
        cap = max(len(a) * len(b), 1)
        out = np.empty((cap, 3), np.float64)
        n = C.c_int(0)
        self._check(self.lib.opb_candidates(self.ctx, _ptr(paf), h, w, _ptr(a), len(a), _ptr(b), len(b), float(img_len),
                                            _ptr(out), cap, C.byref(n)))
        return out[:n.value].copy()

    def group(self, all_connections, peaks):
        pk = np.ascontiguousarray(peaks, np.float64).reshape(-1, 5)
        counts = np.array([len(c) for c in all_connections], np.int32)
        flat = (np.concatenate([np.asarray(c, np.float64).reshape(-1, 3) for c in all_connections], axis=0)
                if counts.sum() else np.zeros((0, 3)))
        flat = np.ascontiguousarray(flat[:, :3], np.float64)
        out = np.empty((self.max_persons, 20), np.float64)
        n = C.c_int(0)
        self._check(self.lib.opb_group(self.ctx, _ptr(flat), _ptr(counts), _ptr(pk), len(pk), _ptr(out),
                                       self.max_persons, C.byref(n)))
        return out[:n.value].copy()

    # -- fused batch path -------------------------------------------------------------------
    def detect_batch(self, imgs, map_h, map_w, img_len=None, inject_paf=None, inject_heat=None, imgs_ptr=None,
                     headers=None, persons=None):
        """imgs: [N,H,W,3] uint8 BGR (network-input size) host array, or a device pointer via
        imgs_ptr=(ptr, n, h, w).  inject_*: device pointers (ints) or None."""
        if imgs_ptr is not None:
            ptr, n, h, w = imgs_ptr
            src, loc = C.c_void_p(int(ptr)), OPB_DEVICE
        else:
            imgs = np.ascontiguousarray(imgs, np.uint8)
            n, h, w, _ = imgs.shape
            src, loc = _ptr(imgs), OPB_HOST
        if headers is None:
            headers = np.empty(n, HEADER_DTYPE)
        if persons is None:
            persons = np.empty((n, self.max_persons), PERSON_DTYPE)
        self._check(self.lib.opb_detect_batch(self.ctx, src, loc, n, h, w, map_h, map_w,
                                              float(map_w if img_len is None else img_len),
                                              C.c_void_p(int(inject_paf)) if inject_paf else None,
                                              C.c_void_p(int(inject_heat)) if inject_heat else None,
                                              _ptr(headers), _ptr(persons), OPB_HOST))
        return headers, persons

    def postprocess_batch(self, paf_lo, heat_lo, map_h, map_w, img_len=None):
        """Network outputs paf_lo [N,38,h8,w8] / heat_lo [N,19,h8,w8] float32 (host) -> (headers[N],
        persons[N, max_persons]): upsample, peaks, connections, grouping (opb_postprocess_batch)."""
        paf_lo = np.ascontiguousarray(paf_lo, np.float32)
        heat_lo = np.ascontiguousarray(heat_lo, np.float32)
        n, _, h8, w8 = paf_lo.shape
        assert paf_lo.shape[1] == 38 and heat_lo.shape == (n, 19, h8, w8)
        headers = np.empty(n, HEADER_DTYPE)
        persons = np.empty((n, self.max_persons), PERSON_DTYPE)
        self._check(self.lib.opb_postprocess_batch(self.ctx, _ptr(paf_lo), _ptr(heat_lo), OPB_HOST, n, h8, w8, map_h, map_w,
                                                   float(map_w if img_len is None else img_len), _ptr(headers),
                                                   _ptr(persons), OPB_HOST))
        return headers, persons

    def resize_linear_u8(self, imgs, out_h, out_w):
        """cv2.resize(img, (out_w, out_h)) (INTER_LINEAR, uint8) on the device; imgs [N,H,W,3] or [H,W,3]."""
        a = np.ascontiguousarray(imgs, np.uint8)
        single = a.ndim == 3
        if single:
            a = a[None]
        n, h0, w0, _ = a.shape
        out = np.empty((n, out_h, out_w, 3), np.uint8)
        self._check(self.lib.opb_resize_linear_u8(self.ctx, _ptr(a), OPB_HOST, n, h0, w0, _ptr(out), OPB_HOST, out_h, out_w))
        return out[0] if single else out

    def resize_cubic_u8(self, imgs, out_h, out_w):
        """cv2.resize(img, (out_w, out_h), interpolation=cv2.INTER_CUBIC) (uint8, OpenCV's own non-IPP path) on the
        device; imgs [N,H,W,3] or [H,W,3]."""
        a = np.ascontiguousarray(imgs, np.uint8)
        single = a.ndim == 3
        if single:
            a = a[None]
        n, h0, w0, _ = a.shape
        out = np.empty((n, out_h, out_w, 3), np.uint8)
        self._check(self.lib.opb_resize_cubic_u8(self.ctx, _ptr(a), OPB_HOST, n, h0, w0, _ptr(out), OPB_HOST, out_h, out_w))
        return out[0] if single else out

    def draw_person_pose(self, img, poses):
        """draw_person_pose(orig_img, poses) (pose_detector.py:520-553) on the device; poses float [P,18,3]."""
        a = np.ascontiguousarray(img, np.uint8)
        h, w, _ = a.shape
        ip = np.ascontiguousarray(np.asarray(poses).round().astype('i').reshape(-1, 18, 3), np.int32)
        out = np.empty_like(a)
        self._check(self.lib.opb_draw_person_pose(self.ctx, _ptr(a), OPB_HOST, h, w, _ptr(ip) if len(ip) else None, len(ip),
                                                  _ptr(out), OPB_HOST))
        return out

    def draw_last_result(self, img, sx, sy, image_index=0):
        """Overlay of the persons of the last detect call, taken from the device-resident records."""
        a = np.ascontiguousarray(img, np.uint8)
        h, w, _ = a.shape
        out = np.empty_like(a)
        self._check(self.lib.opb_draw_last_result(self.ctx, int(image_index), _ptr(a), OPB_HOST, h, w, float(sx), float(sy),
                                                  _ptr(out), OPB_HOST))
        return out

    def detect_image(self, img, in_h, in_w, map_h, map_w, img_len=None):
        """One BGR frame of any size: upload, device resize, full pipeline (opb_detect_image)."""
        img = np.ascontiguousarray(img, np.uint8)
        oh, ow, _ = img.shape
        headers = np.empty(1, HEADER_DTYPE)
        persons = np.empty((1, self.max_persons), PERSON_DTYPE)
        self._check(self.lib.opb_detect_image(self.ctx, _ptr(img), OPB_HOST, oh, ow, in_h, in_w, map_h, map_w,
                                              float(map_w if img_len is None else img_len), _ptr(headers),
                                              _ptr(persons), OPB_HOST))
        return headers, persons

    def stream_submit(self, frames, in_h, in_w, map_h, map_w, slot, img_len=None, inject_paf=None, inject_heat=None,
                      device=False):
        """Enqueue one batch [N,H0,W0,3] uint8 on `slot` (0/1) without waiting (opb_stream_submit).  `frames`: a
        NumPy array (host), or (address, n, h, w) of a pinned host buffer -- or of a device buffer with device=True."""
        if isinstance(frames, np.ndarray):
            frames = np.ascontiguousarray(frames, np.uint8)
            if frames.ndim == 3:
                frames = frames[None]
            n, oh, ow, _ = frames.shape
            ptr = _ptr(frames)
            self._stream_keep = getattr(self, "_stream_keep", {})
            self._stream_keep[slot] = frames          # pinned buffers are read asynchronously: keep them alive
        else:                                         # (data_ptr, n, h, w) of a pinned buffer owned by the caller
            addr, n, oh, ow = frames
            ptr = C.c_void_p(addr)
        self._stream_n = getattr(self, "_stream_n", {})
        self._stream_n[slot] = n
        self._check(self.lib.opb_stream_submit(self.ctx, ptr, OPB_DEVICE if device else OPB_HOST, n, oh, ow, in_h, in_w,
                                               map_h, map_w,
                                               float(map_w if img_len is None else img_len),
                                               C.c_void_p(inject_paf or 0), C.c_void_p(inject_heat or 0), slot))

    # ---- multi-GPU: the ONE collective of the path (include/opb.h: opb_allgather_results)
    def nccl_unique_id(self):
        """128-byte NCCL id (rank 0 creates it and ships it to the other ranks, e.g. torch.distributed.broadcast)."""
        buf = np.zeros(128, np.uint8)
        rc = self.lib.opb_nccl_unique_id(C.c_void_p(buf.ctypes.data))
        if rc:
            raise OpbError("opb_nccl_unique_id failed (%d): %s" % (rc, (self.lib.opb_last_error(None) or b"").decode()))
        return buf

    def nccl_comm_init(self, world, rank, unique_id):
        comm = C.c_void_p()
        uid = np.ascontiguousarray(unique_id, np.uint8)
        self._check(self.lib.opb_nccl_comm_init(self.ctx, C.byref(comm), int(world), int(rank), C.c_void_p(uid.ctypes.data)))
        self._nccl_comm = comm
        return comm

    def record_block_bytes(self, n):
        return int(self.lib.opb_record_block_bytes(self.ctx, int(n)))

    def allgather_results(self, slot, gathered_dev_ptr, comm=None):
        """ncclAllGather of streaming slot `slot`'s device-resident record block into the device buffer at
        gathered_dev_ptr (world x record_block_bytes(n) bytes), on the slot's stream behind its pipeline."""
        self._check(self.lib.opb_allgather_results(self.ctx, comm if comm is not None else self._nccl_comm, int(slot),
                                                   C.c_void_p(int(gathered_dev_ptr))))

    def stream_join(self):
        """Make the context's stream wait for every submitted, uncollected batch (opb_stream_join)."""
        self._check(self.lib.opb_stream_join(self.ctx))

    def stream_collect(self, slot):
        """Block until the batch submitted on `slot` is done; returns (headers[N], persons[N, max_persons])."""
        n = self._stream_n[slot]
        headers = np.empty(n, HEADER_DTYPE)
        persons = np.empty((n, self.max_persons), PERSON_DTYPE)
        self._check(self.lib.opb_stream_collect(self.ctx, slot, _ptr(headers), _ptr(persons)))
        return headers, persons

    # -- face / hand nets (include/opb.h: opb_keypoints_*) ---------------------------------------
    def forward_keypoint_maps(self, x, n_out=None):
        """FaceNet / HandNet forward: x [N,3,H,W] float32 (already /256 - 0.5) or [N,H,W,3] uint8 -> [N,C,h,w]."""
        x = np.ascontiguousarray(x)
        if x.dtype == np.uint8:
            n, h, w, _ = x.shape
            fmt = U8_NHWC_BGR
        else:
            x = np.ascontiguousarray(x, np.float32)
            n, _, h, w = x.shape
            fmt = F32_NCHW
        heat = np.empty((n, n_out or self.kp_channels, h // 8, w // 8), np.float32)
        self._check(self.lib.opb_forward(self.ctx, _ptr(x), fmt, OPB_HOST, n, h, w, None, _ptr(heat), OPB_HOST))
        return heat

    @staticmethod
    def _keypoint_list(out, valid):
        return [[int(x), int(y), np.float32(c)] if v else None for (x, y, c), v in zip(out, valid)]

    def keypoints_detect(self, img, net_size, thresh, mirror=False, return_maps=False):
        """One BGR crop -> list of [x, y, conf] / None per keypoint channel (opb_keypoints_detect)."""
        img = np.ascontiguousarray(img, np.uint8)
        h, w, _ = img.shape
        planes = self.kp_channels - 1
        out = np.empty((planes, 3), np.float64)
        valid = np.empty(planes, np.int32)
        maps = np.empty((planes, h, w), np.float32) if return_maps else None
        self._check(self.lib.opb_keypoints_detect(self.ctx, _ptr(img), OPB_HOST, h, w, net_size, int(bool(mirror)),
                                                  float(thresh), _ptr(out), _ptr(valid),
                                                  _ptr(maps) if return_maps else None))
        kps = self._keypoint_list(out, valid)
        return (kps, maps) if return_maps else kps

    def keypoints_detect_batch(self, imgs, net_size, thresh, mirrors, return_maps=False):
        """A list of BGR crops of any sizes -> one keypoint list per crop, as keypoints_detect returns it, from one
        upload, one forward and one launch per post-process stage (opb_keypoints_detect_batch).  `mirrors`: one flag
        for all crops or one per crop.  With return_maps, also the [C-1, h_i, w_i] maps of every crop."""
        crops = [np.ascontiguousarray(a, np.uint8) for a in imgs]
        n = len(crops)
        mirror = np.array([bool(mirrors)] * n if np.ndim(mirrors) == 0 else [bool(m) for m in mirrors], np.int32)
        if len(mirror) != n:
            raise ValueError("%d mirror flags for %d crops" % (len(mirror), n))
        dims = np.array([a.shape[:2] for a in crops], np.int32).reshape(n, 2)
        packed = np.concatenate([a.ravel() for a in crops]) if n else np.zeros(0, np.uint8)
        planes = self.kp_channels - 1
        out = np.empty((n, planes, 3), np.float64)
        valid = np.empty((n, planes), np.int32)
        sizes = [planes * int(h) * int(w) for h, w in dims]
        maps = np.empty(sum(sizes), np.float32) if return_maps else None
        self._check(self.lib.opb_keypoints_detect_batch(self.ctx, _ptr(packed), OPB_HOST, n, _ptr(dims), _ptr(mirror),
                                                        int(net_size), float(thresh), _ptr(out), _ptr(valid),
                                                        _ptr(maps)))
        kps = [self._keypoint_list(out[i], valid[i]) for i in range(n)]
        if not return_maps:
            return kps
        ends = np.cumsum(sizes)
        return kps, [maps[e - s:e].reshape(planes, int(h), int(w)) for e, s, (h, w) in zip(ends, sizes, dims)]

    def keypoints_from_heatmaps(self, heatmaps, thresh, mirror=False):
        """heatmaps [C,H,W] float32, background channel already dropped (opb_keypoints_from_heatmaps)."""
        hm = np.ascontiguousarray(heatmaps, np.float32)
        planes, h, w = hm.shape
        out = np.empty((planes, 3), np.float64)
        valid = np.empty(planes, np.int32)
        self._check(self.lib.opb_keypoints_from_heatmaps(self.ctx, _ptr(hm), OPB_HOST, planes, h, w, int(bool(mirror)),
                                                         float(thresh), _ptr(out), _ptr(valid)))
        return self._keypoint_list(out, valid)

    def image_detail(self, img):
        pk = np.empty((self.max_peaks, 5), np.float64)
        n_pk, n_sub = C.c_int(0), C.c_int(0)
        cap = 19 * 1024
        conn = np.empty((cap, 3), np.float64)
        counts = np.zeros(N_LIMBS, np.int32)
        subs = np.empty((self.max_persons, 20), np.float64)
        self._check(self.lib.opb_get_image_detail(self.ctx, img, _ptr(pk), self.max_peaks, C.byref(n_pk), _ptr(conn),
                                                  cap, _ptr(counts), _ptr(subs), self.max_persons, C.byref(n_sub)))
        conns, o = [], 0
        for c in counts:
            conns.append(conn[o:o + c].copy() if c else np.zeros((0, 3)))
            o += int(c)
        return pk[:n_pk.value].copy(), conns, subs[:n_sub.value].copy()

    # -- precise path -----------------------------------------------------------------------
    def precise_begin(self, orig_h, orig_w):
        self._check(self.lib.opb_precise_begin(self.ctx, orig_h, orig_w))

    def precise_add_scale_unpadded(self, img, stride, pad_value, scale_index, n_scales):
        """Resized but unpadded uint8 frame; pad_image (pose_detector.py:46-55) runs on the device."""
        img = np.ascontiguousarray(img, np.uint8)
        h, w, _ = img.shape
        pv = (C.c_uint8 * 3)(*[int(v) for v in pad_value])
        self._check(self.lib.opb_precise_add_scale_unpadded(self.ctx, _ptr(img), OPB_HOST, h, w, int(stride), pv,
                                                            scale_index, n_scales))

    def precise_add_scale_orig(self, orig_img, h, w, stride, pad_value, scale_index, n_scales):
        """Original uint8 frame; the cubic resize to (h, w) of pose_detector.py:443 and pad_image run on the device."""
        img = np.ascontiguousarray(orig_img, np.uint8)
        oh, ow, _ = img.shape
        pv = (C.c_uint8 * 3)(*[int(v) for v in pad_value])
        self._check(self.lib.opb_precise_add_scale_orig(self.ctx, _ptr(img), OPB_HOST, oh, ow, int(h), int(w), int(stride),
                                                        pv, scale_index, n_scales))

    def precise_add_scale(self, padded_img, pad, scale_index, n_scales):
        img = np.ascontiguousarray(padded_img, np.uint8)
        ph, pw, _ = img.shape
        self._check(self.lib.opb_precise_add_scale(self.ctx, _ptr(img), OPB_HOST, ph, pw, int(pad[0]), int(pad[1]),
                                                   scale_index, n_scales))

    def precise_finish(self, img_len):
        headers = np.empty(1, HEADER_DTYPE)
        persons = np.empty((1, self.max_persons), PERSON_DTYPE)
        self._check(self.lib.opb_precise_finish(self.ctx, float(img_len), _ptr(headers), _ptr(persons), OPB_HOST))
        return headers, persons

    def download_maps(self, h, w):
        pafs = np.empty((38, h, w), np.float32)
        heat = np.empty((19, h, w), np.float32)
        self._check(self.lib.opb_download_maps(self.ctx, _ptr(pafs), _ptr(heat), OPB_HOST))
        return pafs, heat

    # -- instrumentation ----------------------------------------------------------------------
    def device_buffer(self, which):
        return self.lib.opb_device_buffer(self.ctx, which)

    def launch_count(self):
        return int(self.lib.opb_launch_count(self.ctx))

    def time_stage(self, stage, reps=10):
        ms = C.c_float(0)
        self._check(self.lib.opb_time_stage(self.ctx, stage.encode(), reps, C.byref(ms)))
        return float(ms.value)

    def test_conv(self, x, W, b, relu, precision, pool=False):
        x = np.ascontiguousarray(x, np.float32)
        W = np.ascontiguousarray(W, np.float32)
        b = np.ascontiguousarray(b, np.float32)
        n, h, w, cin = x.shape
        cout, _, ks, _ = W.shape
        y = np.empty((n, h // 2, w // 2, cout) if pool else (n, h, w, cout), np.float32)
        self._check(self.lib.opb_test_conv(self.ctx, _ptr(x), n, h, w, cin, _ptr(W), _ptr(b), cout, ks,
                                           int(bool(relu)) | (2 if pool else 0), int(precision), _ptr(y)))
        return y
