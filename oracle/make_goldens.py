"""ORACLE / TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the
reference's OWN files verbatim (oracle/reference_loader.py) on seeded synthetic inputs.
Run in the build container only (needs /root/reference):

    python oracle/make_goldens.py

The reference has no tests or golden vectors of its own (SURVEY.md section 4); these files are
the pin for oracle/restate.py and for the CUDA path.  Inputs are regenerated from seeds at
test time (weights 209 MB / images are never committed; data/*.png may not be copied).
"""
import hashlib
import importlib
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_loader  # noqa: E402

syn = importlib.import_module("chainer_realtime_multi-person_pose_estimation_b200.synthetic")
GOLD = os.path.join(ROOT, "tests", "golden")
# torch CPU threads the goldens are made with: oneDNN splits some convolutions' sums differently at other counts (1, or
# 16 and more), which changes the last bits of the maps, so the tests that compare bit for bit use this count too
TORCH_THREADS = 8


def conns_to_arrays(conns):
    lens = np.array([len(c) for c in conns], np.int64)
    flat = np.concatenate([np.asarray(c, np.float64).reshape(-1, 3) for c in conns], axis=0)
    return lens, flat


def capture_fast(ref, det, img):
    """Runs PoseDetector.__call__ while recording the intermediate arrays."""
    rec = {}
    model = det.model
    orig_call = type(model).__call__

    def wrapped(self, x):
        h1s, h2s = orig_call(self, x)
        rec.setdefault("paf_lo", []).append(np.array(h1s[-1].data[0]))
        rec.setdefault("heat_lo", []).append(np.array(h2s[-1].data[0]))
        return h1s, h2s

    o_peaks, o_conn, o_group = det.compute_peaks_from_heatmaps, det.compute_connections, det.grouping_key_points

    def peaks(hm):
        r = o_peaks(hm); rec["all_peaks"] = np.array(r, np.float64).copy(); return r

    def conn(p, a, l, prm):
        r = o_conn(p, a, l, prm); rec["conn"] = [np.array(c) for c in r]; rec["img_len"] = l; return r

    def group(c, a, prm):
        r = o_group(c, a, prm); rec["subsets"] = np.array(r).copy(); return r

    type(model).__call__ = wrapped
    det.compute_peaks_from_heatmaps, det.compute_connections, det.grouping_key_points = peaks, conn, group
    try:
        poses, scores = det(img)
    finally:
        type(model).__call__ = orig_call
        det.compute_peaks_from_heatmaps, det.compute_connections, det.grouping_key_points = o_peaks, o_conn, o_group
    rec["poses"], rec["scores"] = np.asarray(poses, np.float64), np.asarray(scores, np.float64)
    return rec


def pack(rec, extra=None):
    out = dict(extra or {})
    out["poses"], out["scores"] = rec["poses"], rec["scores"]
    out["all_peaks"] = rec.get("all_peaks", np.zeros((0, 5)))
    if out["all_peaks"].ndim != 2:
        out["all_peaks"] = np.zeros((0, 5))
    if "conn" in rec:
        out["conn_lens"], out["conn_flat"] = conns_to_arrays(rec["conn"])
        out["subsets"] = rec["subsets"]
        out["img_len"] = np.float64(rec["img_len"])
    for k in ("paf_lo", "heat_lo"):
        if k in rec:
            for i, a in enumerate(rec[k]):
                out["%s_%d" % (k, i)] = a.astype(np.float32)
    return out


def main():
    ref = reference_loader.load()
    os.makedirs(GOLD, exist_ok=True)
    tmp = tempfile.mkdtemp()
    he = os.path.join(tmp, "he0.npz")
    np.savez(he, **syn.he_weights(0))
    lecun = os.path.join(tmp, "lecun0.npz")
    np.savez(lecun, **syn.he_weights(0, bias_scale=0.0, gain=1.0))

    t0 = time.time()
    det = ref.PoseDetector("posenet", he)
    # G1: square 584x584 stand-in for data/person.png, fast path
    img = syn.procedural_image(584, 584, seed=1)
    np.savez_compressed(os.path.join(GOLD, "fast_584_he0.npz"), **pack(capture_fast(ref, det, img)))
    print("G1", time.time() - t0)
    # G3: two 368x656 noise frames (BASELINE shape), fast path
    imgs = syn.random_images(2, 368, 656, seed=0)
    for i in range(2):
        np.savez_compressed(os.path.join(GOLD, "fast_368x656_he0_img%d.npz" % i),
                            **pack(capture_fast(ref, det, imgs[i])))
    print("G3", time.time() - t0)
    # G6: a non-multiple-of-8 landscape frame (640x480 webcam shape, camera_pose_demo.py:16-18)
    img = syn.procedural_image(480, 640, seed=2)
    np.savez_compressed(os.path.join(GOLD, "fast_480x640_he0.npz"), **pack(capture_fast(ref, det, img)))
    print("G6", time.time() - t0)
    # G2: Chainer-default-like init (sigma = sqrt(1/fan_in), b = 0): zero peaks, empty return
    det0 = ref.PoseDetector("posenet", lecun)
    img = syn.procedural_image(584, 584, seed=1)
    np.savez_compressed(os.path.join(GOLD, "fast_584_lecun0.npz"), **pack(capture_fast(ref, det0, img)))
    print("G2", time.time() - t0)
    # G4: synthetic 8-person maps, post-process only (reference functions called directly)
    for seed in (0, 1):
        paf, heat, joints = syn.eight_person_maps(seed=seed)
        peaks = det.compute_peaks_from_heatmaps(heat)
        conns = det.compute_connections(paf, peaks, 576, ref.params)
        subsets = det.grouping_key_points(conns, peaks, ref.params)
        lens, flat = conns_to_arrays(conns)
        np.savez_compressed(os.path.join(GOLD, "synth8_post_seed%d.npz" % seed), all_peaks=peaks,
                            conn_lens=lens, conn_flat=flat, subsets=subsets, joints=joints,
                            poses=det.subsets_to_pose_array(subsets, peaks))
    print("G4", time.time() - t0)
    precise_480(ref, he)
    print("G5", time.time() - t0)
    precise_padded(ref, he)
    host_helper_goldens()


def precise_480(ref, he):
    # G5: multi-scale precise path on a 480x480 stand-in for data/people.png
    detp = ref.PoseDetector("posenet", he, precise=True)
    img = syn.procedural_image(480, 480, seed=3)
    rec = capture_fast(ref, detp, img)
    out = pack(rec)
    out["all_peaks"] = np.asarray(detp.all_peaks, np.float64)
    # full-resolution averaged maps are 52 MB; keep a strided sample for float checks (a stride of 9 keeps the file
    # under 1 MB) and drop the per-scale network outputs, which no test reads
    out["pafs_sample"] = detp.pafs[:, ::9, ::9].astype(np.float32)
    out["heatmaps_sample"] = detp.heatmaps[:, ::9, ::9].astype(np.float32)
    for k in list(out):
        if k.startswith("paf_lo_") or k.startswith("heat_lo_"):
            del out[k]
    np.savez_compressed(os.path.join(GOLD, "precise_480_he0.npz"), **out)


def keypoint_goldens():
    """G8/G9: FaceDetector / HandDetector (face_detector.py:28-41, hand_detector.py:28-51) run verbatim on
    seeded crops with He-initialised FaceNet / HandNet weights (seed 0)."""
    tmp = tempfile.mkdtemp()
    mods = {"face": importlib.import_module("chainer_realtime_multi-person_pose_estimation_b200.models.FaceNet"),
            "hand": importlib.import_module("chainer_realtime_multi-person_pose_estimation_b200.models.HandNet")}
    cases = [("face", reference_loader.load_face, "FaceDetector", "facenet", (150, 170, 11), {}),
             ("face", reference_loader.load_face, "FaceDetector", "facenet", (401, 401, 12), {}),
             ("hand", reference_loader.load_hand, "HandDetector", "handnet", (120, 131, 13), {"hand_type": "right"}),
             ("hand", reference_loader.load_hand, "HandDetector", "handnet", (120, 131, 13), {"hand_type": "left"})]
    dets = {}
    for kind, loader, cls, arch, (h, w, seed), kw in cases:
        if kind not in dets:
            f = os.path.join(tmp, kind + ".npz")
            np.savez(f, **syn.he_weights(0, layers=mods[kind].LAYERS))
            dets[kind] = getattr(loader(), cls)(arch, f, device=-1)
        det = dets[kind]
        rec = {}
        model = det.model
        orig_call = type(model).__call__

        def wrapped(self, x, _o=orig_call, _r=rec):
            hs = _o(self, x)
            _r["heat_lo"] = np.array(hs[-1].data[0], np.float32)
            return hs

        type(model).__call__ = wrapped
        try:
            kps = det(syn.procedural_image(h, w, seed=seed), **kw)
        finally:
            type(model).__call__ = orig_call
        valid = np.array([k is not None for k in kps])
        xy = np.array([[k[0], k[1]] if k is not None else [-1, -1] for k in kps], np.int64)
        conf = np.array([k[2] if k is not None else 0 for k in kps], np.float32)
        name = "%s_%dx%d_he0%s.npz" % (kind, h, w, "_" + kw["hand_type"] if kw else "")
        np.savez_compressed(os.path.join(GOLD, name), heat_lo=rec["heat_lo"], valid=valid, xy=xy, conf=conf,
                            img_hw_seed=np.array([h, w, seed]))
        print(name, int(valid.sum()), "of", len(kps))


def digest(obj):
    """Comparable summary of a helper's return value: the same nesting of dicts / lists / None, every array (or
    scalar) replaced by its shape and a hash of its values as float64 -- two results have equal digests exactly when
    they have the same structure and np.array_equal holds leaf by leaf."""
    if obj is None:
        return None
    if isinstance(obj, dict):
        return {str(k): digest(v) for k, v in sorted(obj.items())}
    if isinstance(obj, (tuple, list)):
        return [digest(x) for x in obj]
    a = np.ascontiguousarray(np.asarray(obj), np.float64)
    return "%s:%s" % ("x".join(map(str, a.shape)), hashlib.sha256(a.tobytes()).hexdigest()[:24])


def random_pose(rs, h, w, p_missing):
    pose = np.zeros((18, 3))
    pose[:, 0] = rs.uniform(0, w, 18)
    pose[:, 1] = rs.uniform(0, h, 18)
    pose[:, 2] = 2
    pose[rs.uniform(size=18) < p_missing] = 0
    return pose


def unit_length_and_crops(det, seed):
    """get_unit_length, crop_face, crop_hands, crop_image, crop_around_keypoint of `det` on random poses."""
    rs = np.random.RandomState(seed)
    h, w = int(rs.randint(120, 500)), int(rs.randint(120, 700))
    img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
    out = []
    for p_missing in (0.0, 0.3, 0.7):
        pose = random_pose(rs, h, w, p_missing)
        ul = det.get_unit_length(pose.copy())
        out.append({"unit_length": None if ul is None else float(ul)})
        if ul is None or not np.isfinite(ul) or ul <= 0:
            continue
        out[-1]["crop_face"] = digest(det.crop_face(img, pose.copy(), ul))
        out[-1]["crop_hands"] = digest(det.crop_hands(img, pose.copy(), ul))
        bbox = (int(rs.randint(-50, w)), int(rs.randint(-50, h)), int(rs.randint(10, w + 80)), int(rs.randint(10, h + 80)))
        if bbox[2] > bbox[0] + 2 and bbox[3] > bbox[1] + 2:
            out[-1]["crop_image"] = digest(det.crop_image(img, bbox))
        kp = (float(rs.uniform(0, w)), float(rs.uniform(0, h)))
        half = float(rs.uniform(10, 120))
        out[-1]["crop_around_keypoint"] = digest(det.crop_around_keypoint(img, kp, half))
    return out


def draw_person_pose_cases(draw, seed):
    rs = np.random.RandomState(100 + seed)
    img = rs.randint(0, 256, (240, 320, 3)).astype(np.uint8)
    poses = np.stack([random_pose(rs, 240, 320, 0.25) for _ in range(int(rs.randint(1, 5)))])
    return [digest(draw(img, poses.copy())), digest(draw(img, np.empty((0, 18, 3))))]


def crop_person_cases(det, seed):
    """crop_person on random poses; "raises" where the call raises (degenerate poses)."""
    rs = np.random.RandomState(300 + seed)
    h, w = int(rs.randint(200, 500)), int(rs.randint(200, 700))
    img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
    random_pose(rs, h, w, 0.0)            # the pose of the shipped-reference NameError check; keeps the stream aligned
    out = []
    for p_missing in (0.0, 0.3, 0.6):
        pose = random_pose(rs, h, w, p_missing)
        if not (pose[:, 2] > 0).any():
            continue
        ul = float(rs.uniform(5, 40))
        try:
            out.append(digest(det.crop_person(img, pose.copy(), ul)))
        except Exception:
            out.append("raises")
    return out


def demo_drawing_case(face_mod, hand_mod):
    """draw_face_keypoints, draw_hand_keypoints and crop_face as demo.py calls them, concatenated."""
    img = np.zeros((100, 120, 3), np.uint8)
    face = [[10 + i, 20 + (i % 7), np.float32(0.5)] if i % 5 else None for i in range(70)]
    hand = [[15 + 3 * i, 30 + (i % 4), np.float32(0.5)] if i % 6 else None for i in range(21)]
    pf, _ = face_mod.crop_face(np.arange(100 * 120 * 3, dtype=np.uint8).reshape(100, 120, 3), (30, 20, 40, 50))
    return digest(np.concatenate([face_mod.draw_face_keypoints(img, face, (3, 4)).ravel(),
                                  hand_mod.draw_hand_keypoints(img, hand, (3, 4)).ravel(), pf.ravel()]))


def optimal_size_cases(n=4000, seed=0):
    """(h, w, size) triples: the corners of the 16..2000 range and seeded random draws."""
    rs = np.random.RandomState(seed)
    sizes = np.array([368, 320, 184, 552, 736])
    hw = np.array([(h, w) for h in (16, 17, 1999, 2000) for w in (16, 17, 1999, 2000)] + [(368, 656), (480, 640)])
    corner = np.array([(h, w, s) for h, w in hw for s in sizes])
    rand = np.stack([rs.randint(16, 2001, n), rs.randint(16, 2001, n), sizes[rs.randint(0, len(sizes), n)]], 1)
    return np.concatenate([corner, rand]).astype(np.int64)


def host_helper_goldens():
    """G10: the host-side helpers of pose_detector.py / face_detector.py / hand_detector.py, run verbatim on
    seeded random poses and images: digests of their results (the crops and drawings themselves are large)."""
    ref = reference_loader.load()
    rdet = ref.PoseDetector.__new__(ref.PoseDetector)
    ref.sys = sys                          # crop_person uses `sys` without importing it (pose_detector.py:1-12)
    try:
        out = {"unit_length_and_crops": [unit_length_and_crops(rdet, s) for s in range(12)],
               "draw_person_pose": [draw_person_pose_cases(ref.draw_person_pose, s) for s in range(6)],
               "crop_person": [crop_person_cases(rdet, s) for s in range(8)],
               "demo_face_hand_drawing": demo_drawing_case(reference_loader.load_face(), reference_loader.load_hand())}
    finally:
        ref.__dict__.pop("sys", None)
    with open(os.path.join(GOLD, "host_helpers_ref.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    cases = optimal_size_cases()
    got = np.array([rdet.compute_optimal_size(np.zeros((h, w, 3), np.uint8), s) for h, w, s in cases], np.int64)
    np.savez_compressed(os.path.join(GOLD, "optimal_size_ref.npz"), h_w_size=cases, optimal_size=got)


def precise_padded(ref, he):
    # G7: precise path on a 200x300 frame: the scaled images (184x276, 368x552, 552x828, 736x1104) need
    # right-padding to a multiple of 8 at scales 0.5 and 1.5 -> exercises pad_image / crop (:445,:462,:466)
    detp = ref.PoseDetector("posenet", he, precise=True)
    img = syn.procedural_image(200, 300, seed=4)
    rec = capture_fast(ref, detp, img)
    out = pack(rec)
    out["all_peaks"] = np.asarray(detp.all_peaks, np.float64)
    out["pafs_sample"] = detp.pafs[:, ::5, ::5].astype(np.float32)
    out["heatmaps_sample"] = detp.heatmaps[:, ::5, ::5].astype(np.float32)
    for k in list(out):
        if k.startswith("paf_lo_") or k.startswith("heat_lo_"):
            del out[k]          # keep this fixture small: the low-res maps are already pinned by G5
    np.savez_compressed(os.path.join(GOLD, "precise_200x300_he0.npz"), **out)


if __name__ == "__main__":
    import torch
    torch.set_num_threads(TORCH_THREADS)
    main()
