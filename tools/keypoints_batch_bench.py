"""Face / hand keypoints of one frame: the per-crop loop of demo.py against FaceDetector.detect_batch +
HandDetector.detect_batch (opb_keypoints_detect_batch), on one GPU.

For K = 1, 2, 4, 8, 16 people: K face crops and 2K hand crops (every other one a left hand) of procedural images, with
sizes in the range the crops of a 640x480 frame take (40-160 px a side).  Each timed sample is a host clock around
calls that end in a device synchronise: either the 3K single-crop calls or the two batch calls; the two are
alternated, after a warm-up of every chain size.  Reports the median and the spread per K and precision, and the
end-to-end rate = useful forward FLOP (the crops' own, padding slots excluded) / time.

    python tools/keypoints_batch_bench.py --reps 30 --out profiles/r03_keypoints_batch.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "chainer_realtime_multi-person_pose_estimation_b200"

KS = (1, 2, 4, 8, 16)
BUCKETS = (1, 2, 4, 8, 16, 32)


def _pkg(sub):
    import importlib
    return importlib.import_module(PKG + "." + sub)


def forward_flop(layers, net=368):
    """2 * Cin * Cout * k^2 * H * W summed over the 52 convolutions of FaceNet / HandNet (models/FaceNet.py: conv1_x at
    the input size, conv2_x / conv3_x after one / two 2x2 pools, everything else at net / 8)."""
    total = 0
    for name, cin, cout, k in layers:
        s = {"conv1": 1, "conv2": 2, "conv3": 4}.get(name[:5], 8)
        total += 2 * cin * cout * k * k * (net // s) ** 2
    return total


def chain_bytes(bucket, kp_out, precision, net=368):
    """Device bytes of one cached chain (build_chain_keypoint's allocations, each at least 256 bytes)."""
    h8 = net // 8
    ctot = 1 if precision == "fast" else 2
    acts = [(net, 64), (net // 2, 64), (net // 2, 128), (net // 4, 128), (net // 4, 256), (net // 4, 256), (h8, 256),
            (h8, 512), (h8, 512), (h8, (128 + kp_out + 63) // 64 * 64), (h8, 128), (h8, 128), (h8, 512)]
    sizes = [bucket * net * net * 3, bucket * net * net * 3 * 4, 64 * 4, bucket * kp_out * h8 * h8 * 4]
    sizes += [bucket * s * s * c * ctot * 2 for s, c in acts]
    return int(sum(max(b, 256) for b in sizes))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi failed: " + r.stdout.strip()


def make_crops(k, seed):
    syn = _pkg("synthetic")
    rs = np.random.RandomState(seed)

    def crop(i):
        s = int(rs.randint(40, 161))
        return syn.procedural_image(s, s + int(rs.randint(-2, 3)), seed=seed * 1000 + i)
    faces = [crop(i) for i in range(k)]
    hands = [crop(k + i) for i in range(2 * k)]
    types = ["left" if i % 2 == 0 else "right" for i in range(2 * k)]
    return faces, hands, types


def stats(xs):
    a = np.asarray(xs) * 1e3
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "p10_ms": float(np.percentile(a, 10)),
            "p90_ms": float(np.percentile(a, 90)), "max_ms": float(a.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--precisions", default="comp,parity")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 20:
        raise SystemExit("--reps must be at least 20")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures on a B200 and has no CPU mode")
    syn = _pkg("synthetic")
    FD, HD = _pkg("face_detector").FaceDetector, _pkg("hand_detector").HandDetector
    fm, hm = _pkg("models.FaceNet"), _pkg("models.HandNet")
    face_flop, hand_flop = forward_flop(fm.LAYERS), forward_flop(hm.LAYERS)
    result = {"gpu": gpu_info(), "reps": args.reps,
              "timing": "host clock around calls that end in a device synchronise; loop and batch alternated",
              "forward_gflop_per_crop": {"face": face_flop / 1e9, "hand": hand_flop / 1e9},
              "chain_mib_per_bucket": {}, "runs": []}
    for prec in args.precisions.split(","):
        face_model, hand_model = fm.FaceNet(), hm.HandNet()
        face_model.load_npz(syn.he_weights(0, layers=fm.LAYERS))
        hand_model.load_npz(syn.he_weights(0, layers=hm.LAYERS))
        face, hand = FD(model=face_model, device=0, precision=prec), HD(model=hand_model, device=0, precision=prec)
        result["chain_mib_per_bucket"][prec] = {
            "face": {b: chain_bytes(b, 71, prec) / 2 ** 20 for b in BUCKETS},
            "hand": {b: chain_bytes(b, 22, prec) / 2 ** 20 for b in BUCKETS}}
        frames = {k: make_crops(k, seed=k) for k in KS}

        def loop(k):
            faces, hands, types = frames[k]
            t0 = time.perf_counter()
            out = [face(f) for f in faces] + [hand(h, hand_type=t) for h, t in zip(hands, types)]
            return time.perf_counter() - t0, out

        def batch(k):
            faces, hands, types = frames[k]
            t0 = time.perf_counter()
            out = face.detect_batch(faces) + hand.detect_batch(hands, types)
            return time.perf_counter() - t0, out

        for k in KS:                                   # warm every chain size (and the workspaces) first
            for _ in range(2):
                loop(k)
                batch(k)
        for k in KS:
            t_loop, t_batch = [], []
            launches = []
            for r in range(args.reps):
                order = (loop, batch) if r % 2 == 0 else (batch, loop)
                for fn in order:
                    before = face.engine.launch_count() + hand.engine.launch_count()
                    dt, _ = fn(k)
                    (t_loop if fn is loop else t_batch).append(dt)
                    if r < 2:
                        launches.append((fn is loop, face.engine.launch_count() + hand.engine.launch_count() - before))
            _, out_loop = loop(k)
            _, out_batch = batch(k)
            same = sum(a == b for a, b in zip(out_loop, out_batch))
            flop = k * face_flop + 2 * k * hand_flop
            sl, sb = stats(t_loop), stats(t_batch)
            run = {"precision": prec, "people": k, "face_crops": k, "hand_crops": 2 * k,
                   "loop": sl, "batch": sb, "speedup_median": sl["median_ms"] / sb["median_ms"],
                   "loop_tflops_end_to_end": flop / (sl["median_ms"] * 1e-3) / 1e12,
                   "batch_tflops_end_to_end": flop / (sb["median_ms"] * 1e-3) / 1e12,
                   "kernel_launches": {"loop": [n for lp, n in launches if lp][0],
                                       "batch": [n for lp, n in launches if not lp][0]},
                   "crops_with_identical_keypoints": "%d of %d" % (same, 3 * k)}
            print(json.dumps(run), flush=True)
            result["runs"].append(run)
        del face, hand
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
