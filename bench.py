#!/usr/bin/env python
"""bench.py -- frames/sec of the OpenPose inference hot path at 368x656, batch 32 per GPU.

    python bench.py --gpus N --steps K --warmup W            (ours; N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic input (BASELINE.json
configs[2]: "full pipeline (conv + NMS + PAF integral + grouping) synthetic 8-person 368x656
batch 32"): the 92-conv CocoPoseNet chain runs on 32 random uint8 BGR frames per GPU; because
random weights cannot produce people, the synthetic 8-person low-resolution maps are injected
as the network output in front of upsample -> peaks -> PAF integrals -> assignment -> grouping
(SURVEY.md 8d).  N GPUs: images shard by rank (weak scaling), one NCCL all-gather of the
fixed-size person records per step.

`value` = whole-job frames/s with the input batch already resident in HBM; `e2e` = the same
through the host-buffer entry (pinned uint8 frames H2D and the result records D2H inside the
timed region).  `roofline` is for the dominant kernel, the grouped 7x7 128->128 conv launch.
`--impl reference` times the CPU restatement of the reference path (oracle/, torch-CPU conv +
NumPy/SciPy post-process; Chainer itself is not installable offline) on the host cores.

`--dump-outputs DIR` writes what the timed path returned in its last step (the person records of one batch; poses and
scores with --impl reference) as DIR/<name>.npy in float64.  Inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "chainer_realtime_multi-person_pose_estimation_b200"
H, W, MAP_H, MAP_W = 368, 656, 320, 576
FLOPS_PER_IMAGE = 484634285056            # SURVEY.md 8d, true channel counts
METRIC = "frames/sec at 368x656 batch32 (full pipeline: conv + NMS + PAF integral + grouping)"


DTYPES = {"fast": "f16 (fp32 accumulate)", "parity": "split-f16 (hi+lo, 3 MMAs, two-level fp32 accumulation)",
          "comp": "f16 + f8 rounding corrections (2 MMAs, fp32 accumulate, two-level on the 7x7 layers)"}
MAP_ERR = {"fast": "2.8e-3 (outside north_star's 1e-3: reported for the fp16 roofline config only)",
           "parity": "1.9e-5", "comp": "1.6e-4 .. 5.3e-4 on the three fast goldens (profiles/r02_precision_ladder.txt)"}


def pkg(sub=None):
    return importlib.import_module(PKG + ("." + sub if sub else ""))


def traffic_from_profile(precision):
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, read from the committed
    ncu summary of this precision (profiles/r02_ncu_<precision>_swap7x7_summary.txt); None when there is none."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_%s_swap7x7_summary.txt" % precision)
    if not os.path.isfile(path):
        return None, "no committed ncu --set full summary for this precision (%s)" % os.path.basename(path)
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, seen = 0.0, 0
    for ln in open(path):
        f = ln.split()
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[2] in mult:
            tot += float(f[1].replace(",", "")) * mult[f[2]]
            seen += 1
    if seen != 2:
        return None, "dram__bytes_read/write not found in " + os.path.basename(path)
    return tot, "ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch, profiles/" + os.path.basename(path)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured")
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source="fallback")


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.th = index, [], False, None

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True, timeout=5)
                self.samples.append([s.strip() for s in out.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if len(s) >= 6 and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 6 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) >= 6 and s[2 + i] == "Active" for s in self.samples)]
        def num(i):
            out = []
            for smp in self.samples:
                try:
                    out.append(float(smp[i]))
                except (IndexError, ValueError):
                    pass
            return out
        pw, pl = num(6), num(7)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm),
                    power_w=float(np.median(pw)) if pw else None, power_limit_w=max(pl) if pl else None,
                    power_note="nvidia-smi power.draw is a ~1 s running average: a timed region of a few hundred ms reads low "
                               "while the throttle reason already reports the instantaneous cap")


def cpu_reference_step(weights, img, paf_lo, heat_lo):
    """One frame through the CPU restatement of the reference path."""
    from oracle import restate as R
    x = R.preprocess(img)
    R.forward(weights, x)                                                   # conv chain (torch CPU fp32)
    pafs = R.resize_bilinear_align_corners(paf_lo[None], (MAP_H, MAP_W))[0]   # injected maps, as in our arm
    heat = R.resize_bilinear_align_corners(heat_lo[None], (MAP_H, MAP_W))[0]
    return R.postprocess_fast(pafs, heat, MAP_W, W, H, MAP_H)


def pick_cpu_threads(weights, frame, paf_lo, heat_lo, budget_s=30.0):
    """oneDNN does not scale to every logical core of a big host (128 threads: 30 s/frame, 16 threads: <1 s):
    try a few thread counts (1 warm-up + 1 timed frame each) within `budget_s` and keep the fastest."""
    import torch
    best, t_start = None, time.perf_counter()
    for nt in sorted({min(os.cpu_count(), t) for t in (16, 32, 64, os.cpu_count())}):
        torch.set_num_threads(nt)
        cpu_reference_step(weights, frame, paf_lo, heat_lo)
        t0 = time.perf_counter()
        cpu_reference_step(weights, frame, paf_lo, heat_lo)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
        if time.perf_counter() - t_start > budget_s:
            break
    torch.set_num_threads(best[1])
    return best


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    syn = pkg("synthetic")
    wd = syn.he_weights(0)
    weights = {k[:-2]: (wd[k], wd[k[:-2] + "/b"]) for k in wd if k.endswith("/W")}
    imgs = syn.random_images(2, H, W, seed=0)
    paf_lo, heat_lo = syn.eight_person_lowres(H // 8, W // 8, seed=0)
    _, cores = pick_cpu_threads(weights, imgs[0], paf_lo, heat_lo)      # threads actually used
    for i in range(max(args.warmup, 1)):
        cpu_reference_step(weights, imgs[i % 2], paf_lo, heat_lo)
    t0 = time.perf_counter()
    for i in range(args.steps):
        poses, scores = cpu_reference_step(weights, imgs[i % 2], paf_lo, heat_lo)
    dt = time.perf_counter() - t0
    assert len(scores) == 8
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "poses.npy"), np.asarray(poses, np.float64))
        np.save(os.path.join(args.dump_outputs, "scores.npy"), np.asarray(scores, np.float64))
    value = args.steps / dt
    sample = ("1 frame per step (the reference is batch-1), %d steps, %d torch threads (fastest of 16/32/64/all on a "
              "%d-core host)" % (args.steps, cores, os.cpu_count()))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[2]: full pipeline, synthetic 8-person maps injected, 368x656, "
                               "batch %d per GPU" % args.batch,
                   "impl_note": "CPU oracle port of the reference path (pose_detector.py restated in oracle/restate.py; "
                                "torch-CPU fp32 conv; Chainer is not installable offline); the reference is batch-1, so a "
                                "step is one frame of that workload",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def dump_records(out_dir, hdr, per):
    """The person records of one batch as float64 .npy files: per-image header fields, and per-person fields with the
    slots past each image's n_persons zeroed (the device leaves them unwritten)."""
    os.makedirs(out_dir, exist_ok=True)
    used = np.arange(per.shape[1])[None, :] < hdr["n_persons"][:, None]
    arrays = {"n_peaks": hdr["n_peaks"], "n_persons": hdr["n_persons"], "status": hdr["status"],
              "n_connections": hdr["n_connections"]}
    for f in ("score", "count", "peak_id", "x", "y"):
        v = per[f].astype(np.float64)
        arrays["person_" + f] = np.where(used.reshape(used.shape + (1,) * (v.ndim - 2)), v, 0.0)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    native, syn, mg = pkg("_native"), pkg("synthetic"), pkg("multi_gpu")
    B = args.batch
    model = pkg("models.CocoPoseNet").CocoPoseNet()
    model.load_npz(syn.he_weights(0))
    prm = pkg("pose_detector").make_opb_params(max_peaks=2048, max_candidates=8192, max_persons=args.max_persons)
    eng = native.Engine(local_rank, prm, {"fast": native.PRECISION_FAST, "parity": native.PRECISION_PARITY,
                                          "comp": native.PRECISION_COMP}[args.precision])
    eng.load_model(model)
    # a dedicated (non-default) torch stream: libopb launches on it, torch events time it
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)

    imgs_host = torch.from_numpy(syn.random_images(B, H, W, seed=rank)).pin_memory()
    imgs_dev = imgs_host.cuda()
    imgs_host2 = [imgs_host, imgs_host.clone().pin_memory()]      # one pinned source per streaming slot
    imgs_dev2 = [imgs_dev, imgs_dev.clone()]
    paf_lo, heat_lo = syn.eight_person_lowres(H // 8, W // 8, seed=0)
    d_paf = torch.from_numpy(np.repeat(paf_lo[None], B, 0)).cuda()
    d_heat = torch.from_numpy(np.repeat(heat_lo[None], B, 0)).cuda()
    hdr_dev = torch.zeros(B * native.HEADER_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    per_dev = torch.zeros(B * args.max_persons * native.PERSON_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    # N > 1: the ONE collective of the path is opb_allgather_results -- an ncclAllGather of the slot's device-resident
    # record block [B headers | B x max_persons persons] on the slot's stream, straight behind its pipeline (no host hop).
    # The library's own communicator: rank 0 creates the NCCL id, torch.distributed ships it.
    rec_bytes = eng.record_block_bytes(B)
    gathered = [torch.zeros(world * rec_bytes, dtype=torch.uint8, device="cuda") for _ in range(2)]
    if world > 1:
        uid = torch.from_numpy(eng.nccl_unique_id() if rank == 0 else np.zeros(128, np.uint8)).cuda()
        dist.broadcast(uid, 0)
        eng.nccl_comm_init(world, rank, uid.cpu().numpy())
    hdr_host = np.empty(B, native.HEADER_DTYPE)
    per_host = np.empty((B, args.max_persons), native.PERSON_DTYPE)
    import ctypes as C

    def step_resident_sync():
        eng._check(eng.lib.opb_detect_batch(eng.ctx, C.c_void_p(imgs_dev.data_ptr()), native.OPB_DEVICE, B, H, W,
                                            MAP_H, MAP_W, float(MAP_W), C.c_void_p(d_paf.data_ptr()),
                                            C.c_void_p(d_heat.data_ptr()), C.c_void_p(hdr_dev.data_ptr()),
                                            C.c_void_p(per_dev.data_ptr()), native.OPB_DEVICE))

    # `value`: frames resident in HBM, the same two-slot streaming entry as `e2e` but with device frames (no upload):
    # slot 1 runs on its own stream, so the tails and launch gaps of one batch's kernels are filled by the other's.
    # One batch is in flight when the timed region starts and the region ends with opb_stream_join, so K steps contain
    # K complete pipeline passes, K record downloads and (N > 1) K all-gathers.
    res_state = {"slot": 0, "hdr": None, "per": None}

    def res_submit():
        sl = res_state["slot"]
        eng.stream_submit((imgs_dev2[sl].data_ptr(), B, H, W), H, W, MAP_H, MAP_W, sl,
                          img_len=MAP_W, inject_paf=d_paf.data_ptr(), inject_heat=d_heat.data_ptr(), device=True)
        if world > 1:
            eng.allgather_results(sl, gathered[sl].data_ptr())     # ONE NCCL all-gather per step, device to device
        res_state["slot"] ^= 1

    def step_resident():
        res_submit()
        # the batch submitted one step earlier (and its all-gather)
        res_state["hdr"], res_state["per"] = eng.stream_collect(res_state["slot"])

    def step_e2e_sync():
        eng._check(eng.lib.opb_detect_batch(eng.ctx, C.c_void_p(imgs_host.data_ptr()), native.OPB_HOST, B, H, W,
                                            MAP_H, MAP_W, float(MAP_W), C.c_void_p(d_paf.data_ptr()),
                                            C.c_void_p(d_heat.data_ptr()), C.c_void_p(hdr_host.ctypes.data),
                                            C.c_void_p(per_host.ctypes.data), native.OPB_HOST))

    # streaming entry (opb_stream_submit / opb_stream_collect): every step uploads one batch from pinned host
    # memory on the copy stream, runs the pipeline and reads its records back; the upload of batch i+1 overlaps
    # the kernels of batch i.  One batch is in flight when the timed region starts and one when it ends, so K
    # steps contain exactly K uploads, K pipeline passes and K result downloads.
    e2e_state = {"slot": 0, "hdr": None}

    def e2e_submit():
        sl = e2e_state["slot"]
        eng.stream_submit((imgs_host2[sl].data_ptr(), B, H, W), H, W, MAP_H, MAP_W, sl,
                          img_len=MAP_W, inject_paf=d_paf.data_ptr(), inject_heat=d_heat.data_ptr())
        if world > 1:
            eng.allgather_results(sl, gathered[sl].data_ptr())     # the collective is inside the end-to-end step too
        e2e_state["slot"] ^= 1

    def step_e2e():
        e2e_submit()                                               # batch i+1 goes up ...
        e2e_state["hdr"], _ = eng.stream_collect(e2e_state["slot"])   # ... while batch i finishes; read its records

    def timed(fn, steps, warmup, prime=None):
        # `prime` puts the first batch in flight before the warm-up, so that with any --warmup (0 included) the timed
        # region holds exactly `steps` submits
        if prime is not None:
            prime()
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count()
        e0.record(stream)
        for _ in range(steps):
            fn()
        eng.stream_join()                  # streaming slot 1 runs on its own stream: e1 must cover it
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        per_rank = [float(ms.item())]
        if world > 1:
            allms = torch.zeros(world, device="cuda")
            dist.all_gather_into_tensor(allms, ms)
            per_rank = [float(v) for v in allms.cpu()]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        timed.per_rank_ms = per_rank
        return float(ms.item()), eng.launch_count() - l0

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total, launches = timed(step_resident, args.steps, args.warmup, prime=res_submit)
    per_rank_ms = [m / args.steps for m in timed.per_rank_ms]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        if world > 1:   # the caller's view at N > 1: every rank's records, all-gathered with the last collected batch
            g = gathered[res_state["slot"]].cpu().numpy().reshape(world, rec_bytes)
            hb = B * native.HEADER_DTYPE.itemsize
            hdr = np.concatenate([np.frombuffer(g[r, :hb].tobytes(), native.HEADER_DTYPE) for r in range(world)])
            per = np.concatenate([np.frombuffer(g[r, hb:].tobytes(), native.PERSON_DTYPE).reshape(B, -1) for r in range(world)])
        else:
            hdr, per = res_state["hdr"], res_state["per"]
        dump_records(args.dump_outputs, hdr, per)
    # correctness of the timed path: 8 persons per frame (last collected batch and the one still in flight)
    hdr_last, _ = eng.stream_collect(res_state["slot"] ^ 1)
    for hdr in (res_state["hdr"], hdr_last):
        assert (hdr["status"] == 0).all() and (hdr["n_persons"] == 8).all(), hdr
    ms_sync, _ = timed(step_resident_sync, args.steps, args.warmup)
    if world > 1:   # every rank holds every rank's records after the all-gather (both slots' buffers)
        for gbuf in gathered:
            g = gbuf.cpu().numpy().reshape(world, -1)
            for r in range(world):
                gh = np.frombuffer(g[r, :hdr_dev.numel()].tobytes(), native.HEADER_DTYPE)
                assert (gh["status"] == 0).all() and (gh["n_persons"] == 8).all(), (r, gh)
    ms_e2e, _ = timed(step_e2e, args.steps, args.warmup, prime=e2e_submit)
    hdr_last, _ = eng.stream_collect(e2e_state["slot"] ^ 1)         # drain the batch still in flight
    for hh in (e2e_state["hdr"], hdr_last):
        assert (hh["status"] == 0).all() and (hh["n_persons"] == 8).all()
    ms_e2e_sync, _ = timed(step_e2e_sync, args.steps, args.warmup)
    assert (hdr_host["status"] == 0).all() and (hdr_host["n_persons"] == 8).all()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    value = world * B * args.steps / (ms_total * 1e-3)
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
    # dominant kernel: the grouped 7x7 128->128 launch (both branches), 20 launches per step
    n77 = 20
    if args.no_stage_timing:
        print(json.dumps({"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "gpu_launches": launches,
                          "e2e": {"value": e2e_value, "unit": "frames/s"}, "note": "stage timing skipped"}))
        return
    ms77 = eng.time_stage("Mconv7x7", reps=5) / n77
    flops77 = 2 * (2.0 * B * (H // 8) * (W // 8) * 128 * 128 * 49)
    ach = flops77 / (ms77 * 1e-3) / 1e12
    ms_chain = eng.time_stage("conv_chain", reps=3)
    # PAF HBM figures (SURVEY 8d).  The default pipeline no longer materialises the full-resolution PAFs (the line
    # integrals sample the network-resolution maps on demand, OPB_PAF_LOWRES=1), so the HBM-bound kernel of the
    # reference's data flow (F.resize_images, pose_detector.py:501) is timed on its own here, and then together with the
    # line-integral stage over the materialised maps, each against its own algorithmic bytes.
    ms_up = eng.time_stage("upsample_paf", reps=10)
    up_bytes = B * (38 * (H // 8) * (W // 8) * 4 + 38 * MAP_H * MAP_W * 4)          # low-res read + full-res write
    stage_ms = {s_: eng.time_stage(s_, reps=5) for s_ in ("upsample_heat", "peaks", "paf_integral", "group")}
    n_pairs = 1193                                                                 # candidate pairs per synthetic 8-person frame (SURVEY App. B-3)
    both_bytes = up_bytes + 80 * n_pairs * B
    extra = {
        "conv_chain_ms": ms_chain,
        "conv_chain_tflops": B * FLOPS_PER_IMAGE / (ms_chain * 1e-3) / 1e12,
        "conv_chain_frac_of_sustained_peak": B * FLOPS_PER_IMAGE / (ms_chain * 1e-3) / 1e12 / (peaks["tflops_sustained"] or peaks["tflops"]),
        "paf_upsample_materialise": {"bound": "hbm", "kernel": "upsample_bilinear_ac_v4_kernel (38 PAF planes per image)",
                                     "bytes": up_bytes, "achieved": up_bytes / (ms_up * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                                     "unit": "GB/s", "frac": up_bytes / (ms_up * 1e-3) / 1e9 / peaks["hbm_gbs"], "ms": ms_up,
                                     "note": "the upsample launch alone; not part of the default pipeline any more"},
        "paf_upsample_plus_line_integral": {"bound": "hbm", "bytes": both_bytes, "ms": ms_up + stage_ms["paf_integral"],
                                            "achieved": both_bytes / ((ms_up + stage_ms["paf_integral"]) * 1e-3) / 1e9,
                                            "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                            "frac": both_bytes / ((ms_up + stage_ms["paf_integral"]) * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                            "note": "upsample launch + the paf_integral stage (paf_candidates + limb_assign, as the default "
                                                    "pipeline runs them) over upsample bytes + 80 B per candidate pair"},
        "stage_ms": stage_ms,
    }
    # camera-style latency: one 640x480 BGR frame through the public PoseDetector.__call__ (host resize,
    # H2D, conv chain, post-process, D2H), the loop of camera_pose_demo.py:20-31
    try:
        det = pkg("pose_detector").PoseDetector(model=model, device=local_rank, precision=args.precision)
        frame = syn.procedural_image(480, 640, seed=2)
        for _ in range(3):
            det(frame)
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            det(frame)
            ts.append(time.perf_counter() - t0)
        extra["single_frame_640x480_ms"] = {"median": 1e3 * float(np.median(ts)), "min": 1e3 * float(np.min(ts)),
                                            "note": "wall clock of PoseDetector.__call__ (random-weight noise maps: "
                                                    "~2000 peaks, so the post-process is far heavier than on real frames)"}
        del det
    except Exception as e:  # the headline numbers must not depend on this extra
        extra["single_frame_640x480_ms"] = {"error": str(e)[:200]}
    # SURVEY 8f#2: one FaceNet / HandNet crop through FaceDetector / HandDetector.__call__ (demo.py:33-55), and the
    # CPU restatement of the same call (torch-CPU conv + SciPy) once, for scale
    try:
        kp = {}
        for kind, modname, cls, netmod in (("face", "face_detector", "FaceDetector", "models.FaceNet"),
                                           ("hand", "hand_detector", "HandDetector", "models.HandNet")):
            nm = pkg(netmod)
            net = getattr(nm, "FaceNet" if kind == "face" else "HandNet")()
            wd = syn.he_weights(0, layers=nm.LAYERS)
            net.load_npz(wd)
            d = getattr(pkg(modname), cls)(model=net, device=local_rank, precision=args.precision)
            crop = syn.procedural_image(200, 200, seed=21)
            for _ in range(3):
                d(crop)
            ts = []
            for _ in range(20):
                t0 = time.perf_counter()
                d(crop)
                ts.append(time.perf_counter() - t0)
            kp[kind + "_200x200_crop_ms"] = 1e3 * float(np.median(ts))
            if not args.no_cpu_baseline and kind == "face" and world == 1:
                from oracle import restate as R
                import torch as _t
                _t.set_num_threads(16)
                weights = {n: (wd[n + "/W"], wd[n + "/b"]) for n, _, _, _ in nm.LAYERS}
                R.detect_keypoints(weights, crop)
                t0 = time.perf_counter()
                R.detect_keypoints(weights, crop)
                kp["face_200x200_crop_cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
            del d
        extra["keypoint_nets"] = kp
    except Exception as e:
        extra["keypoint_nets"] = {"error": str(e)[:200]}
    # SURVEY.md 8d: the PAF gather alone under a dense-candidate load -- 64 peaks of every joint type per frame (an 8 x 8
    # grid of impulses in each low-resolution heat map) => 64 x 64 x 19 = 77 824 candidate pairs per frame, 80 B of
    # 4-byte gathers each.  Times paf_candidates + limb_assign on the full-resolution PAFs of that batch.
    try:
        hl = np.zeros((19, H // 8, W // 8), np.float32)
        for c in range(18):
            for i in range(8):
                for j in range(8):
                    hl[c, 2 + 5 * i + (c % 3), 3 + 9 * j + (c % 5)] = 1.0
        pl = (np.random.RandomState(1).standard_normal((38, H // 8, W // 8)) * 0.02).astype(np.float32)   # below the 0.05 threshold: every pair is scored, none accepted
        d_p2 = torch.from_numpy(np.repeat(pl[None], B, 0)).cuda()
        d_h2 = torch.from_numpy(np.repeat(hl[None], B, 0)).cuda()
        eng._check(eng.lib.opb_detect_batch(eng.ctx, C.c_void_p(imgs_dev.data_ptr()), native.OPB_DEVICE, B, H, W, MAP_H, MAP_W,
                                            float(MAP_W), C.c_void_p(d_p2.data_ptr()), C.c_void_p(d_h2.data_ptr()),
                                            C.c_void_p(hdr_host.ctypes.data), C.c_void_p(per_host.ctypes.data), native.OPB_HOST))
        pk = eng.image_detail(0)[0]
        per_type = np.bincount(pk[:, 0].astype(int), minlength=18)
        limbs = pkg("entity").params["limbs_point"]
        pairs = int(sum(int(per_type[int(a)]) * int(per_type[int(b)]) for a, b in limbs))
        ms_dense = eng.time_stage("paf_integral", reps=10)
        extra["paf_gather_dense"] = {"peaks_per_frame": int(len(pk)), "pairs_per_frame": pairs, "ms": ms_dense,
                                     "gather_bytes": 80 * pairs * B,
                                     "achieved_gbs": 80.0 * pairs * B / (ms_dense * 1e-3) / 1e9,
                                     "note": "paf_candidates + limb_assign; 4-byte gathers use 1/8 of each 32 B sector, "
                                             "so sector traffic is ~8x the algorithmic bytes (latency-bound, not an HBM roofline)"}
    except Exception as e:
        extra["paf_gather_dense"] = {"error": str(e)[:200]}
    # The other precisions on the same workload, each in a child process so that nothing they do can cost the headline line:
    # "fast" = plain fp16, the precision BASELINE.json configs[1] names for the conv roofline (map error 2.8e-3: outside the
    # 1e-3 tolerance, so it is an extra, not the headline); "parity" = split fp16, the most accurate (1.9e-5).
    if world == 1 and not args.no_parity_extra:
        for other in [p for p in ("fast", "parity") if p != args.precision]:
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--precision", other, "--steps", "5", "--warmup", "3",
                                    "--no-cpu-baseline", "--no-parity-extra", "--batch", str(B), "--max-persons", str(args.max_persons)],
                                   stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=240)
                line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                d = json.loads(line[-1]) if line else None
                extra[other + "_precision"] = ({"value": d["value"], "unit": "frames/s", "ms_per_step": d["ms_per_step"],
                                                "e2e": d["e2e"]["value"], "dtype": d["dtype"], "map_error_vs_reference": MAP_ERR[other],
                                                "roofline": {k: d["roofline"][k] for k in ("achieved", "peak", "frac", "ms_per_launch", "kernel")},
                                                "conv_chain_ms": d["extra"].get("conv_chain_ms"),
                                                "conv_chain_tflops": d["extra"].get("conv_chain_tflops"),
                                                "note": "child process, 5 steps after 3 warm-ups"}
                                               if d else {"error": (r.stderr or "no output")[-200:]})
            except Exception as e:
                extra[other + "_precision"] = {"error": str(e)[:200]}
    # CPU baseline: the oracle port on this box's host cores, bounded sample
    cpu = None
    if not args.no_cpu_baseline and world == 1:            # rank 0 at N = 1 only
        wd = syn.he_weights(0)
        weights = {k[:-2]: (wd[k], wd[k[:-2] + "/b"]) for k in wd if k.endswith("/W")}
        fr = imgs_host[0].numpy()
        best = pick_cpu_threads(weights, fr, paf_lo, heat_lo)
        cpu = {"value": 1.0 / best[0], "unit": "frames/s", "cores": best[1], "kind": "port",
               "sample": "1 timed frame after 1 warm-up per thread setting (reference is batch-1), best of the "
                         "settings tried within 30 s; host has %d logical cores; torch-CPU fp32 conv + NumPy/SciPy "
                         "post-process" % os.cpu_count()}
    traffic, traffic_note = traffic_from_profile(args.precision)
    mma_per_kstep = {"fast": 1, "parity": 3, "comp": 2}[args.precision]
    roofline = {"bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                "traffic": traffic, "traffic_note": traffic_note,
                "kernel": "grouped L1+L2 7x7 128->128 launch (Mconv2..5 of stages 2-6), 20 launches/step: "
                          + {"fast": "conv_tcgen05_swap7_kernel<COMP=0,DRAIN=0>",
                             "comp": "conv_tcgen05_swap7_kernel<COMP=1,DRAIN=1> (kind::f16 + kind::f8f6f4, two-level accumulation)",
                             "parity": "conv_tcgen05_kernel<7,128,1,3,6,2,DRAIN> (split fp16: 3 kind::f16 MMAs per k-step)"}[args.precision],
                "issued_tensor_work": {"mma_per_kstep": mma_per_kstep, "fp16_equivalent_tflops": ach * (2.0 if args.precision == "comp" else 3.0 if args.precision == "parity" else 1.0),
                                       "note": "tensor-pipe time actually issued, in units of fp16 MMA work (an 8-bit-float K=32 MMA occupies the pipe as long as an fp16 K=16 MMA); "
                                               "ncu tensor-pipe-active of the isolated launch: profiles/r02_ncu_%s_swap7x7_summary.txt" % args.precision},
                "flops_per_launch": flops77, "ms_per_launch": ms77,
                "note": "achieved = ALGORITHMIC flops (2*Cin*Cout*49 per pixel, true channels) / CUDA-event time; this precision "
                        "issues %d MMA(s) per k-step (8-bit-float correction MMAs run at twice the fp16 rate), so the tensor pipe is "
                        "busy for %.2f of the launch at the measured fp16 peak" % (
                            mma_per_kstep, (1.0 if args.precision != "comp" else 2.0) * (1 if args.precision != "parity" else 3) * ach / peaks["tflops"])}
    out = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPES[args.precision], "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[2]: full pipeline, synthetic 8-person maps injected, 368x656, "
                               "batch %d per GPU" % B,
                   "precision": args.precision, "map_error_vs_reference": MAP_ERR[args.precision], "global_batch": world * B,
                   "per_rank_ms_per_step": per_rank_ms,
                   "parallelism": "image-sharded x%d, 1 ncclAllGather of the device-resident person records per step "
                                  "(opb_allgather_results, inside the timed region of value and e2e)" % world,
                   "l2": "no explicit flush: activations written/read per step (~4.5 GB) exceed the 126 MB L2",
                   "peaks": peaks["source"]},
        "gpu_launches": launches,
        "value_api": {"api": "opb_stream_submit/opb_stream_collect with device-resident frames (two slots on two streams)",
                      "sync_api": {"value": world * B * args.steps / (ms_sync * 1e-3), "ms_per_step": ms_sync / args.steps,
                                   "api": "opb_detect_batch, device frames, one batch at a time"}},
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(imgs_host.numel()),
                "d2h_bytes_per_step": int(hdr_host.nbytes + per_host.nbytes), "ms_per_step": ms_e2e / args.steps,
                "api": "opb_stream_submit/opb_stream_collect, host frames (two slots on two streams: upload and kernels of "
                       "batch i+1 overlap batch i)",
                "sync_api": {"value": world * B * args.steps / (ms_e2e_sync * 1e-3), "ms_per_step": ms_e2e_sync / args.steps,
                             "api": "opb_detect_batch with host buffers (upload, kernels, download serialised)"}},
        "roofline": roofline,
        "cpu_baseline": cpu, "clocks": clocks, "extra": extra,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--precision", default="comp", choices=["fast", "parity", "comp"],
                    help="comp (default): the fastest precision inside the 1e-3 map tolerance; fast: fp16 (roofline config); parity: split fp16")
    ap.add_argument("--max-persons", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stage-timing", action="store_true", help="skip the per-stage re-launches (clean ncu launch lists)")
    ap.add_argument("--no-parity-extra", action="store_true", help="skip the other-precision throughput extras (child processes)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the person records the timed path returned in its last step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
