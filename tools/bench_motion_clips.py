"""CPTVMotionDetector over whole recordings (cpt_motion_clips, csrc/motion_kernels.cu) against the per-frame loop.

  (1) kernel rate: one cpt_motion_clips call over device-resident frames (synthetic.make_clips_torch), step tables planned
      once and the call repeated; frames/s, and achieved bytes/s against a device-to-device copy measured in the same run
      (bytes per frame from shapes, ``bytes_per_frame``)
  (2) API rate: process_clips from host frame objects, wall clock, and the host planning on its own
  (3) the per-frame process_frame loop on a subset of the same clips
  (4) bench.py's streaming latency (motion_detector p50 / p99) of this tree and of ``--before-tree`` (the parent commit,
      built), alternating the two in child processes

The detectors keep their running sums and background records on the device (154 KB per 160x120 detector) and the frames
stream from HBM: 1024 clips x 900 frames are 35 GB.  Prints one JSON object; ``--out`` also writes it.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, EDGE = 160, 120, 1
NPX, NCROP = W * H, (W - 2 * EDGE) * (H - 2 * EDGE)


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def bytes_per_frame():
    """Device bytes one steady-state step moves (running mean full, background and detection on, one_diff_only):
    the new frame, the frame leaving the ring and the oldest non-FFC frame read (crop only); the uint32 running sum
    read and written; background and weight counters (uint16 each) read and written on the crop."""
    return dict(frame=2 * NPX, oldest=2 * NPX, nonffc=2 * NCROP, sum=2 * 4 * NPX, background=2 * 2 * NCROP, weights=2 * 2 * NCROP)


class Window:
    start = end = types.SimpleNamespace(dt="00:00")

    def use_sunrise_sunset(self):
        return False

    def inside_window(self):
        return True


def make_detector(model):
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import CPTVMotionDetector

    lepton35 = model == 1
    cfg = types.SimpleNamespace(
        motion=types.SimpleNamespace(temp_thresh=28000 if lepton35 else 2750, delta_thresh=150 if lepton35 else 50, count_thresh=3,
                                     frame_compare_gap=45, one_diff_only=True, trigger_frames=2, edge_pixels=EDGE, warmer_only=True),
        recorder=types.SimpleNamespace(use_low_power_mode=False, rec_window=Window(), preview_secs=5, min_secs=5, max_secs=600),
        location=types.SimpleNamespace())
    CPTVMotionDetector.BACKGROUND_WEIGHT_ADD = 0.1
    headers = types.SimpleNamespace(model="lepton3.5" if lepton35 else "lepton3", res_x=W, res_y=H, fps=9)
    return CPTVMotionDetector(cfg, None, headers, detect_after=None)


def frame_objects(pix_clips):
    """Frame objects of each clip (pix: a host array per frame, or None when the frames are staged on the device)."""
    return [[types.SimpleNamespace(pix=None if pix is None else pix[t], time_on=10_000_000 + t * 111, last_ffc_time=0)
             for t in range(n)] for pix, n in pix_clips]


def copy_rate(torch, n_bytes, reps=5):
    src = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    return 2 * n_bytes * reps / (e0.elapsed_time(e1) / 1e3)


def streaming_latency(tree):
    """bench.py's motion_detector leg in a child process, from the source tree ``tree`` and the library built in it."""
    code = "import json, bench; print(json.dumps(bench.bench_motion()))"
    env = {k: v for k, v in os.environ.items() if k != "CPT_LIB"}
    out = subprocess.run([sys.executable, "-c", code], cwd=tree, env=env, capture_output=True, text=True, check=True).stdout
    r = json.loads(out.strip().splitlines()[-1])
    return dict(p50_us=r["p50_us"], p99_us=r["p99_us"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--frames", type=int, default=900)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--api-clips", type=int, default=64)
    ap.add_argument("--loop-clips", type=int, default=4)
    ap.add_argument("--before-tree", default=None, help="a built source tree of the parent commit, for the streaming A/B")
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import plan_clips, process_clips
    from classifier_pipeline_b200.synthetic import make_clips_torch

    assert torch.cuda.is_available(), "needs a CUDA device"
    res = dict(gpu=gpu_identity(), torch_device=torch.cuda.get_device_name(0), width=W, height=H)
    n, T = args.clips, args.frames

    # (1) kernel rate on device-resident frames
    d_clips, models = make_clips_torch(n, T, "cuda")
    torch.cuda.synchronize()
    dets = [make_detector(m) for m in models]
    steps = plan_clips(dets, frame_objects([(None, T)] * n))
    d_frames = d_clips.view(n * T, H, W)
    steps.run(d_frames)  # warm-up: module load, scratch growth
    times = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        steps.run(d_frames)  # returns after the results are on the host
        times.append(time.perf_counter() - t0)
    bpf = bytes_per_frame()
    per_frame = sum(bpf.values())
    best = min(times)
    copy_bps = copy_rate(torch, 4 << 30)
    res["kernel"] = dict(clips=n, frames_per_clip=T, calls_s=times, frames_per_s=n * T / best, bytes_per_frame=bpf,
                         bytes_per_frame_total=per_frame, achieved_bytes_per_s=per_frame * n * T / best,
                         d2d_copy_bytes_per_s=copy_bps, share_of_copy=per_frame * n * T / best / copy_bps,
                         note="host wall clock of the whole call (step table upload, kernel, ring refresh, results back); best of reps")
    del steps, dets

    # (2) API rate from host frame objects, and the planning on its own
    a = args.api_clips
    h_pix = d_clips[:a].view(torch.int16).cpu().numpy().view(np.uint16)
    del d_clips, d_frames
    torch.cuda.empty_cache()
    lists = frame_objects([(h_pix[i], T) for i in range(a)])
    dets = [make_detector(m) for m in models[:a]]
    process_clips(dets[:2], [lst[:50] for lst in lists[:2]])  # warm-up on two throw-away detectors
    dets = [make_detector(m) for m in models[:a]]
    t0 = time.perf_counter()
    process_clips(dets, lists)
    api_s = time.perf_counter() - t0
    dets = [make_detector(m) for m in models[:a]]
    t0 = time.perf_counter()
    plan_clips(dets, lists)
    plan_s = time.perf_counter() - t0
    res["api"] = dict(clips=a, frames_per_clip=T, wall_s=api_s, frames_per_s=a * T / api_s, plan_s=plan_s,
                      plan_frames_per_s=a * T / plan_s)

    # (3) the per-frame loop on a subset
    k = args.loop_clips
    dets = [make_detector(m) for m in models[:k]]
    t0 = time.perf_counter()
    for det, lst in zip(dets, lists[:k]):
        for f in lst:
            det.process_frame(f)
    loop_s = time.perf_counter() - t0
    res["loop"] = dict(clips=k, frames_per_clip=T, wall_s=loop_s, frames_per_s=k * T / loop_s)

    # (4) streaming latency, the two builds alternating
    if args.before_tree:
        ab = dict(before=[], after=[])
        for _ in range(args.ab_rounds):
            ab["before"].append(streaming_latency(os.path.abspath(args.before_tree)))
            ab["after"].append(streaming_latency(ROOT))
        res["streaming_ab"] = ab
    res["gpu_after"] = gpu_identity()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
