"""OpenCV's MOG2 on the host (cv2) and on the device (csrc/mog2_kernels.cu), at the IR camera's 640x480.

  (1) cv2 apply + getBackgroundImage per frame on the host, with all cores and with one (cv2.setNumThreads)
  (2) the device model, one frame per call (T = 1): the kernel's duration (torch.profiler device records), CUDA events
      around each cpt_mog2_apply call (the GPU waits for the host's enqueue in between, so this is the call's latency),
      and the host wall clock of MOG2Background.update_background on a device frame (Python + enqueue + synchronise)
  (3) IRMotionDetector.process_frame from a host BGR frame to the motion flag, with CVBackground and with MOG2Background
      (frames past the detector's 100-frame warm-up, so every timed frame runs the erosion and counts)
  (4) one call over many frames: frames/s and achieved bytes/s against a device-to-device copy measured in the same run
      (bytes: 1 frame byte read + 1 mask byte written per pixel and frame, plus 61 state bytes per pixel read and written once
      per launch of at most 256 frames)

The state of a 640x480 model is 18.7 MB and stays in the B200's 126 MB L2 between per-frame calls; the multi-frame leg
streams 1024 distinct frames (315 MB) so the frames come from HBM.  Prints one JSON object; ``--out`` also writes it.
Needs a CUDA device.
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

W, H = 640, 480
NPX = W * H
STATE_BYTES = 61  # per pixel: 15 floats (weight, variance, mean of five modes) + the mode count


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def summary(xs):
    xs = np.asarray(xs, np.float64)
    return dict(p50=float(np.median(xs)), p99=float(np.percentile(xs, 99)), min=float(xs.min()), max=float(xs.max()), n=int(xs.size))


def scene_frames(n, seed=0):
    """Grey 640x480 frames: a textured scene with sensor noise and a bright block walking through."""
    rng = np.random.default_rng(seed)
    scene = rng.integers(30, 200, (H // 8, W // 8)).repeat(8, 0).repeat(8, 1).astype(np.int16)
    out = np.empty((n, H, W), np.uint8)
    for t in range(n):
        f = scene + rng.integers(-3, 4, (H, W))
        x0 = (t * 13) % (W - 80)
        f[200:280, x0 : x0 + 70] += 80
        out[t] = np.clip(f, 0, 255)
    return out


def host_cv2(frames, threads):
    import cv2

    cv2.setNumThreads(threads)
    m = cv2.createBackgroundSubtractorMOG2(history=1000, detectShadows=False)
    ap, bg = [], []
    for i, f in enumerate(frames):
        t0 = time.perf_counter()
        m.apply(f, None, -1)
        t1 = time.perf_counter()
        m.getBackgroundImage()
        t2 = time.perf_counter()
        if i >= 20:
            ap.append((t1 - t0) * 1e3)
            bg.append((t2 - t1) * 1e3)
    return dict(threads=threads, apply_ms=summary(ap), background_ms=summary(bg))


def device_per_frame(ctx, frames):
    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.track.cliptracker import MOG2Background

    ctx.use_torch_stream()
    d = torch.from_numpy(frames).cuda()
    masks = torch.empty_like(d)
    m = native.Mog2(ctx, W, H, history=1000)
    n = len(frames)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    m.apply(d[:20], -1, d_masks=masks[:20])  # warm-up
    for i in range(n):
        ev[i][0].record()
        m.apply(d[i], [-1.0], d_masks=masks[i], n_frames=1)
        ev[i][1].record()
    torch.cuda.synchronize()
    call_us = [a.elapsed_time(b) * 1e3 for a, b in ev]
    # the kernel alone: torch.profiler's device records of mog2_apply_kernel over the same loop, in a run of its own
    from torch.profiler import ProfilerActivity, profile

    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n):
                m.apply(d[i], [-1.0], d_masks=masks[i], n_frames=1)
            torch.cuda.synchronize()
        kernel_us = [e.time_range.elapsed_us() for e in prof.events() if "mog2_apply_kernel" in e.name]
    except Exception as e:  # the JSON then says "not measured"
        print("profiler:", e, file=sys.stderr)
        kernel_us = []
    bg = MOG2Background()
    bg.update_background(d[0])
    wall = []
    for i in range(n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bg.update_background(d[i])
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e6)
    out = torch.empty((H, W), dtype=torch.uint8, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(100):
        m.background(out)
    e1.record()
    torch.cuda.synchronize()
    state_mb = 2 * STATE_BYTES * NPX / 1e6
    return dict(apply_T1_kernel_us=summary(kernel_us) if kernel_us else "not measured", apply_T1_call_event_us=summary(call_us),
                update_background_wall_us=summary(wall),
                background_image_event_us=e0.elapsed_time(e1) * 10.0, state_traffic_mb_per_frame=state_mb,
                note="state (18.7 MB) is L2-resident between calls")


def detector(frames_bgr, background):
    import torch

    from classifier_pipeline_b200.piclassifier.irmotiondetector import IRMotionDetector
    from tests import ir_helpers

    cfg, headers = ir_helpers.ir_config()
    det = IRMotionDetector(cfg, headers, background=background)
    ms = []
    for i, f in enumerate(frames_bgr):
        t0 = time.perf_counter()
        det.process_frame(f)
        ms.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    return summary(ms[120:])


def multi_frame(ctx, n_frames):
    import torch

    from classifier_pipeline_b200 import native

    ctx.use_torch_stream()
    rng = np.random.default_rng(3)
    base = torch.from_numpy(scene_frames(64, seed=4)).cuda()
    d = base.repeat(n_frames // 64, 1, 1).contiguous()
    d += torch.from_numpy(rng.integers(0, 3, (n_frames, 1, 1), dtype=np.uint8)).cuda()  # distinct frames
    masks = torch.empty_like(d)
    m = native.Mog2(ctx, W, H, history=1000)
    m.apply(d, -1, d_masks=masks)  # warm-up (and a model with several modes per pixel)
    times = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.apply(d, -1, d_masks=masks)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    launches = -(-n_frames // 256)
    nbytes = NPX * (2 * n_frames + 2 * STATE_BYTES * launches)
    t = float(np.median(times)) * 1e-3
    # HBM reference: a device-to-device copy of 4 GiB (read + write), the median of 5
    a = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    cp = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        cp.append(e0.elapsed_time(e1))
    peak = 2 * a.numel() / (float(np.median(cp)) * 1e-3)
    del a, b
    return dict(frames=n_frames, launches=launches, ms=summary(times), frames_per_s=n_frames / t, us_per_frame=t / n_frames * 1e6,
                bytes=nbytes, achieved_gb_s=nbytes / t / 1e9, copy_peak_gb_s=peak / 1e9, share_of_copy_peak=nbytes / t / peak)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=300, help="frames per host / per-frame leg")
    ap.add_argument("--multi", type=int, default=1024, help="frames of the multi-frame call")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    assert torch.cuda.is_available(), "bench_mog2 measures the device: it needs a CUDA device"
    from classifier_pipeline_b200 import engine
    from classifier_pipeline_b200.track.cliptracker import CVBackground, MOG2Background
    from tests import ir_helpers

    ctx = engine.get_engine().ctx
    frames = scene_frames(args.frames)
    res = dict(gpu=gpu_identity(), host_cpus=os.cpu_count(), width=W, height=H)
    import cv2

    res["cv2_version"] = cv2.__version__
    res["host_cv2_all_cores"] = host_cv2(frames, os.cpu_count())
    res["host_cv2_one_core"] = host_cv2(frames, 1)
    cv2.setNumThreads(os.cpu_count())
    res["device_per_frame"] = device_per_frame(ctx, frames)
    bgr = ir_helpers.ir_video(3, frames=args.frames)
    res["detector_cv_background_ms"] = detector(bgr, CVBackground())
    res["detector_mog2_background_ms"] = detector(bgr, MOG2Background())
    res["detector_cv_background_ms_repeat"] = detector(bgr, CVBackground())
    res["detector_mog2_background_ms_repeat"] = detector(bgr, MOG2Background())
    res["multi_frame"] = multi_frame(ctx, args.multi)
    res["gpu_after"] = gpu_identity()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
