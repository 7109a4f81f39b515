"""IRMotionDetector over whole recordings (cpt_ir_motion_clips, csrc/ir_kernels.cu) against the per-frame loop.

  (0) agreement first: the device-input call, the host-input call and the process_frame loop give the same trace on every
      frame of the same clips
  (1) device-resident BGR frames: process_clips for 1, 8 and 32 clips x 600 frames at 640x480; frames/s of the native call
      (host wall clock to its final synchronise) and of the whole process_clips, and achieved bytes/s (bytes per
      clip-frame from shapes, ``bytes_per_frame``) against a device-to-device copy measured in the same run
  (2) host BGR frames: process_clips, wall clock (the call synchronises before it returns)
  (3) the per-frame process_frame loop with MOG2Background on a subset
  (4) IRMotionDetector.process_frame latency p50 / p99 of this tree and of ``--before-tree`` (the parent commit, built),
      alternating the two in child processes

Every detector has MOG2Background(history=1000) and a ring of 10 frames.  Prints one JSON object; ``--out`` also writes it.
Needs a CUDA device.
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

W, H = 640, 480
NPX, WPR = W * H, (W + 31) // 32


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def bytes_per_frame():
    """Device bytes one detecting step moves: the BGR frame read; the MOG2 state (5 modes x weight / var / mean fp32 and the
    mode count) read and written; the grey ring's new byte written and oldest byte read; the mask byte written; the two bit
    planes written and read."""
    return dict(bgr=3 * NPX, state=2 * 61 * NPX, ring=2 * NPX, mask=NPX, bits=2 * 2 * H * WPR * 4)


class Window:
    start = end = types.SimpleNamespace(dt="00:00")

    def use_sunrise_sunset(self):
        return False

    def inside_window(self):
        return True


def make_detector():
    from classifier_pipeline_b200.piclassifier.irmotiondetector import IRMotionDetector
    from classifier_pipeline_b200.track.cliptracker import MOG2Background

    cfg = types.SimpleNamespace(recorder=types.SimpleNamespace(use_low_power_mode=False, rec_window=Window(), preview_secs=1, min_secs=5,
                                                               max_secs=600), location=types.SimpleNamespace())
    headers = types.SimpleNamespace(model="IR", res_x=W, res_y=H, fps=10)
    return IRMotionDetector(cfg, headers, background=MOG2Background())


def make_clip(torch, seed, T):
    """uint8 BGR [T][H][W][3] on the device: a textured scene with noise of +-3 and a 120 x 80 box walking through from frame
    150 to 400 (so every clip records for a while)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    scene = torch.randint(30, 120, (H // 8, W // 8, 3), generator=g, device="cuda", dtype=torch.int16)
    scene = scene.repeat_interleave(8, 0).repeat_interleave(8, 1)
    out = torch.empty((T, H, W, 3), dtype=torch.uint8, device="cuda")
    for t in range(T):
        f = scene + torch.randint(-3, 4, (H, W, 3), generator=g, device="cuda", dtype=torch.int16)
        if 150 <= t < 400:
            x0 = (20 + (t - 150) * 4 + seed * 13) % (W - 120)
            f[200:280, x0 : x0 + 120] += 90
        out[t] = f.clamp_(0, 255).to(torch.uint8)
    return out


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


LATENCY = """
import json, time, types
import numpy as np
from classifier_pipeline_b200.piclassifier.irmotiondetector import IRMotionDetector
from classifier_pipeline_b200.track.cliptracker import MOG2Background

class Window:
    start = end = types.SimpleNamespace(dt="00:00")
    def use_sunrise_sunset(self):
        return False
    def inside_window(self):
        return True

cfg = types.SimpleNamespace(recorder=types.SimpleNamespace(use_low_power_mode=False, rec_window=Window(), preview_secs=1, min_secs=5,
                                                           max_secs=600), location=types.SimpleNamespace())
det = IRMotionDetector(cfg, types.SimpleNamespace(model="IR", res_x=640, res_y=480, fps=10), background=MOG2Background())
rng = np.random.default_rng(0)
scene = rng.integers(30, 120, (480, 640, 3)).astype(np.int16)
frames = [np.clip(scene + rng.integers(-3, 4, scene.shape), 0, 255).astype(np.uint8) for _ in range(16)]
for t in range(150):
    det.process_frame(frames[t % 16])
lat = []
for t in range(400):
    t0 = time.perf_counter()
    det.process_frame(frames[t % 16])
    lat.append(time.perf_counter() - t0)
lat = np.array(lat) * 1e6
print(json.dumps(dict(p50_us=float(np.percentile(lat, 50)), p99_us=float(np.percentile(lat, 99)))))
"""


def streaming_latency(tree):
    """process_frame latency of a 640x480 detector with MOG2Background, detecting on every timed frame, in a child process
    from the source tree ``tree`` and the library built in it."""
    env = {k: v for k, v in os.environ.items() if k != "CPT_LIB"}
    out = subprocess.run([sys.executable, "-c", LATENCY], cwd=tree, env=env, capture_output=True, text=True, check=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def timed_clips(native, process_clips, dets, lists):
    """process_clips wall clock and the native call's own wall clock (it ends in a synchronise)."""
    spent = []
    inner = native.Context.ir_motion_clips

    def timed(self, *a):
        t0 = time.perf_counter()
        inner(self, *a)
        spent.append(time.perf_counter() - t0)

    native.Context.ir_motion_clips = timed
    try:
        t0 = time.perf_counter()
        traces = process_clips(dets, lists)
        wall = time.perf_counter() - t0
    finally:
        native.Context.ir_motion_clips = inner
    return traces, wall, sum(spent)


def same(a, b):
    return all(np.array_equal(x, y) for ta, tb in zip(a, b) for x, y in zip(ta, tb))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", default="1,8,32")
    ap.add_argument("--frames", type=int, default=600)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-clips", type=int, default=8)
    ap.add_argument("--loop-clips", type=int, default=2)
    ap.add_argument("--before-tree", default=None, help="a built source tree of the parent commit, for the streaming A/B")
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    assert torch.cuda.is_available(), "needs a CUDA device"
    res = dict(gpu=gpu_identity(), torch_device=torch.cuda.get_device_name(0), width=W, height=H, ring_frames=10, history=1000)
    T, counts = args.frames, [int(c) for c in args.clips.split(",")]
    clips = [make_clip(torch, s, T) for s in range(max(counts))]
    torch.cuda.synchronize()

    # (0) the three paths agree on every frame
    k = args.loop_clips
    host = [c.cpu().numpy() for c in clips[: max(k, args.host_clips)]]
    dev_tr = process_clips([make_detector() for _ in range(k)], clips[:k])
    host_tr = process_clips([make_detector() for _ in range(k)], [list(h) for h in host[:k]])
    dets = [make_detector() for _ in range(k)]
    t0 = time.perf_counter()
    loop_rows = [[(det.process_frame(f), det.triggered) for f in h] for det, h in zip(dets, host[:k])]
    loop_s = time.perf_counter() - t0
    loop_tr = [(np.array([r[0] for r in rows]), np.array([r[1] for r in rows])) for rows in loop_rows]
    assert same([t[:2] for t in dev_tr], loop_tr) and same(dev_tr, host_tr), "the paths disagree"
    res["agreement"] = dict(clips=k, frames_per_clip=T, frames_recording=[int(t.movement_detected.sum()) for t in dev_tr])
    # (3) the loop just timed
    res["loop"] = dict(clips=k, frames_per_clip=T, wall_s=loop_s, frames_per_s=k * T / loop_s, us_per_frame=loop_s / (k * T) * 1e6)

    # (1) device-resident frames
    bpf = bytes_per_frame()
    per_frame = sum(bpf.values())
    copy_bps = copy_rate(torch, 4 << 30)
    res["device"] = dict(bytes_per_frame=bpf, bytes_per_frame_total=per_frame, d2d_copy_bytes_per_s=copy_bps, runs=[])
    process_clips([make_detector()], [clips[0][:20]])  # warm-up: module load, scratch growth
    for n in counts:
        walls, calls = [], []
        for _ in range(args.reps):
            dets = [make_detector() for _ in range(n)]
            torch.cuda.synchronize()
            _, wall, call = timed_clips(native, process_clips, dets, clips[:n])
            walls.append(wall), calls.append(call)
            del dets
        best = min(calls)
        res["device"]["runs"].append(dict(clips=n, frames_per_clip=T, call_s=calls, wall_s=walls, frames_per_s=n * T / best,
                                          us_per_clip_frame=best / (n * T) * 1e6, process_clips_frames_per_s=n * T / min(walls),
                                          achieved_bytes_per_s=per_frame * n * T / best, share_of_copy=per_frame * n * T / best / copy_bps))

    # (2) host frames
    a = args.host_clips
    lists = [list(h) for h in host[:a]]
    process_clips([make_detector()], [lists[0][:20]])
    dets = [make_detector() for _ in range(a)]
    _, wall, call = timed_clips(native, process_clips, dets, lists)
    res["host"] = dict(clips=a, frames_per_clip=T, wall_s=wall, call_s=call, frames_per_s=a * T / wall)

    # (4) streaming latency, the two builds alternating
    del clips, host, lists, dets
    torch.cuda.empty_cache()
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
