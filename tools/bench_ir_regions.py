"""Regions of whole IR clips at 640x480: MOG2, open, threshold, components and rectangle merging for every frame.

  (a) the per-frame loop: MOG2Background.update_background + detect_ir_regions(compute_filtered(None)) for each frame
  (b) ir_clip_regions: one MOG2 call, one components call and one merge launch for the clip
  (c) cv2 on the host: MOG2 apply, open, threshold, connectedComponentsWithStats and merge_components per frame, with the
      thread count cv2 reports

The clips are seeded grey frames (tests/ir_region_designs.py ir_gray_clip: a textured scene, sensor noise and a few warm
objects moving across it).  Four clips of 500 frames: each clip's 500 masks (154 MB) exceed the B200's 126 MB L2.  The three
paths are checked equal on every frame before anything is timed.  Wall times end in a device synchronise.  Kernel times
come from CUDA events around the components call (cpt_detect_objects_batch) and the merge launch
(cpt_ir_merge_components) on the masks of (b).  Prints one JSON object; ``--out`` also writes it.  Needs a CUDA device.
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


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else None


def per_frame_loop(clip):
    import torch

    from classifier_pipeline_b200.track.cliptracker import MOG2Background
    from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions

    bg = MOG2Background()
    out = []
    for f in clip:
        bg.update_background(f)
        out.append(detect_ir_regions(bg.compute_filtered(None)))
    torch.cuda.synchronize()
    return out


def clip_call(d_clip):
    import torch

    from classifier_pipeline_b200.track.cliptracker import MOG2Background
    from classifier_pipeline_b200.track.irtrackextractor import ir_clip_regions

    out = ir_clip_regions(d_clip, MOG2Background())
    torch.cuda.synchronize()
    return out


def host_cv2(clip):
    import cv2

    from classifier_pipeline_b200.track.irtrackextractor import merge_components

    m = cv2.createBackgroundSubtractorMOG2(history=1000, varThreshold=16, detectShadows=False)
    out = []
    for f in clip:
        mask = m.apply(f, None, -1)
        _, t = cv2.threshold(cv2.morphologyEx(mask, cv2.MORPH_OPEN, (15, 15)), 0, 255, cv2.THRESH_BINARY)
        n, labels, stats, _ = cv2.connectedComponentsWithStats(t)
        out.append((labels, stats, merge_components(list(stats[1:]))))
    return out


def kernel_times(d_masks, reps):
    """CUDA-event times (ms) of the components call and of the merge launch over one clip's device masks."""
    import torch

    from classifier_pipeline_b200 import engine, native
    from classifier_pipeline_b200.ml_tools import detect
    from classifier_pipeline_b200.track.irtrackextractor import merge_limits

    eng = engine.get_engine()
    eng.ctx.use_torch_stream()
    n, h, w = d_masks.shape
    mc = detect.MAX_COMPONENTS
    i32 = dict(dtype=torch.int32, device=d_masks.device)
    counts, stats = torch.empty(n, **i32), torch.empty((n, mc + 1, 5), **i32)
    mcounts, merged = torch.empty(n, **i32), torch.empty((n, mc, 5), **i32)
    comp, merge = [], []
    for _ in range(reps + 1):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        eng.ctx.detect_objects_batch(d_masks, n, w, h, 0, native.DETECT_OPEN_GRAY, mc, counts, stats)
        e[1].record()
        eng.ctx.ir_merge_components(stats, counts, n, mc, *merge_limits(), merged, mcounts)
        e[2].record()
        torch.cuda.synchronize()
        comp.append(e[0].elapsed_time(e[1]))
        merge.append(e[1].elapsed_time(e[2]))
    comp, merge = comp[1:], merge[1:]  # the first call warms up
    return dict(components_ms=float(np.median(comp)), merge_ms=float(np.median(merge)),
                components_us_per_frame=float(np.median(comp)) * 1e3 / n, merge_us_per_frame=float(np.median(merge)) * 1e3 / n,
                components_per_frame=float(counts.float().mean()) - 1, merged_per_frame=float(mcounts.float().mean()), reps=reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=4)
    ap.add_argument("--frames", type=int, default=500)
    ap.add_argument("--out")
    args = ap.parse_args()

    import cv2
    import torch

    from tests import ir_region_designs as ird

    assert torch.cuda.is_available(), "bench_ir_regions needs a CUDA device"
    ident = gpu_identity()
    clips = [ird.ir_gray_clip(100 + c, args.frames) for c in range(args.clips)]
    d_clips = [torch.from_numpy(c).cuda() for c in clips]
    total = args.clips * args.frames

    # equal outputs first (this also warms every path up)
    for clip, d in zip(clips, d_clips):
        a, b, c = per_frame_loop(clip), clip_call(d), host_cv2(clip)
        for t in range(len(clip)):
            want = np.array(c[t][2], np.int32).reshape(-1, 5)
            assert np.array_equal(a[t][0], c[t][0]) and np.array_equal(np.array(a[t][1], np.int32).reshape(-1, 5), want), t
            assert np.array_equal(b[0][t], c[t][1]) and np.array_equal(b[1][t], want), t

    res = dict(gpu=ident, torch=torch.__version__, cv2=cv2.__version__, cv2_threads=cv2.getNumThreads(), clips=args.clips,
               frames_per_clip=args.frames, width=ird.W, height=ird.H, outputs_equal=True)
    timings = {}
    for name, fn, inputs in (("a_per_frame_loop", per_frame_loop, clips), ("b_ir_clip_regions", clip_call, d_clips),
                             ("c_cv2_host", host_cv2, clips)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for x in inputs:
            fn(x)
        torch.cuda.synchronize()
        timings[name] = dict(wall_s=time.perf_counter() - t0)
        timings[name]["wall_us_per_frame"] = timings[name]["wall_s"] * 1e6 / total
    res["wall"] = timings
    # kernel times of the components passes and the merge on one clip's masks, as (b) produces them
    from classifier_pipeline_b200.track.cliptracker import MOG2Background

    masks = MOG2Background().update_backgrounds(d_clips[0])
    res["kernels_one_clip"] = kernel_times(masks, reps=10)
    # the per-frame loop's components for comparison: one frame per call
    single = []
    for t in range(0, args.frames, 10):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions

        detect_ir_regions(masks[t].cpu().numpy())
        e[1].record()
        torch.cuda.synchronize()
        single.append(e[0].elapsed_time(e[1]))
    res["detect_ir_regions_single_call_ms_p50"] = float(np.median(single))
    res["speedup_b_over_a"] = timings["a_per_frame_loop"]["wall_s"] / timings["b_ir_clip_regions"]["wall_s"]
    res["speedup_b_over_c"] = timings["c_cv2_host"]["wall_s"] / timings["b_ir_clip_regions"]["wall_s"]
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=2) + "\n")


if __name__ == "__main__":
    main()
