"""Recordings -> classifier inputs, with and without the frames leaving the device.

  (a) wall clock of the whole API path on N synthetic clips (in-memory reader, as bench.py's parse_clips_api):
      existing:  parse_clips (frames copied back) + Interpreter.preprocess per track (frames uploaded again per clip)
      new:       parse_clips(keep_on_device=True) with keep_frames=False + Interpreter.preprocess_clips
  (b) device time of one preprocessing pass on BASELINE configs[2] (10 000 tracks x 45 frames, one 25-frame segment each),
      with the medians recomputed from the frames and with the extraction's frame medians reused (CUDA events, the two
      alternated in one process)
  (c) the algorithmic bytes of that pass under both accountings of SURVEY.md section 8d

Prints one JSON object; ``--out`` also writes it to a file.  Needs a CUDA device.
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

W, H = 160, 120
NPX = W * H


def gpu_identity():
    """Card name, power limit and max SM clock, read in the same run as the numbers."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def api_path(n_clips, frames, reps):
    """(a): the existing and the device-resident path, alternated ``reps`` times after one untimed warm-up of each;
    median, min and max over the repetitions."""
    import torch

    from classifier_pipeline_b200.config import Config
    from classifier_pipeline_b200.ml_tools.interpreter import HyperParams, Interpreter
    from classifier_pipeline_b200.synthetic import make_clip
    from classifier_pipeline_b200.track.clip import Clip
    from classifier_pipeline_b200.track.cliptrackextractor import ClipTrackExtractor
    from tests.tracking_helpers import MemReader

    store = {"c{}".format(i): make_clip(i, frames=frames) for i in range(n_clips)}
    config = Config.get_defaults()
    config.tracking["thermal"].denoise = False
    interp = Interpreter(HyperParams(), seed=1)

    def run(keep_on_device):
        ext = ClipTrackExtractor(config.tracking, False, cache_to_disk=False, keep_frames=not keep_on_device)
        ext.reader_factory = lambda path: MemReader(*store[path])
        clips = [Clip(config.tracking["thermal"], name) for name in store]
        np.random.seed(5)  # (the masked segment selection shuffles with the global generator: the same draws on both paths)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ext.parse_clips(clips, keep_on_device=keep_on_device)
        t1 = time.perf_counter()
        if keep_on_device:
            out = interp.preprocess_clips(clips)
        else:
            out = [[interp.preprocess(c, t) for t in c.tracks] for c in clips]
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return dict(parse_s=t1 - t0, preprocess_s=t2 - t1, total_s=t2 - t0), out, clips

    paths = (("existing", False), ("keep_on_device", True))
    outs = {}
    for key, kod in paths:
        _, outs[key], clips = run(kod)
    same = all(len(a) == len(b) and all(np.array_equal(x[1], y[1]) for x, y in zip(a, b))
               for a, b in zip(outs["existing"], outs["keep_on_device"]))
    samples = {key: [] for key, _ in paths}
    for _ in range(reps):
        for key, kod in paths:
            samples[key].append(run(kod)[0])
    res = {}
    for key, _ in paths:
        res[key] = {}
        for part in ("parse_s", "preprocess_s", "total_s"):
            v = np.array([t[part] for t in samples[key]])
            res[key][part] = {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}
        res[key]["frames_per_s"] = n_clips * frames / res[key]["total_s"]["median"]
    n_seg = sum(len(d) for c in outs["keep_on_device"] for _, d, _ in c)
    tracks = sum(len(c.tracks) for c in clips)
    res.update(workload="{} synthetic clips x {} frames -> {} tracks, {} segments (default HyperParams)".format(n_clips, frames, tracks, n_seg),
               reps=reps, outputs_identical=bool(same),
               speedup_total=res["existing"]["total_s"]["median"] / res["keep_on_device"]["total_s"]["median"],
               speedup_preprocess=res["existing"]["preprocess_s"]["median"] / res["keep_on_device"]["preprocess_s"]["median"])
    return res


def device_pass(n_clips, frames, n_tracks, steps):
    """(b) + (c) on frames and filtered images an extraction left in HBM."""
    import torch

    import bench
    from classifier_pipeline_b200 import engine
    from classifier_pipeline_b200.batch import BatchPreprocessor, linear_clips
    from classifier_pipeline_b200.synthetic import MODELS, make_clips_torch

    ex = engine.get_engine(None, W, H, 1)
    ex.ctx.use_torch_stream()
    slots = [ex.ctx.weight_table(m[3], max_frames=max(frames, 1024)) for m in MODELS]
    d_frames, models = make_clips_torch(n_clips, frames, torch.device("cuda", 0))
    clips = linear_clips([frames] * n_clips, np.array([MODELS[m][2] for m in models]), np.array([slots[m] for m in models]))
    out = ex.extract_device(d_frames, clips, keep_filtered=True, keep_labels=False, out={})
    d_t = d_frames.reshape(-1, H, W)
    total = n_clips * frames
    d_med = torch.empty(total, dtype=torch.float32, device="cuda")
    ex.ctx.frame_medians(d_t, total, d_med)  # (what the extraction computes whenever ClipStats are on)
    bp = BatchPreprocessor(ex)
    tracks = bench.synthetic_tracks(n_tracks, n_clips, frames, np.random.default_rng(77))
    lim, smp, seg, _ = bp.build_tables(tracks, seed=1)
    crop = (1, 1, W - 2, H - 2)
    outs = {"recomputed": {}, "reused": {}}
    kws = {"recomputed": {}, "reused": dict(frame_medians=d_med)}

    def one(key):
        return bp.run_tables(d_t, out["filtered"], lim, smp, seg, n_tracks, crop, out=outs[key], **kws[key])

    for key in kws:
        for _ in range(2):
            one(key)
    torch.cuda.synchronize()
    same = np.array_equal(outs["recomputed"]["segments"].cpu().numpy(), outs["reused"]["segments"].cpu().numpy())
    ms = {k: [] for k in kws}
    for _ in range(steps):
        for key in kws:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one(key)
            e1.record()
            torch.cuda.synchronize()
            ms[key].append(e0.elapsed_time(e1))
    n_seg, n_smp = seg.shape[0], len(smp)
    crop_bytes = int((smp["width"].astype(np.int64) * smp["height"] * 6).sum()) + int((lim["width"].astype(np.int64) * lim["height"] * 4).sum())
    bytes_recomputed = n_seg * 204800 + n_smp * NPX * 2 + crop_bytes
    bytes_reused = n_seg * 204800 + n_smp * 4 + crop_bytes
    res = {"workload": "BASELINE configs[2]: {} tracks x 45 frames, one 25-frame segment each -> ({}, 160, 160, 2) float32, frames of {} "
                       "clips x {} frames in HBM".format(n_tracks, n_seg, n_clips, frames),
           "outputs_identical": bool(same), "unique_track_frames": n_smp, "segments": n_seg, "steps": steps}
    for key, b in (("recomputed", bytes_recomputed), ("reused", bytes_reused)):
        v = np.array(ms[key])
        res["medians_" + key] = {"ms_median": float(np.median(v)), "ms_min": float(v.min()), "ms_max": float(v.max()),
                                 "segments_per_s": n_seg / (np.median(v) * 1e-3), "algorithmic_bytes": b,
                                 "bytes_per_segment": b / n_seg, "achieved_GBps": b / (np.median(v) * 1e-3) / 1e9}
    res["medians_recomputed"]["accounting"] = "SURVEY 8d, medians recomputed: 204800 B written per segment + one full-frame read per unique track-frame + the crops"
    res["medians_reused"]["accounting"] = "SURVEY 8d, medians reused: 204800 B written per segment + the crops + one 4-byte median per unique track-frame"
    res["pass_speedup"] = res["medians_recomputed"]["ms_median"] / res["medians_reused"]["ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--clips", type=int, default=8, help="(a): synthetic clips")
    ap.add_argument("--frames", type=int, default=300, help="(a): frames per clip")
    ap.add_argument("--reps", type=int, default=7, help="(a): timed repetitions of each path (after one warm-up)")
    ap.add_argument("--pass-clips", type=int, default=148, help="(b): clips whose frames the tracks are drawn from")
    ap.add_argument("--pass-frames", type=int, default=300, help="(b): frames per clip")
    ap.add_argument("--tracks", type=int, default=10000, help="(b): tracks (BASELINE configs[2]: 10 000)")
    ap.add_argument("--steps", type=int, default=20, help="(b): timed passes of each kind")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_classify_inputs: no CUDA device")
    res = {"gpu": gpu_identity(), "torch_device": torch.cuda.get_device_name(0)}
    res["device_pass"] = device_pass(args.pass_clips, args.pass_frames, args.tracks, args.steps)
    res["api_path"] = api_path(args.clips, args.frames, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
