#!/usr/bin/env python
"""bench.py -- thermal frames/s tracked (160x120) on N B200s, with roofline and CPU baseline.

One *step* = one pass of the extraction hot path (ClipTrackExtractor.parse_clip arithmetic:
K1,K2,K4,K5,K6,K7 of SURVEY.md section 8) over one batch of synthetic Lepton clips resident in
HBM: BASELINE.json configs[1], 1024 clips x 900 frames x 160x120 uint16 per GPU, emitting
filtered fp32 + uint8 label image + region lists for every frame.  Clips are independent, so
N GPUs each take their own 1024 clips (weak scaling, no collective on the data path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--clips C] [--frames T] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference      # CPU port of the reference path on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 160, 120
NPX = W * H
# SURVEY.md section 8(d): algorithmic bytes per frame = read uint16 frame + write fp32 filtered +
# write uint8 label image (region lists and per-clip state ignored).
BYTES_PER_FRAME = NPX * 2 + NPX * 4 + NPX * 1
METRIC = "thermal frames/sec tracked+preprocessed (160x120)"
UNIT = "frames/s"


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    QUERY = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop = threading.Event()
        self.thread = threading.Thread(target=self.run, daemon=True)

    def run_nvml(self):
        """NVML from this process: a sample every 25 ms (an nvidia-smi process takes longer to start than a step to run)."""
        import pynvml as nv

        nv.nvmlInit()
        index = self.index
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        if vis:  # the CUDA ordinal counts visible devices only
            ids = [v.strip() for v in vis.split(",")]
            if index < len(ids) and ids[index].isdigit():
                index = int(ids[index])
        h = nv.nvmlDeviceGetHandleByIndex(index)
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self.stop.is_set():
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            r = reasons(h)
            self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for _, b in bits])
            self.stop.wait(0.025)

    def run(self):
        try:
            return self.run_nvml()
        except Exception:
            pass
        while not self.stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits"],
                    capture_output=True, text=True, timeout=5,
                ).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=10)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max((int(s[1]) for s in self.samples if s[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.samples)}


def measured_traffic(total_frames):
    """DRAM bytes of one launch of the dominant kernel, CAPTURED ONCE under `ncu --set full` (profiles/extract_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum of the captured launch) and SCALED per frame to this launch -- not a
    measurement of this run (a profiler cannot run inside a timed bench).  Returns (bytes, description)."""
    path = os.path.join(ROOT, "profiles", "extract_traffic.json")
    try:
        d = json.load(open(path))
        return float(d["dram_bytes_per_frame"]) * total_frames, "captured ({} frames, {}) and scaled per frame to this launch".format(
            d.get("frames_in_captured_launch"), os.path.basename(d.get("source", "ncu")))
    except Exception:
        return None, "no capture committed"


def synthetic_tracks(n_tracks, n_clips, frames, rng, span=45, pick=25):
    """BASELINE configs[2]: tracks of `span` consecutive frames with drifting boxes inside the crop rectangle
    (w, h in U(6, 40)); one segment per track = `pick` of its `span` frames (the README's 25-of-45)."""
    tracks = []
    for i in range(n_tracks):
        clip = i % n_clips
        t0 = int(rng.integers(0, max(frames - span, 1)))
        n = min(span, frames - t0)
        w, h = int(rng.integers(6, 41)), int(rng.integers(6, 41))
        x = rng.integers(1, 159 - w + 1) + np.cumsum(rng.integers(-2, 3, n))
        y = rng.integers(1, 119 - h + 1) + np.cumsum(rng.integers(-2, 3, n))
        x = np.clip(x, 1, 159 - w)
        y = np.clip(y, 1, 119 - h)
        f = clip * frames + t0 + np.arange(n)
        regions = np.stack([f, x, y, np.full(n, w), np.full(n, h), np.zeros(n, np.int64)], axis=1)
        seg = np.sort(rng.choice(f, min(pick, n), replace=False))
        tracks.append((regions, [seg]))
    return tracks


def bench_preprocess(ex, d_frames, d_filtered, n_clips, frames, n_tracks, steps, torch):
    """Config C: Interpreter.preprocess_segments for n_tracks tracks (3 launches) on frames resident in HBM."""
    from classifier_pipeline_b200.batch import BatchPreprocessor

    bp = BatchPreprocessor(ex)
    rng = np.random.default_rng(77)
    tracks = synthetic_tracks(n_tracks, n_clips, frames, rng)
    t_host = time.perf_counter()
    lim, smp, seg, _ = bp.build_tables(tracks, seed=1)
    host_tables_s = time.perf_counter() - t_host
    # the same tables from flat arrays (what a pipeline holding device-produced region lists would pass)
    flat_R = np.concatenate([r for r, _ in tracks])
    flat_t = np.repeat(np.arange(n_tracks), [len(r) for r, _ in tracks])
    flat_f = np.concatenate([sg[0] for _, sg in tracks])
    flat_n = np.array([len(sg[0]) for _, sg in tracks])
    t_host = time.perf_counter()
    bp.build_tables_flat(flat_R, flat_t, flat_f, flat_n, np.arange(n_tracks), seed=1)
    host_tables_flat_s = time.perf_counter() - t_host
    d_t = d_frames.reshape(-1, H, W)
    out = {}
    crop = (1, 1, W - 2, H - 2)
    for _ in range(2):
        bp.run_tables(d_t, d_filtered, lim, smp, seg, n_tracks, crop, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        bp.run_tables(d_t, d_filtered, lim, smp, seg, n_tracks, crop, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    n_seg, n_smp = seg.shape[0], len(smp)
    # algorithmic bytes (SURVEY.md section 8d, medians recomputed): 204800 B written per segment + one full-frame
    # read per unique track-frame for its median + the crops (thermal u16 + filtered f32)
    crop_bytes = int((smp["width"].astype(np.int64) * smp["height"] * 6).sum()) + int((lim["width"].astype(np.int64) * lim["height"] * 4).sum())
    alg_bytes = n_seg * 204800 + n_smp * NPX * 2 + crop_bytes
    return {
        "workload": "BASELINE configs[2]: {} tracks x 45 frames, one 25-frame segment each -> ({}, 160, 160, 2) float32".format(n_tracks, n_seg),
        "segments_per_s": n_seg / (ms * 1e-3), "track_frames_per_s": n_smp / (ms * 1e-3), "ms": ms, "launches_per_pass": 4,
        "achieved_GBps": alg_bytes / (ms * 1e-3) / 1e9, "algorithmic_bytes": alg_bytes,
        "roofline": {"bound": "hbm", "achieved": alg_bytes / (ms * 1e-3) / 1e9, "peak": measured_peak()[0], "unit": "GB/s",
                     "frac": alg_bytes / (ms * 1e-3) / 1e9 / measured_peak()[0],
                     "accounting": "204800 B written per segment + one full-frame read per unique track-frame (medians recomputed) + the crops"},
        "host_table_build_s": host_tables_s, "host_table_build_flat_s": host_tables_flat_s,
    }


class _Window:
    start = type("T", (), {"dt": "00:00"})()
    end = type("T", (), {"dt": "00:00"})()

    def use_sunrise_sunset(self):
        return False

    def inside_window(self):
        return True


def bench_motion(n_frames=400):
    """Config D: CPTVMotionDetector.process_frame at batch 1 -- host frame in, one fused launch, 32 bytes back."""
    import types

    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import CPTVMotionDetector
    from classifier_pipeline_b200.synthetic import make_clip

    pix, _ = make_clip(0, frames=n_frames)
    cfg = types.SimpleNamespace(
        motion=types.SimpleNamespace(temp_thresh=2750, delta_thresh=50, count_thresh=3, frame_compare_gap=45, one_diff_only=True,
                                     trigger_frames=2, edge_pixels=1, warmer_only=True),
        recorder=types.SimpleNamespace(use_low_power_mode=False, rec_window=_Window(), preview_secs=5, min_secs=5, max_secs=600),
        location=types.SimpleNamespace())
    headers = types.SimpleNamespace(model="lepton3", res_x=W, res_y=H, fps=9)
    CPTVMotionDetector.BACKGROUND_WEIGHT_ADD = 0.1
    det = CPTVMotionDetector(cfg, None, headers, detect_after=0)
    frames = [types.SimpleNamespace(pix=pix[t], time_on=10_000_000 + t * 111, last_ffc_time=0) for t in range(n_frames)]
    lat, moved = [], 0
    for t, f in enumerate(frames):
        t0 = time.perf_counter()
        moved += bool(det.process_frame(f))
        if t >= 50:
            lat.append(time.perf_counter() - t0)
    lat = np.sort(np.array(lat)) * 1e6
    return {"workload": "BASELINE configs[3]: one stream, batch 1, host frame in / motion flag out", "frames": n_frames,
            "p50_us": float(lat[len(lat) // 2]), "p99_us": float(lat[int(len(lat) * 0.99)]), "max_us": float(lat[-1]),
            "frames_with_motion": int(moved), "realtime_budget_us": 111111}


def cpu_baseline(n_threads, clips_per_thread, frames, pix=None, want_regions=False):
    """The C port of the reference path (oracle/) on the host cores, regions-only outputs."""
    from classifier_pipeline_b200.synthetic import clip_model, make_clip
    from oracle import oracle as orc

    n_clips = n_threads * clips_per_thread
    if pix is None:
        pix = np.stack([make_clip(i, frames=frames)[0] for i in range(n_clips)])
    n_clips, frames = pix.shape[0], pix.shape[1]
    params = [orc.make_params(background_thresh=clip_model(i)[2], weight_add=clip_model(i)[3], max_comp=16) for i in range(n_clips)]
    orc.extract_batch(pix[:1, : min(frames, 20)], params[:1], 1)  # warm the library
    t0 = time.perf_counter()
    res = orc.extract_batch(pix, params, n_threads)
    dt = time.perf_counter() - t0
    if want_regions:
        return n_clips * frames / dt, dt, n_clips, res
    return n_clips * frames / dt, dt, n_clips


def check_parity(hout, port, n_clips, frames, max_regions=16):
    """The GPU's e2e region lists against the C port's on the clips both processed: component counts and the stats rows
    (x, y, width, height, area) of every stored region must be identical.  Returns the number of regions compared."""
    ncomp, comp, _ = port
    info, regions = hout["info"], hout["regions"]
    got_n = info["n_components"][: n_clips * frames].reshape(n_clips, frames)
    if not np.array_equal(got_n, ncomp):
        bad = np.argwhere(got_n != ncomp)[0]
        raise SystemExit("PARITY FAILURE: clip {} frame {}: {} components on the GPU, {} in the CPU port".format(
            bad[0], bad[1], got_n[tuple(bad)], ncomp[tuple(bad)]))
    r = regions[: n_clips * frames].reshape(n_clips, frames, -1)
    got = np.stack([r["x"], r["y"], r["width"], r["height"], r["area"]], axis=-1)[:, :, :max_regions]
    live = np.arange(max_regions)[None, None, :] < np.minimum(ncomp, max_regions)[:, :, None]
    if not np.array_equal(got[live], comp[:, :, :max_regions, :5][live]):
        raise SystemExit("PARITY FAILURE: region statistics differ between the GPU and the CPU port")
    return int(live.sum())


DUMP_FRAMES = 256  # frames written by --dump-outputs: about 40 MB in all


def dump_outputs(out, total, directory, seed=0):
    """Write what one extraction step returned for a fixed, seeded sample of DUMP_FRAMES frames of the batch, so that two
    builds can be compared output for output: filtered images and label images (float32), and the frame records and region
    lists (float64, one file per field; region slots past the frame's stored regions carry no result and are written as
    zero)."""
    import torch

    from classifier_pipeline_b200.batch import BatchExtractor

    idx = np.sort(np.random.default_rng(seed).choice(total, min(total, DUMP_FRAMES), replace=False))
    d_idx = torch.from_numpy(idx).to(out["info"].device)
    info = BatchExtractor.info_numpy(out["info"].index_select(0, d_idx))
    regions = BatchExtractor.regions_numpy(out["regions"].index_select(0, d_idx))
    live = np.arange(regions.shape[1])[None, :] < np.minimum(info["n_components"], regions.shape[1])[:, None]
    arrays = {"frame_index": idx.astype(np.float64),
              "filtered": out["filtered"].index_select(0, d_idx).cpu().numpy().astype(np.float32),
              "labels": out["labels"].index_select(0, d_idx).cpu().numpy().astype(np.float32)}
    for name in info.dtype.names:
        if name != "reserved":
            arrays["info_" + name] = info[name].astype(np.float64)
    for name in regions.dtype.names:
        arrays["region_" + name] = np.where(live, regions[name], 0).astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def workload_config(C, T):
    """The workload both arms (`--impl b200` and `--impl reference`) are quoted on."""
    return {
        "workload": "BASELINE configs[1]: {} clips x {} frames 160x120 uint16 per GPU, full track extraction (filtered fp32 + labels u8 + regions)".format(C, T),
        "clips_per_gpu": C, "frames_per_clip": T, "denoise": False,
        "l2": "inputs ({:.1f} GB) far larger than L2".format(C * T * NPX * 2 / 1e9),
    }


def reference_python_record():
    """The UNMODIFIED reference's own extractor (Python + numpy + OpenCV) cannot travel to the GPU box (/root/reference is
    absent there); its throughput was timed in the build container with tools/time_reference.py and is committed."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "reference_python_cpu.json")))
    except Exception:
        return None


def bench_extras(ex, d_frames, clips, bts, wts, C, T, torch):
    """Measurement legs beside the headline: TrackingConfig.denoise (the reference's default config) through the device NLM
    passes, the Python API (parse_clips: decode + launch + D2H + the host matcher) and streaming process_frame latency."""
    import types

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.config import Config
    from classifier_pipeline_b200.track.clip import Clip
    from classifier_pipeline_b200.track.cliptrackextractor import ClipTrackExtractor

    res = {}
    # ---- denoise on: 32 clips x 100 frames (NLM is compute-bound: 441 search offsets per pixel)
    n_c, n_t = min(32, C), min(100, T)
    sub = d_frames[:n_c, :n_t].contiguous()
    dc = linear_clips([n_t] * n_c, bts[:n_c], wts[:n_c], flags=native.CLIP_UPDATE_BACKGROUND | native.CLIP_DENOISE)
    o = {}
    ex.extract_device(sub, dc, keep_filtered=True, keep_labels=True, out=o)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ex.extract_device(sub, dc, keep_filtered=True, keep_labels=True, out=o)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    res["denoise_on"] = {"workload": "{} clips x {} frames, CPT_CLIP_DENOISE (cv2.fastNlMeansDenoising bit-exact on the device)".format(n_c, n_t),
                         "frames_per_s": n_c * n_t / (ms * 1e-3), "ms": ms}
    del o, sub

    # ---- the Python API: parse_clips on in-memory clips (device launch, D2H of frames / masks / regions, host matcher)
    class Mem:
        def __init__(self, pix, model):
            self.pix, self.i, self.model = pix, 0, model

        def get_header(self):
            return types.SimpleNamespace(x_resolution=W, y_resolution=H, model=self.model, brand="flir", timestamp=1_600_000_000_000_000)

        def next_frame(self):
            if self.i >= len(self.pix):
                return None
            f = types.SimpleNamespace(pix=self.pix[self.i], time_on=10_000_000 + self.i * 111, last_ffc_time=0, temp_c=20.0,
                                      last_ffc_temp_c=20.0, background_frame=False)
            self.i += 1
            return f

    n_api, t_api = min(8, C), min(300, T)
    host = d_frames[:n_api, :t_api].view(torch.int16).cpu().numpy().view(np.uint16)
    config = Config.get_defaults()
    config.tracking["thermal"].denoise = False
    ext = ClipTrackExtractor(config.tracking, False, cache_to_disk=False)
    store = {"c{}".format(i): (host[i], "lepton3" if i % 2 == 0 else "lepton3.5") for i in range(n_api)}
    ext.reader_factory = lambda path: Mem(*store[path])
    for rep in range(2):
        api_clips = [Clip(config.tracking["thermal"], name) for name in store]
        t0 = time.perf_counter()
        ext.parse_clips(api_clips)
        api_dt = time.perf_counter() - t0
    res["parse_clips_api"] = {"workload": "{} clips x {} frames through ClipTrackExtractor.parse_clips (launch + D2H of frames, masks, regions + host "
                              "matcher / Kalman / track filtering in Python)".format(n_api, t_api),
                              "frames_per_s": n_api * t_api / api_dt, "tracks": int(sum(len(c.tracks) for c in api_clips)), "seconds": api_dt}

    # ---- streaming: process_frame one frame at a time (ring upload, one launch, region read-back, host matcher)
    clip = Clip(config.tracking["thermal"], "c0")
    ext2 = ClipTrackExtractor(config.tracking, False, cache_to_disk=False, keep_frames=False, calc_stats=False)
    ext2.reader_factory = ext.reader_factory
    ext2.init_clip(clip)
    lat = []
    for t in range(min(250, t_api)):
        f = types.SimpleNamespace(pix=host[0][t], time_on=10_000_000 + t * 111, last_ffc_time=0, background_frame=False)
        t0 = time.perf_counter()
        ext2.process_frame(clip, f, update_background=True)
        if t >= 50:
            lat.append(time.perf_counter() - t0)
    lat = np.sort(np.array(lat)) * 1e6
    res["process_frame_streaming"] = {"workload": "ClipTrackExtractor.process_frame, one frame per call (host frame in, tracks out)",
                                      "p50_us": float(lat[len(lat) // 2]), "p99_us": float(lat[int(len(lat) * 0.99)]),
                                      "realtime_budget_us": 111111}
    res["ir_640x480"] = bench_ir(ex)
    return res


def bench_ir(ex, n_frames=120):
    """The 640x480 IR part of BASELINE configs[4] (ird.py): the device half of IRMotionDetector.process_frame -- BGR to grey,
    difference against the frame three back, threshold, 3x3 erosion, count -- one host frame per call, and detect_objects_ir
    on one grey image."""
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.ml_tools import detect

    rng = np.random.default_rng(5)
    base = rng.integers(0, 80, size=(480, 640, 3)).astype(np.uint8)
    frames = []
    for t in range(8):
        f = base.copy()
        f[100 + 4 * t : 160 + 4 * t, 200 + 6 * t : 280 + 6 * t] += 120
        frames.append(f)
    ir = native.IrMotion(ex.ctx, 640, 480, 4)
    lat = []
    for t in range(n_frames):
        t0 = time.perf_counter()
        ir.gray(frames[t % 8], t % 4)
        if t >= 3:
            ir.detect(t % 4, (t - 3) % 4, 30, 3)
        if t >= 20:
            lat.append(time.perf_counter() - t0)
    ir.close()
    lat = np.sort(np.array(lat)) * 1e6
    gray = frames[0][:, :, 1].copy()
    det = []
    for _ in range(12):
        t0 = time.perf_counter()
        n, _, _ = detect.detect_objects_ir(gray, threshold=100)
        det.append(time.perf_counter() - t0)
    det = np.sort(np.array(det[2:])) * 1e6
    bytes_in = 640 * 480 * 3
    return {"workload": "BASELINE configs[4], IR part: 640x480 BGR frames, IRMotionDetector device half (grey, absdiff vs 3 frames back, "
                        "threshold, 3x3 erode, count), one host frame in / two counters out per call",
            "p50_us": float(lat[len(lat) // 2]), "p99_us": float(lat[int(len(lat) * 0.99)]), "frames_per_s": float(1e6 / lat.mean()),
            "h2d_bytes_per_frame": bytes_in, "pcie_GBps": float(bytes_in / (lat.mean() * 1e-6) / 1e9),
            "bound": "latency: five small launches and a 0.9 MB pageable host-to-device copy per frame; the camera delivers 10-30 fps",
            "detect_objects_ir_p50_us": float(det[len(det) // 2]), "detect_objects_ir_components": int(n)}


def bind_to_gpu_node(torch, local_rank):
    """One rank per GPU: run on the cores of the GPU's NUMA node, so that the rank's pinned staging buffers (first touch) and
    its copy threads sit next to the PCIe root the GPU hangs off.  Returns the node, or None when the box does not say."""
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/{:04x}:{:02x}:{:02x}.0/numa_node".format(dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node{}/cpulist".format(node)).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except (OSError, ValueError, AttributeError):
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, 64))
    frames = args.frames
    per_thread = 2  # ~3 s of work per step on every host thread
    values = []
    sample = ""
    for step in range(args.warmup + args.steps):
        v, dt, n_clips = cpu_baseline(threads, per_thread, frames)
        sample = "{} clips x {} frames of the bench workload ({} synthetic clips family), {:.1f} s".format(n_clips, frames, "seeded", dt)
        if step >= args.warmup:
            values.append((v, dt))
    value = float(np.mean([v for v, _ in values]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(np.mean([dt for _, dt in values]) * 1e3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u16/int32 (fp32+fp64 scalars)", "data": "synthetic",
        "config": workload_config(args.clips, args.frames),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample + " per step (a bounded sample of the workload)",
                         "reference_python": reference_python_record()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--clips", type=int, default=1024, help="clips per GPU")
    ap.add_argument("--frames", type=int, default=900)
    ap.add_argument("--e2e-clips", type=int, default=0, help="clips per e2e step (0 = auto from host RAM)")
    ap.add_argument("--e2e-chunk", type=int, default=16, help="clips per staged chunk of the host-staged e2e calls (measured: 64 -> 2.39, 32 -> 2.58, 16 -> 2.68, 8 -> 2.70 M frames/s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tracks", type=int, default=10000, help="tracks of the preprocessing measurement (0 = skip)")
    ap.add_argument("--no-motion", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the denoise / parse_clips / streaming legs")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs as DIR/<name>.npy "
                    "(rank 0's clips)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import BatchExtractor, linear_clips
    from classifier_pipeline_b200.synthetic import MODELS, make_clips_torch

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_node(torch, local_rank) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    C, T = args.clips, args.frames
    ex = BatchExtractor(device=local_rank, max_regions=16)
    slots = [ex.ctx.weight_table(m[3], max_frames=max(T, 1024)) for m in MODELS]
    first = rank * C  # each rank owns its own clips (clip-wise sharding, SURVEY.md section 8e)
    d_frames, models = make_clips_torch(C, T, torch.device("cuda", local_rank), first_index=first)
    bts = np.array([MODELS[m][2] for m in models])
    wts = np.array([slots[m] for m in models])
    clips = linear_clips([T] * C, bts, wts)
    total = C * T
    out = {}
    torch.cuda.synchronize()

    def step():
        ex.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, out=out)

    for _ in range(max(args.warmup, 1)):
        step()
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_events = []
    with ClockSampler(local_rank) as clocks:
        barrier()
        start.record()
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            kernel_events.append((e0, e1))
        stop.record()
        barrier()
    ms_total = start.elapsed_time(stop)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kernel_events]))
    if args.dump_outputs and rank == 0:
        dump_outputs(out, total, args.dump_outputs)
    # per-kernel durations of a step: CUDA events recorded by the library around its own launches, on its own stream
    # (torch events only see torch's current stream), averaged over a few extra steps outside the timed region
    import ctypes

    kt = np.zeros(5, dtype=np.float64)
    buf5 = (ctypes.c_float * 5)()
    native.check(ex.ctx.lib.cpt_debug_kernel_times_ex(ex.ctx._h, 1, None, 5))
    n_kt = max(2, min(args.steps, 5))
    for _ in range(n_kt):
        step()
        native.check(ex.ctx.lib.cpt_debug_kernel_times_ex(ex.ctx._h, 1, buf5, 5))
        kt += np.array(list(buf5), dtype=np.float64)
    native.check(ex.ctx.lib.cpt_debug_kernel_times_ex(ex.ctx._h, 0, None, 5))
    kt /= n_kt
    if dist is not None:
        tt = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
    ms_per_step = ms_total / args.steps
    value = world * total / (ms_per_step * 1e-3)
    info = ex.info_numpy(out["info"])
    regions_total = int(np.minimum(info["n_components"], 16).sum())

    # ---- classifier-input preprocessing (configs[2]) on the frames / filtered images still resident in HBM
    preprocess = None
    if args.tracks > 0 and rank == 0:
        preprocess = bench_preprocess(ex, d_frames, out["filtered"], C, T, args.tracks, max(2, min(args.steps, 5)), torch)

    # ---- e2e: host frames in, host region lists out, through the C-ABI host call
    e2e = None
    try:
        import psutil

        avail = psutil.virtual_memory().available
    except Exception:
        avail = 16 << 30
    # (every rank pins its own staging copy at the same time: share the host's free memory between the ranks)
    e2e_clips = args.e2e_clips or int(max(8, min(C, (avail // (4 * world)) // (T * NPX * 2), 256)))
    from classifier_pipeline_b200.synthetic import pack_clips_torch

    h_frames = native.pinned_empty((e2e_clips * T, H, W), np.uint16)
    h_frames[:] = d_frames.view(torch.int16)[:e2e_clips].reshape(-1, H, W).cpu().numpy().view(np.uint16)
    # the same clips PACKED as their CPTV v2 frame payloads (what a reader holds after inflating a .cptv file)
    p_stream, p_table, p_first = pack_clips_torch(d_frames[:e2e_clips])
    e_clips = linear_clips([T] * e2e_clips, bts[:e2e_clips], wts[:e2e_clips])
    # ---- the other measurement legs that need the device-resident batch (rank 0 only)
    extras = {}
    if rank == 0 and not args.no_extras:
        extras = bench_extras(ex, d_frames, clips, bts, wts, C, T, torch)
    del d_frames
    out.clear()
    torch.cuda.empty_cache()

    def time_host(call):
        for _ in range(2):
            call()
        barrier()
        t0 = time.perf_counter()
        n = max(2, min(args.steps, 5))
        for _ in range(n):
            call()
        barrier()
        dt = (time.perf_counter() - t0) / n
        if dist is not None:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        return dt

    hout, hraw = {}, {}
    e2e_dt = time_host(lambda: ex.extract_host_packed(p_stream, p_table, p_first, e_clips, chunk_clips=args.e2e_chunk, out=hout))
    raw_dt = time_host(lambda: ex.extract_host(h_frames, e_clips, chunk_clips=args.e2e_chunk, out=hraw))
    d2h = int(e2e_clips * T * (16 * native.REGION_DTYPE.itemsize + native.INFO_DTYPE.itemsize))
    e2e = {
        "value": world * e2e_clips * T / e2e_dt, "unit": UNIT,
        "h2d_bytes_per_step": int(p_stream.size + p_table.nbytes), "d2h_bytes_per_step": d2h,
        "clips_per_step": e2e_clips,
        "api": "cpt_extract_batch_cptv_host (pinned inflated CPTV frame payloads, {:.2f} B/pixel -> device decode -> host region lists)".format(
            p_stream.size / (e2e_clips * T * NPX)),
        "raw_u16": {"value": world * e2e_clips * T / raw_dt, "h2d_bytes_per_step": int(e2e_clips * T * NPX * 2),
                    "api": "cpt_extract_batch_host (pinned decoded uint16 frames -> host region lists)"},
    }
    same = np.array_equal(hout["info"]["n_components"], hraw["info"]["n_components"]) and np.array_equal(hout["info"]["thermal_sum"], hraw["info"]["thermal_sum"])
    if not same:
        raise SystemExit("PARITY FAILURE: the packed and the raw host-staged calls disagree")

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peak()
    # dominant kernel: the recurrence (strip_sweep_kernel) reads every frame and writes every filtered image and the
    # zeroed label image, i.e. all of the algorithmic bytes; the per-frame kernels and region_variance_kernel only
    # touch the marked groups / component boxes.  `step_*` is the same figure over all launches of a step.
    sweep_ms = float(kt[0]) if kt[0] > 0 else kernel_ms
    achieved = BYTES_PER_FRAME * total / (sweep_ms * 1e-3) / 1e9
    step_achieved = BYTES_PER_FRAME * total / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic(total)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16/int32 (fp32+fp64 scalars)", "data": "synthetic",
        "config": workload_config(C, T),
        "run_info": {"regions_found": regions_total, "step": "clip descriptors are re-uploaded every step (pessimistic, a few kB)"},
        "roofline": {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_source": traffic_src,
            "kernel": "strip_sweep_kernel", "kernel_ms": sweep_ms, "algorithmic_bytes_per_frame": BYTES_PER_FRAME, "peak_source": peak_src,
            "kernel_share_of_step": sweep_ms / kernel_ms,
            "step_ms": kernel_ms, "step_achieved": step_achieved, "step_frac": step_achieved / peak,
            "kernel_times_ms": {"strip_sweep_kernel": float(kt[0]), "frame_scalars_kernel": float(kt[1]),
                                "frame_regions_kernel+frame_components_kernel": float(kt[2]), "denoise_passes": float(kt[3]),
                                "region_variance_kernel": float(kt[4])},
            "kernels_per_step": ["strip_sweep_kernel", "frame_scalars_kernel", "frame_regions_kernel",
                                 "frame_components_kernel (the frames frame_regions_kernel left on its list: nearly always none)",
                                 "region_variance_kernel"],
        },
        "e2e": e2e, "gpu_launches": 5 * args.steps, "clocks": clocks.summary(),
    }
    line.update(extras)
    if world > 1:
        line["run_info"]["numa_node_of_rank0"] = numa  # every rank runs on the cores of its GPU's NUMA node (bind_to_gpu_node)
    if preprocess is not None:
        line["preprocess"] = preprocess
    if not args.no_motion:
        line["motion_detector"] = bench_motion()
    if preprocess is not None:
        # the metric's name: frames tracked AND preprocessed -- one extraction pass plus one preprocessing pass over the batch
        line["tracked_and_preprocessed"] = {
            "frames_per_s": total / ((kernel_ms + preprocess["ms"]) * 1e-3), "unit": UNIT,
            "what": "frames of the batch / (extraction step + preprocessing of {} segments drawn from it)".format(args.tracks)}
    if not args.no_cpu_baseline and world >= 1:
        cores = min(os.cpu_count() or 1, 64)
        n_cpu = min(8 * cores, e2e_clips)  # ~10 s of CPU work: 8 whole clips per host thread
        sample = np.ascontiguousarray(h_frames.reshape(e2e_clips, T, H, W)[:n_cpu])
        v, dt, n_clips, port = cpu_baseline(cores, 1, T, pix=sample, want_regions=True)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "first {} clips x {} frames of this run's batch, {:.1f} s".format(n_clips, sample.shape[1], dt),
                                "reference_python": reference_python_record()}
        # parity of THIS run: the e2e region lists of the GPU against the CPU port's on the clips both processed
        line["parity_checked_clips"] = n_clips
        line["parity_checked_regions"] = check_parity(hout, port, n_clips, T)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
