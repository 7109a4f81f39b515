"""CPTVMotionDetector.process_frames / process_clips (one cpt_motion_clips launch for whole recordings of many
detectors) against the reference fixtures, the numpy oracle and the per-frame process_frame loop: per-frame rows, the
host state and the device state (frame ring, running sum and count, delta ring, background record) bit for bit."""
import ctypes

import numpy as np
import pytest

from tests import motion_helpers as mh

pytestmark = pytest.mark.gpu

FPS = 9


class ListWindow(mh.Window):
    """Recording window answering inside_window() from a per-frame list; counts the calls."""

    def __init__(self, inside):
        super().__init__()
        self.flags = list(inside)
        self.calls = 0

    def inside_window(self):
        v = self.flags[self.calls]
        self.calls += 1
        return v


def detector(model, preview_secs=5, detect_after=None, inside=(), res=(160, 120), **overrides):
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import CPTVMotionDetector

    CPTVMotionDetector.BACKGROUND_WEIGHT_ADD = 0.1  # a lepton3.5 detector sets 1 in its constructor
    cfg = mh.thermal_config(model, preview_secs, **overrides)
    cfg.recorder.rec_window = ListWindow(inside)
    return CPTVMotionDetector(cfg, None, mh.Headers(model, res_x=res[0], res_y=res[1], fps=FPS), detect_after=detect_after)


class _MotionHead(ctypes.Structure):
    # the leading members of struct cpt_motion (csrc/motion_kernels.cu): where the handle keeps its device buffers
    _fields_ = [("ctx", ctypes.c_void_p), ("ring_frames", ctypes.c_int), ("mean_frames", ctypes.c_int),
                ("diff_frames", ctypes.c_int), ("weight_slot", ctypes.c_int), ("d_ring", ctypes.c_void_p),
                ("d_sum", ctypes.c_void_p), ("d_diff", ctypes.c_void_p), ("d_mean_count", ctypes.c_void_p)]


def device_state(det):
    from classifier_pipeline_b200 import native

    h = _MotionHead.from_address(det._m)
    ctx, H, W, e = det._ctx, det.res_y, det.res_x, det.config.edge_pixels
    out = dict(ring=np.empty((h.ring_frames, H, W), np.uint16), sum=np.empty((H, W), np.uint32), count=np.empty(1, np.int32),
               diff=np.empty((h.diff_frames, (H - 2 * e) * (W - 2 * e)), np.float64))
    for key, ptr in (("ring", h.d_ring), ("sum", h.d_sum), ("count", h.d_mean_count), ("diff", h.d_diff)):
        if out[key].size:
            native.check(ctx.lib.cpt_copy_to_host(ctx._h, out[key].ctypes.data, ptr, out[key].nbytes))
    ctx.synchronize()
    out["state"] = det._background.d_state.cpu().numpy()
    return out


def host_state(det):
    win = det.thermal_window
    s = dict(cursors=(win.last_index, win.oldest_index, win.non_ffc_index, win.ffc), processed=det.processed,
             num_frames=det.num_frames, triggered=det.triggered, moved=det.movement_detected, ffc=det.ffc_affected,
             last_diff=det.last_diff, mean=det.running_mean, frames=[id(f) for f in win.frames])
    if not det.config.one_diff_only:
        dw = det.diff_window
        s["diff_cursors"] = (dw.last_index, dw.oldest_index, dw.non_ffc_index, dw.ffc)
    return s


def assert_same(a, b):
    """Two detectors fed the same frames are in the same state, host and device."""
    assert host_state(a) == host_state(b)
    assert all(x is y for x, y in zip(a.preview_frames(), b.preview_frames()))
    assert len(a.preview_frames()) == len(b.preview_frames())
    assert a.get_recent_frame() is b.get_recent_frame()
    da, db = device_state(a), device_state(b)
    for k in da:
        assert np.array_equal(da[k], db[k]), k


def stream(det, frames):
    rows = []
    for f in frames:
        det.process_frame(f)
        rows.append((det.movement_detected, det.triggered, float(det.temp_thresh), det.processed, det.last_diff))
    return np.array(rows, dtype=np.float64).reshape(-1, 5)


def trace_rows(tr):
    return np.stack([tr.movement_detected, tr.triggered, tr.temp_thresh, tr.processed, tr.diff], 1).astype(np.float64)


# ---------------------------------------------------------------- 1. reference fixtures
def fixture_run(name):
    source, model, overrides, preview_secs, detect_after, ffc_frames, outside = mh.CASES[name]
    pix = mh.frames_for(source)
    det = detector(model, preview_secs, detect_after, [t not in outside for t in range(len(pix))], **overrides)
    return det, [mh.StreamFrame(p, t, ffc=t in ffc_frames) for t, p in enumerate(pix)]


def check_fixture(name, det, tr):
    d, _ = mh.load_fixture(name)
    assert det.rec_window.calls == len(tr.processed)
    assert np.array_equal(trace_rows(tr)[:, :4], d["rows"])
    assert np.array_equal(det.background, d["background"])
    assert np.array_equal(det._background.background_weight, d["background_weight"])


@pytest.mark.parametrize("name", list(mh.CASES))
def test_fixture_in_one_call(name):
    det, frames = fixture_run(name)
    check_fixture(name, det, det.process_frames(frames))


def test_fixtures_as_four_detectors_in_one_call():
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import process_clips

    runs = [fixture_run(name) for name in mh.CASES]
    traces = process_clips([r[0] for r in runs], [r[1] for r in runs])
    for name, (det, _), tr in zip(mh.CASES, runs, traces):
        check_fixture(name, det, tr)


# ---------------------------------------------------------------- 2. randomised against the oracle and the loop
def runs(rng, n, p_start, max_len):
    """Frame indices of random runs (lengths 1..max_len), the first one at frame 0 with probability p_start."""
    out, t = set(), 0 if rng.random() < p_start else int(rng.integers(1, max(2, n)))
    while t < n:
        k = int(rng.integers(1, max_len + 1))
        out.update(range(t, min(n, t + k)))
        t += k + int(rng.integers(5, 80))
    return out


def random_case(k):
    from classifier_pipeline_b200.synthetic import make_clip

    rng = np.random.default_rng(1000 + k)
    n = [1, 2, 7, 15, 30, 60, 95, 140, 230, 380][k % 10]
    pix, model = make_clip(k, frames=n)
    overrides = dict(one_diff_only=bool(k & 2), warmer_only=bool(k & 4), frame_compare_gap=int(rng.choice([2, 8, 45])),
                     delta_thresh=int(rng.choice([20, 50, 150])), count_thresh=int(rng.choice([1, 3, 10])))
    preview_secs = int(rng.choice([0, 1, 2, 5, 6]))  # rings of 1, 10, 19, 46 and 55 frames
    detect_after = [None, 0, 3, 40][(k >> 3) % 4]
    ffc = runs(rng, n, 0.3, 3)
    outside = runs(rng, n, 0.5, 6) - ffc if k % 3 else set()
    if not overrides["one_diff_only"]:
        # the oracle reads the delta ring's oldest entry from the fourth processed frame on, so its first entry must be
        # stored by then: detection from the second processed frame, no FFC or recording gap before it
        detect_after = 0
        ffc = {t for t in ffc if t >= 6}
        outside = {t for t in outside if t >= 6}
    return pix, model, overrides, preview_secs, detect_after, ffc, outside


def test_random_detectors_match_oracle_and_loop():
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import process_clips
    from oracle.motion_oracle import run_motion

    batch, twins, frame_lists, expected = [], [], [], []
    for k in range(72):
        pix, model, overrides, preview_secs, detect_after, ffc, outside = random_case(k)
        inside = [t not in outside for t in range(len(pix))]
        batch.append(detector(model, preview_secs, detect_after, inside, **overrides))
        twins.append(detector(model, preview_secs, detect_after, inside, **overrides))
        frames = [mh.StreamFrame(p, t, ffc=t in ffc) for t, p in enumerate(pix)]
        frame_lists.append(frames)
        m = dict(mh.MOTION_DEFAULTS[model], **overrides)
        expected.append(run_motion(pix, 1.0 if model == "lepton3.5" else 0.1, m["temp_thresh"], m["delta_thresh"],
                                   m["count_thresh"], m["trigger_frames"], m["edge_pixels"], m["warmer_only"],
                                   m["one_diff_only"], m["frame_compare_gap"], preview_secs * FPS, detect_after, ffc, outside))
    traces = process_clips(batch, frame_lists)
    for k, (det, twin, frames, tr, (rows, st)) in enumerate(zip(batch, twins, frame_lists, traces, expected)):
        got = trace_rows(tr)
        assert np.array_equal(got[:, :4], rows), k
        assert np.array_equal(got, stream(twin, frames)), k
        assert det.rec_window.calls == len(frames)
        assert_same(det, twin)
        if st["background"] is not None:
            assert np.array_equal(det.background, st["background"]), k
            assert np.array_equal(det._background.background_weight, st["weight"]), k
        if st["running_sum"] is not None:
            dev = device_state(det)
            assert np.array_equal(dev["sum"], st["running_sum"]), k
            assert int(dev["count"][0]) == st["running_frames"], k


# ---------------------------------------------------------------- 3. continuation both ways
CONT_OUTSIDE = set(range(0, 4)) | set(range(50, 56))
CONT_FFC = {20, 21, 22, 70}


@pytest.mark.parametrize("preview_secs,k", [
    (2, 2),    # inside the leading outside-window run, before the mean starts
    (2, 5),    # after the mean started, before the ring of 19 fills
    (2, 21),   # inside an FFC run
    (2, 30),   # after the ring filled
    (2, 52),   # inside an outside-window run
    (5, 40),   # before the ring of 46 fills
    (5, 60),   # after it filled
])
@pytest.mark.parametrize("batch_first", [True, False])
def test_continuation(preview_secs, k, batch_first):
    from classifier_pipeline_b200.synthetic import make_clip

    pix, _ = make_clip(4, frames=120)
    frames = [mh.StreamFrame(p, t, ffc=t in CONT_FFC) for t, p in enumerate(pix)]
    inside = [t not in CONT_OUTSIDE for t in range(len(pix))]
    opts = dict(one_diff_only=False, warmer_only=False, frame_compare_gap=8, delta_thresh=30)
    ref = detector("lepton3", preview_secs, 5, inside, **opts)
    det = detector("lepton3", preview_secs, 5, inside, **opts)
    want = stream(ref, frames)
    if batch_first:
        got = np.concatenate([trace_rows(det.process_frames(frames[:k])), stream(det, frames[k:])])
    else:
        got = np.concatenate([stream(det, frames[:k]), trace_rows(det.process_frames(frames[k:]))])
    assert np.array_equal(got, want)
    assert_same(det, ref)


# ---------------------------------------------------------------- 4. edges
def test_empty_list():
    pix, _ = make_frames(30)
    det, ref = detector("lepton3", 2, 0, [True] * 30), detector("lepton3", 2, 0, [True] * 30)
    tr = det.process_frames([])
    assert all(len(a) == 0 for a in tr)
    assert_same(det, ref)
    assert np.array_equal(stream(det, pix), stream(ref, pix))
    assert_same(det, ref)


def test_all_outside_then_streaming():
    frames, _ = make_frames(40)
    inside = [False] * 12 + [True] * 28
    det, ref = detector("lepton3", 2, 0, inside), detector("lepton3", 2, 0, inside)
    tr = det.process_frames(frames[:12])
    assert not tr.movement_detected.any() and not tr.processed.any()
    assert np.array_equal(np.concatenate([trace_rows(tr), stream(det, frames[12:])]), stream(ref, frames))
    assert_same(det, ref)


def test_one_frame():
    frames, _ = make_frames(20)
    det, ref = detector("lepton3", 2, 0, [True] * 20), detector("lepton3", 2, 0, [True] * 20)
    assert np.array_equal(trace_rows(det.process_frames(frames[:1])), stream(ref, frames[:1]))
    assert_same(det, ref)
    assert np.array_equal(stream(det, frames[1:]), stream(ref, frames[1:]))
    assert_same(det, ref)


def make_frames(n, index=6):
    from classifier_pipeline_b200.synthetic import make_clip

    pix, model = make_clip(index, frames=n)
    return [mh.StreamFrame(p, t) for t, p in enumerate(pix)], model


# ---------------------------------------------------------------- 5. rejections
@pytest.mark.parametrize("bad", ["dtype", "shape"])
def test_bad_frame_changes_nothing(bad):
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import process_clips

    frames, _ = make_frames(30)
    det, other, ref, ref_other = (detector("lepton3", 2, 0, [True] * 30) for _ in range(4))
    broken = list(frames[:10])
    p = frames[5].pix
    broken[5] = mh.StreamFrame(p.astype(np.float32) if bad == "dtype" else p[:, :-8].copy(), 5)
    with pytest.raises(TypeError if bad == "dtype" else ValueError):
        process_clips([other, det], [frames[:10], broken])
    for a, b in ((det, ref), (other, ref_other)):
        assert a.rec_window.calls == 0
        assert_same(a, b)
        assert np.array_equal(stream(a, frames), stream(b, frames))


def test_mixed_geometry_rejected():
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import process_clips

    frames, _ = make_frames(20)
    small = [mh.StreamFrame(f.pix[:64, :80].copy(), t) for t, f in enumerate(frames)]
    det, ref = detector("lepton3", 2, 0, [True] * 20), detector("lepton3", 2, 0, [True] * 20)
    other = detector("lepton3", 2, 0, [True] * 20, res=(80, 64))
    with pytest.raises(ValueError):
        process_clips([det, other], [frames, small])
    assert det.rec_window.calls == 0 and other.rec_window.calls == 0
    assert np.array_equal(stream(det, frames), stream(ref, frames))
    assert_same(det, ref)


def test_out_of_range_indices_rejected():
    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.piclassifier.cptvmotiondetector import plan_clips

    frames, _ = make_frames(60)
    inside = [False, False] + [True] * 58
    det = detector("lepton3", 2, 0, inside, one_diff_only=False, frame_compare_gap=8)
    steps = plan_clips([det], [frames])
    ring, diff_frames = det.thermal_window.size, det.diff_window.size
    staged = np.stack([f.pix for f in frames])
    d_frames = torch.from_numpy(staged.view(np.int16)).to(det._background.engine.device)
    ctx, lib = det._ctx, det._ctx.lib
    before = device_state(det)

    def call():
        return lib.cpt_motion_clips(ctx._h, steps._clips, 1, d_frames.data_ptr(), steps.n_frames, steps._steps, steps.n_steps,
                                    steps._mean_rows.ctypes.data, len(steps._mean_rows), steps.results)

    detect = next(i for i in range(steps.n_steps) if steps._steps[i].flags & native.MOTION_DETECT)
    mean = next(i for i in range(steps.n_steps) if steps._steps[i].mean_count)
    cases = [
        (steps._steps[0], "frame", len(frames)),       # a row past the staged frames
        (steps._steps[1], "oldest", -1 - ring),        # a ring slot past the ring
        (steps._steps[detect], "nonffc", len(frames)),
        (steps._steps[detect], "diff_slot_new", diff_frames),
        (steps._steps[detect], "diff_slot_old", diff_frames),
        (steps._steps[mean], "mean_count", 46),        # more than RunningMean's 45 frames
        (steps._steps[mean], "mean_first", len(steps._mean_rows)),
        (steps._clips[0], "n_steps", steps.n_steps + 1),
        (steps._clips[0], "first_step", -1),
    ]
    for obj, field, value in cases:
        keep = getattr(obj, field)
        setattr(obj, field, value)
        assert call() == -1, field  # CPT_ERR_INVALID
        setattr(obj, field, keep)
    for table in (steps._mean_rows, steps._ring_rows[0]):  # a mean row, then a ring row, past the staged frames
        keep = int(table[0])
        table[0] = len(frames)
        assert call() == -1
        table[0] = keep
    after = device_state(det)
    for key in before:
        assert np.array_equal(before[key], after[key]), key
    assert call() == 0
