"""IRMotionDetector.process_frames / process_clips (cpt_ir_motion_clips: whole recordings of many detectors with each
frame's trigger decided on the device) against tests/golden/ir.npz, the process_frame loop with MOG2Background (trace, host
state and device state: grey ring and MOG2 state bytes) and the loop with CVBackground (cv2 on the host), plus the
bit-parallel erosion against cv2.erode through the per-frame call and through the new call."""
import ctypes
import os

import numpy as np
import pytest

from tests import helpers, ir_helpers
from tests import ir_clip_scenes as sc

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


class ListWindow(ir_helpers._Window):
    """Recording window answering inside_window() from a per-frame list (then True)."""

    def __init__(self, inside=()):
        self.flags = list(inside)
        self.calls = 0

    def inside_window(self):
        v = self.flags[self.calls] if self.calls < len(self.flags) else True
        self.calls += 1
        return v


def detector(shape=(120, 160), ring=10, background="mog2", history=1000, var_threshold=16, inside=()):
    from classifier_pipeline_b200.piclassifier.irmotiondetector import IRMotionDetector
    from classifier_pipeline_b200.track.cliptracker import CVBackground, MOG2Background

    cfg, headers = ir_helpers.ir_config()
    cfg.recorder.rec_window = ListWindow(inside)
    cfg.recorder.preview_secs = 1
    headers.fps, headers.res_y, headers.res_x = ring, shape[0], shape[1]
    bg = MOG2Background(history=history, var_threshold=var_threshold) if background == "mog2" else CVBackground()
    if background == "cv" and (history, var_threshold) != (1000, 16):
        bg.algorithm = cv2.createBackgroundSubtractorMOG2(history=history, varThreshold=var_threshold, detectShadows=False)
    return IRMotionDetector(cfg, headers, background=bg)


def loop(det, frames, force=False):
    """The process_frame loop; rows (movement, triggered, diff, mask) as IrMotionTrace has them."""
    counts = []
    apply = det._apply

    def record(step, diff, mask):
        counts.append((diff, mask) if step is not None and step.detect else (-1, -1))
        apply(step, diff, mask)

    det._apply = record
    rows = []
    try:
        for f in frames:
            moved = det.process_frame(f, force)
            rows.append((moved, det.triggered) + counts[-1])
    finally:
        del det._apply
    return np.array(rows, dtype=np.int64).reshape(-1, 4)


def rows(tr):
    return np.stack([tr.movement_detected, tr.triggered, tr.diff_pixels, tr.mask_pixels], 1).astype(np.int64).reshape(-1, 4)


class _Mog2Head(ctypes.Structure):
    # the leading members of struct cpt_mog2 (csrc/mog2.cuh)
    _fields_ = [("ctx", ctypes.c_void_p), ("W", ctypes.c_int), ("H", ctypes.c_int), ("npx", ctypes.c_int64), ("history", ctypes.c_int),
                ("complexity_reduction", ctypes.c_float), ("c", ctypes.c_float * 6), ("nframes", ctypes.c_int),
                ("d_state", ctypes.c_void_p)]


def device_state(det):
    from classifier_pipeline_b200 import native

    ctx, dev = det._dev.ctx, det._dev
    ring = np.empty((dev.ring_frames, dev.height, dev.width), np.uint8)
    for s in range(dev.ring_frames):
        native.check(ctx.lib.cpt_copy_to_host(ctx._h, ring[s].ctypes.data, dev.ring_slot(s), ring[s].nbytes))
    out = dict(ring=ring)
    model = det._background._model
    if model is not None:
        h = _Mog2Head.from_address(model.address)
        state = np.empty(h.npx * 61, np.uint8)
        native.check(ctx.lib.cpt_copy_to_host(ctx._h, state.ctypes.data, h.d_state, state.nbytes))
        out.update(state=state, nframes=np.array([model.frames]), background=det.background,
                   mask=det._background.device_mask.cpu().numpy(), filtered=det._background.compute_filtered(None))
    ctx.synchronize()
    return out


def host_state(det):
    rw, gw = det.rgb_window, det.gray_window
    return dict(rgb=(rw.last_index, rw.oldest_index), gray=(gw.last_index, gw.oldest_index), num_frames=det.num_frames,
                moved=det.movement_detected, triggered=det.triggered, prev=det.prev_triggered, bg_frames=det._background._frames)


def _host(f):
    return None if f is None else np.asarray(f.cpu() if hasattr(f, "cpu") else f)


def assert_same(a, b):
    assert host_state(a) == host_state(b)
    fa, fb = a.rgb_window.frames, b.rgb_window.frames
    assert len(fa) == len(fb) and all((x is None) == (y is None) for x, y in zip(fa, fb))
    assert all(np.array_equal(_host(x), _host(y)) for x, y in zip(fa, fb) if x is not None)
    da, db = device_state(a), device_state(b)
    assert da.keys() == db.keys()
    for k in da:
        assert np.array_equal(da[k], db[k]), k


# ---------------------------------------------------------------- golden and designed scenes
def test_golden_trace_in_one_call():
    gold = np.load(os.path.join(helpers.GOLDEN, "ir.npz"))
    det = detector(shape=(ir_helpers.H, ir_helpers.W))
    tr = det.process_frames(ir_helpers.ir_video(3))
    assert np.array_equal(tr.movement_detected, gold["motion_flags"])
    assert np.array_equal(tr.triggered, gold["motion_triggered"])


@pytest.mark.parametrize("name", list(sc.DESIGNS))
def test_designed_scene_against_loop_and_cv2(name):
    frames = sc.design(name)
    batch, ref, cvd = detector(), detector(), detector(background="cv")
    want = loop(ref, frames)
    sc.check_design(name, want)
    assert np.array_equal(loop(cvd, frames), want)
    assert np.array_equal(sc.cv2_trace(frames), want)
    assert np.array_equal(rows(batch.process_frames(frames)), want)
    assert_same(batch, ref)


@pytest.mark.parametrize("shape", [(480, 640), (120, 160), (61, 97)], ids=lambda s: "{}x{}".format(s[1], s[0]))
def test_geometries_against_loop_and_cv2(shape):
    frames = sc.scene(7, 150, shape, boxes=[(104, 140, min(shape) // 3, 4)])
    batch, ref = detector(shape), detector(shape)
    want = loop(ref, frames)
    assert want[:, 0].any()
    assert np.array_equal(sc.cv2_trace(frames), want)
    assert np.array_equal(rows(batch.process_frames(frames)), want)
    assert_same(batch, ref)


# ---------------------------------------------------------------- many clips in one call
def test_many_clips_in_one_call():
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    rng = np.random.default_rng(21)
    rings = [1, 2, 10, 50, 1, 2, 10, 50, 10, 3, 7, 10]
    batch, ref, lists = [], [], []
    for i, ring in enumerate(rings):
        n = int(rng.integers(1, 230))
        inside = [bool(v) for v in rng.random(n) > (0.3 if i % 3 == 0 else 0.0)]
        hist, vt = [(1000, 16), (50, 16), (1000, 9), (7, 25)][i % 4]
        frames = sc.scene(100 + i, n, (61, 97), boxes=[(int(rng.integers(90, 140)), 200, 20, int(rng.integers(1, 6)))])
        a = detector((61, 97), ring, history=hist, var_threshold=vt, inside=inside * 2)
        b = detector((61, 97), ring, history=hist, var_threshold=vt, inside=inside * 2)
        if i == 5:  # one detector after disconnected(), with frames streamed before
            for d in (a, b):
                loop(d, frames[:40])
                d.disconnected()
                d.rec_window.calls = 0
        batch.append(a), ref.append(b), lists.append(frames)
    want = [loop(d, f) for d, f in zip(ref, lists)]
    assert any(w[:, 0].any() for w in want) and any((w[:, 2] == -1).any() for w in want)
    for d, w, f in zip(ref, want, lists):
        assert np.array_equal(sc.cv2_trace(f, ring=d._dev.ring_frames, history=d._background.history,
                                           var_threshold=d._background.var_threshold, inside=d.rec_window.flags[: len(f)]), w) or d is ref[5]
    traces = process_clips(batch, lists)
    for a, b, tr, w in zip(batch, ref, traces, want):
        assert np.array_equal(rows(tr), w)
        assert_same(a, b)


def test_force_process_and_outside_frames():
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    frames = sc.design("saturate")
    inside = [t % 7 != 3 for t in range(len(frames))]
    a, b = detector(inside=inside), detector(inside=inside)
    c, d = detector(inside=[False] * len(frames)), detector(inside=[False] * len(frames))
    want_ab, want_cd = loop(b, frames), loop(d, frames, force=True)
    assert (want_ab[:, 2] == -1).sum() > 101
    ta, tc = process_clips([a], [frames])[0], process_clips([c], [frames], force_process=True)[0]
    assert np.array_equal(rows(ta), want_ab) and np.array_equal(rows(tc), want_cd)
    assert_same(a, b)
    assert_same(c, d)


# ---------------------------------------------------------------- continuation
@pytest.mark.parametrize("cut", [1, 9, 10, 11, 100, 101, 102, 112, 140, 199])
def test_continuation_both_ways(cut):
    """Batch then loop and loop then batch, cut at a ring wrap (ring 10), at the MIN_FRAMES boundary and mid-recording."""
    frames = sc.design("saturate")
    ref, a, b = detector(), detector(), detector()
    want = loop(ref, frames)
    got_a = np.concatenate([rows(a.process_frames(frames[:cut])), loop(a, frames[cut:])])
    got_b = np.concatenate([loop(b, frames[:cut]), rows(b.process_frames(frames[cut:]))])
    assert np.array_equal(got_a, want) and np.array_equal(got_b, want)
    assert_same(a, ref)
    assert_same(b, ref)
    if 106 < cut < 150:
        assert want[cut - 1, 0]  # the cut is inside a recording


def test_continuation_in_several_calls_and_a_fresh_model():
    frames = sc.design("box_switch")
    ref, a = detector(), detector()
    want = loop(ref, frames)
    cuts = [0, 1, 2, 57, 101, 108, 160, 239, 240]
    got = np.concatenate([rows(a.process_frames(frames[x:y])) for x, y in zip(cuts[:-1], cuts[1:])])
    assert np.array_equal(got, want)
    assert_same(a, ref)


# ---------------------------------------------------------------- edge cases
def test_empty_outside_and_one_frame_lists():
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    assert process_clips([], []) == []
    frames = sc.scene(3, 5, (61, 97))
    a, b, c = detector((61, 97)), detector((61, 97), inside=[False] * 5), detector((61, 97))
    ta, tb, tc = process_clips([a, b, c], [[], frames, frames[:1]])
    assert len(ta.triggered) == 0 and a.num_frames == 0 and a._background._model is None
    assert b.num_frames == 5 and b._background._model is None and np.array_equal(b.rgb_window.current, frames[4])
    assert not tb.movement_detected.any()
    assert (tb.diff_pixels == -1).all()
    ref = detector((61, 97))
    assert np.array_equal(rows(tc), loop(ref, frames[:1]))
    assert_same(c, ref)


def test_host_call_longer_than_one_chunk_and_device_input():
    import torch

    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    n = 310  # a staging chunk holds about 291 frames of 640 x 480
    frames = sc.scene(5, n, (480, 640), boxes=[(104, 300, 80, 7)])
    ref, a, b = detector((480, 640)), detector((480, 640)), detector((480, 640))
    want = loop(ref, frames)
    assert want[:, 0].any()
    ta, tb = process_clips([a], [list(frames)])[0], process_clips([b], [torch.from_numpy(frames).cuda()])[0]
    assert np.array_equal(rows(ta), want) and np.array_equal(rows(tb), want)
    assert_same(a, ref)
    assert_same(b, ref)
    assert b.rgb_window.current.is_cuda and np.array_equal(b.rgb_window.current.cpu().numpy(), frames[-1])


# ---------------------------------------------------------------- erosion against cv2.erode
WIDTHS, HEIGHTS, KS = [1, 31, 32, 33, 63, 64, 65, 97, 640], [1, 61, 480], [1, 2, 10, 15, 31, 32, 33, 64]


def masks(rng, h, w):
    blocks = np.zeros((h, w), np.uint8)
    blocks[h // 4 : h // 4 + max(1, h // 2), w // 5 : w // 5 + max(1, w // 2)] = 255
    blocks[: max(1, h // 5), : max(1, w // 6)] = 255
    return [(rng.random((h, w)) > 0.03).astype(np.uint8) * 255, blocks, np.full((h, w), 255, np.uint8), np.zeros((h, w), np.uint8)]


def cv2_count(mask, k):
    return int((cv2.erode(mask, np.ones((k, k), np.uint8)) > 0).sum())


@pytest.mark.parametrize("h", HEIGHTS)
def test_erosion_counts_match_cv2(h):
    """Per frame (IrMotion.detect) and through cpt_ir_motion_clips (the step's diff count, erode_idle = k): every width, box
    and designed mask."""
    import torch

    from classifier_pipeline_b200 import engine, native

    ctx = engine.get_engine().ctx
    ctx.use_torch_stream()
    rng = np.random.default_rng(h)
    for w in WIDTHS:
        dev = native.IrMotion(ctx, w, h, 2)
        model = native.Mog2(ctx, w, h)
        d_mask = torch.empty((h, w), dtype=torch.uint8, device="cuda")
        zero = np.zeros((h, w, 3), np.uint8)
        dev.gray(zero, 0, copy_out=False)
        for mi, m in enumerate(masks(rng, h, w)):
            bgr = np.repeat(m[:, :, None], 3, 2)  # equal channels: the grey frame is the mask itself
            dev.gray(bgr, 1, copy_out=False)
            for k in KS:
                want = cv2_count(m, k)
                assert dev.detect(1, 0, 12, k, mask=m) == (want, want), (w, h, mi, k)
                # through the new call: zero frame then the mask frame, the second step detects with the box k
                frames = torch.from_numpy(np.stack([zero, bgr])).cuda()
                table = np.array([frames.data_ptr(), frames.data_ptr() + h * w * 3], np.uint64)
                steps = (native.CptIrMotionClipStep * 2)(native.CptIrMotionClipStep(0, 0, 0, 0, 0), native.CptIrMotionClipStep(1, 1, 0, 1, 0))
                clips = (native.CptIrMotionClip * 1)(dev.clip_record(model, d_mask, 0, 2, False, 0))
                res = (native.CptIrMotionClipResult * 2)()
                ctx.ir_motion_clips(clips, 1, table, 2, steps, 2, native.CptIrMotionClipParams(12, 2, 30, k, k, 0), res)
                assert res[0].diff_pixels == -1 and res[1].diff_pixels == want, (w, h, mi, k)


# ---------------------------------------------------------------- rejected input and round trips
def test_rejected_input_changes_nothing():
    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    frames = sc.scene(9, 12, (61, 97))
    a, b = detector((61, 97)), detector((61, 97))
    loop(a, frames[:3]), loop(b, frames[:3])
    bad_dtype = frames[5].astype(np.int16)
    cases = [([a], [[frames[0], bad_dtype]]), ([a], [[frames[0], frames[1][:, :-1]]]), ([a, a], [frames, frames]),
             ([a, detector((120, 160))], [frames, sc.scene(1, 2)]), ([a, detector((61, 97), background="cv")], [frames, frames]),
             ([a], [torch.from_numpy(frames).cuda().float()]), ([a, b], [frames, torch.from_numpy(frames).cuda()])]
    for dets, lists in cases:
        with pytest.raises(ValueError):
            process_clips(dets, lists)
        assert_same(a, b)
    with pytest.raises(ValueError, match="MOG2Background"):
        detector((61, 97), background="cv").process_frames(frames)
    with pytest.raises(ValueError):
        a.process_frame(bad_dtype)
    assert_same(a, b)
    # at the C ABI: every out-of-range index is refused before anything runs, and the context stays usable
    ctx = a._dev.ctx
    d_frames = torch.from_numpy(frames).cuda()
    table = np.array([d_frames.data_ptr() + t * frames[0].nbytes for t in range(len(frames))], np.uint64)
    mask = torch.empty((61, 97), dtype=torch.uint8, device="cuda")
    model = native.Mog2(ctx, 97, 61)
    params = native.CptIrMotionClipParams(12, 2, 30, 15, 10, 0)

    def call(steps, clip_args=(), n_frames=len(table), p=params, n_steps=None):
        st = (native.CptIrMotionClipStep * len(steps))(*[native.CptIrMotionClipStep(*s) for s in steps])
        rec = a._dev.clip_record(model, mask, *(clip_args or (0, len(steps), False, 0)))
        clips = (native.CptIrMotionClip * 1)(rec)
        res = (native.CptIrMotionClipResult * max(1, len(steps)))()
        return ctx.lib.cpt_ir_motion_clips(ctx._h, clips, 1, table.ctypes.data, n_frames, st, len(steps) if n_steps is None else n_steps,
                                           ctypes.byref(p), res)

    ring = a._dev.ring_frames
    assert call([(len(table), 0, 0, 0, 0)]) == -1          # row
    assert call([(-1, 0, 0, 0, 0)]) == -1
    assert call([(0, ring, 0, 0, 0)]) == -1                # slots
    assert call([(0, 0, -1, 0, 0)]) == -1
    assert call([(0, 0, 0, 0, 0)], (0, 2, False, 0)) == -1  # step range
    assert call([(0, 0, 0, 0, 0)], (-1, 1, False, 0)) == -1
    assert call([(0, 0, 0, 1, 0)], p=native.CptIrMotionClipParams(12, 2, 30, 65, 10, 0)) == -1  # erosion size
    assert call([(0, 0, 0, 1, 0)], p=native.CptIrMotionClipParams(12, 2, 30, 15, 0, 0)) == -1
    bad = (native.CptIrMotionClip * 2)(a._dev.clip_record(model, mask, 0, 1, False, 0), b._dev.clip_record(model, mask, 0, 1, False, 0))
    st = (native.CptIrMotionClipStep * 1)(native.CptIrMotionClipStep(0, 0, 0, 0, 0))
    res = (native.CptIrMotionClipResult * 2)()
    assert ctx.lib.cpt_ir_motion_clips(ctx._h, bad, 2, table.ctypes.data, len(table), st, 1, ctypes.byref(params), res) == -1  # shared
    other = native.IrMotion(ctx, 96, 61, 3)
    bad = (native.CptIrMotionClip * 1)(other.clip_record(model, mask, 0, 1, False, 0))
    assert ctx.lib.cpt_ir_motion_clips(ctx._h, bad, 1, table.ctypes.data, len(table), st, 1, ctypes.byref(params), res) == -1  # geometry
    bad[0].m = None
    assert ctx.lib.cpt_ir_motion_clips(ctx._h, bad, 1, table.ctypes.data, len(table), st, 1, ctypes.byref(params), res) == -1  # handle
    assert model.frames == 0
    assert_same(a, b)
    # the context still works: the detectors continue, and agree with each other and with cv2
    tr = a.process_frames(frames[3:])
    assert np.array_equal(rows(tr), loop(b, frames[3:]))
    assert_same(a, b)


def test_no_per_frame_round_trips(monkeypatch):
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.piclassifier.irmotiondetector import process_clips

    frames = sc.design("trigger")
    ref = [detector(), detector(ring=3)]
    want = [loop(d, frames) for d in ref]
    dets = [detector(), detector(ring=3)]

    def fail(*a, **k):
        raise AssertionError("a per-frame native call")

    calls = []
    clips = native.Context.ir_motion_clips

    def counted(self, *a):
        calls.append(1)
        return clips(self, *a)

    for name in ("gray", "detect", "step"):
        monkeypatch.setattr(native.IrMotion, name, fail)
    monkeypatch.setattr(native.Mog2, "apply", fail)
    monkeypatch.setattr(native.Context, "ir_motion_clips", counted)
    traces = process_clips(dets, [frames, frames])
    assert len(calls) == 1
    for tr, w in zip(traces, want):
        assert np.array_equal(rows(tr), w)
