"""OpenCV's MOG2 on the device (csrc/mog2_kernels.cu, native.Mog2, track.cliptracker.MOG2Background) against live
cv2.createBackgroundSubtractorMOG2(detectShadows=False): every foreground mask and getBackgroundImage() are equal
(np.array_equal), over designed scenes that reach every branch of the update (checked on the C restatement,
oracle/mog2_oracle.c), learning-rate schedules, geometries with a partial last CTA, and any split of a sequence into launches.
Also the IR motion detector with the device model against the trace tests/golden/ir.npz pins."""
import ctypes
import os

import numpy as np
import pytest

from tests import helpers, ir_helpers
from tests import mog2_helpers as mh

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

SHAPES = [(480, 640), (120, 160), (61, 97)]


@pytest.fixture(scope="module")
def ctx():
    from classifier_pipeline_b200 import engine

    return engine.get_engine().ctx


class Device:
    """native.Mog2 with cv2's surface, one frame per call unless told otherwise."""

    def __init__(self, ctx, shape, history):
        import torch

        from classifier_pipeline_b200 import native

        ctx.use_torch_stream()
        self.h, self.w = shape
        self.m = native.Mog2(ctx, self.w, self.h, history=history)
        self.out = torch.empty(shape, dtype=torch.uint8, device="cuda")

    def apply_many(self, frames, lrs):
        import torch

        d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
        masks = torch.empty_like(d)
        self.m.apply(d, lrs, d_masks=masks)
        return masks.cpu().numpy()

    def apply(self, frame, lr):
        return self.apply_many(frame[None], [lr])[0]

    def background(self):
        self.m.background(self.out)
        return self.out.cpu().numpy()


def compare(ctx, frames, lrs, history, bg_every=1):
    from oracle.mog2_oracle import Mog2Oracle

    cvm = cv2.createBackgroundSubtractorMOG2(history=history, detectShadows=False)
    dev = Device(ctx, frames.shape[1:], history)
    orc = Mog2Oracle(frames.shape[1:], history=history)
    for t, (f, lr) in enumerate(zip(frames, lrs)):
        a = cvm.apply(f, None, lr)
        b = dev.apply(f, lr)
        orc.apply(f, lr)
        assert np.array_equal(a, b), "mask of frame {} (lr {}): {} pixels differ".format(t, lr, int((a != b).sum()))
        if t % bg_every == 0 or t == len(frames) - 1:
            assert np.array_equal(cvm.getBackgroundImage(), dev.background()), "background after frame {}".format(t)
    assert dev.m.frames == orc.nframes
    return orc


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "{}x{}".format(s[1], s[0]))
@pytest.mark.parametrize("history", [1000, 4])
@pytest.mark.parametrize("name", mh.SCENES)
def test_designed_scenes_equal_cv2(ctx, shape, history, name):
    frames = mh.scene(name, shape, 60, seed=11)
    orc = compare(ctx, frames, mh.scene_rates(name, len(frames)), history, bg_every=1 if shape[0] < 200 else 4)
    for branch in mh.BRANCHES[name]:
        assert orc.stat(branch) > 0, (name, branch, orc.stats.tolist())


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "{}x{}".format(s[1], s[0]))
@pytest.mark.parametrize("sched", mh.SCHEDULES)
def test_learning_rate_schedules_equal_cv2(ctx, shape, sched):
    frames = mh.scene("mixed", shape, 50, seed=12)
    for history in (1000, 3):
        compare(ctx, frames, mh.schedule(sched, len(frames)), history, bg_every=1 if shape[0] < 200 else 5)


@pytest.mark.parametrize("history", [1000, 5])
def test_long_sequence_one_launch_equals_cv2(ctx, history):
    """300 frames (two launches of at most 256) through one call, and re-initialisations inside it."""
    frames = np.concatenate([mh.scene("walk", (61, 97), 150, seed=13), mh.scene("mixed", (61, 97), 150, seed=14)])
    lrs = [1.0 if t in (0, 200) else (0.0 if 120 <= t < 140 else -1.0) for t in range(len(frames))]
    cvm = cv2.createBackgroundSubtractorMOG2(history=history, detectShadows=False)
    want = np.stack([cvm.apply(f, None, lr) for f, lr in zip(frames, lrs)])
    dev = Device(ctx, frames.shape[1:], history)
    assert np.array_equal(dev.apply_many(frames, lrs), want)
    assert np.array_equal(dev.background(), cvm.getBackgroundImage())
    assert dev.m.frames == len(frames) - 200


def test_chunking_gives_the_same_masks_and_state(ctx):
    """One T-frame call, T single-frame calls and calls split at arbitrary points give the same masks, and the same model
    afterwards (background image and the masks of the frames that follow)."""
    frames = mh.scene("mixed", (61, 97), 280, seed=15)
    lrs = mh.schedule("reinit", 270) + [-1.0] * 10
    head, tail = frames[:270], frames[270:]
    runs = []
    for cuts in ([0, 270], list(range(271)), [0, 1, 2, 9, 17, 18, 100, 255, 256, 257, 269, 270]):
        dev = Device(ctx, frames.shape[1:], 1000)
        masks = np.concatenate([dev.apply_many(head[a:b], lrs[a:b]) for a, b in zip(cuts[:-1], cuts[1:])])
        runs.append((masks, dev.background(), dev.apply_many(tail, lrs[270:]), dev.m.frames))
    for other in runs[1:]:
        for x, y in zip(runs[0], other):
            assert np.array_equal(x, y)


def test_mog2_background_surface_equals_cv_background():
    """MOG2Background against CVBackground: masks (host copy and device), background, set_background, update_backgrounds."""
    import torch

    from classifier_pipeline_b200.track.cliptracker import CVBackground, MOG2Background

    frames = mh.scene("walk", (120, 160), 30, seed=16)
    ref, dev = CVBackground(), MOG2Background()
    ref.set_background(frames[0])
    dev.set_background(frames[0])
    for t, f in enumerate(frames[1:20]):
        lr = 0 if 8 <= t < 12 else -1
        ref.update_background(f, learning_rate=lr)
        dev.update_background(torch.from_numpy(f).cuda() if t % 2 else f, learning_rate=lr)
        assert np.array_equal(ref.compute_filtered(None), dev.compute_filtered(None))
        assert np.array_equal(ref.compute_filtered(None), dev.device_mask.cpu().numpy())
        assert np.array_equal(ref.background, dev.background)
    want = np.stack([ref.algorithm.apply(f, None, -1) for f in frames[20:]])
    assert np.array_equal(dev.update_backgrounds(frames[20:25]), want[:5])
    got = dev.update_backgrounds(torch.from_numpy(frames[25:]).cuda())
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), want[5:])
    assert np.array_equal(ref.background, dev.background) and dev.frames == 30


def test_ir_motion_detector_with_device_mog2(monkeypatch):
    """IRMotionDetector(background=MOG2Background()) reproduces the motion flags and trigger counts of the cv2 trace in
    tests/golden/ir.npz, with neither the grey frame nor the mask crossing to the host: one device step per frame."""
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.piclassifier.irmotiondetector import IRMotionDetector
    from classifier_pipeline_b200.track.cliptracker import MOG2Background

    gold = np.load(os.path.join(helpers.GOLDEN, "ir.npz"))
    step = native.IrMotion.step
    calls = {"step": 0}

    def counted_step(self, *a):
        calls["step"] += 1
        return step(self, *a)

    def no_host_copy(self, *a, **k):
        raise AssertionError("the grey frame or the foreground mask was copied to the host")

    monkeypatch.setattr(native.IrMotion, "step", counted_step)
    monkeypatch.setattr(native.IrMotion, "gray", no_host_copy)
    monkeypatch.setattr(native.IrMotion, "detect", no_host_copy)
    monkeypatch.setattr(MOG2Background, "compute_filtered", no_host_copy)
    cfg, headers = ir_helpers.ir_config()
    det = IRMotionDetector(cfg, headers, background=MOG2Background())
    flags, trig = [], []
    for f in ir_helpers.ir_video(3):
        flags.append(bool(det.process_frame(f)))
        trig.append(det.triggered)
    assert np.array_equal(np.array(flags), gold["motion_flags"])
    assert np.array_equal(np.array(trig), gold["motion_triggered"])
    assert calls["step"] == len(flags)


def test_invalid_arguments_leave_the_context_usable(ctx):
    import torch

    from classifier_pipeline_b200 import native

    lib = ctx.lib
    p = native.CptMog2Params(500, 16.0, 0.9, 9.0, 15.0, 4.0, 75.0, 0.05, 1)
    assert not lib.cpt_mog2_open(ctx._h, 97, 61, ctypes.byref(p))  # detect_shadows
    assert b"shadow" in lib.cpt_last_error()
    p.detect_shadows = 0
    assert not lib.cpt_mog2_open(ctx._h, 0, 61, ctypes.byref(p))  # geometry
    assert not lib.cpt_mog2_open(ctx._h, 97, 61, None)
    with pytest.raises(native.NativeError):
        native.Mog2(ctx, 97, 61, detect_shadows=True)
    m = native.Mog2(ctx, 97, 61)
    frames = torch.zeros((2, 61, 97), dtype=torch.uint8, device="cuda")
    lrs = np.full(2, -1.0)
    assert lib.cpt_mog2_apply(m._h, frames.data_ptr(), 2, 97 * 61 - 1, lrs.ctypes.data, None) == -1  # frames overlap: wrong size
    assert lib.cpt_mog2_apply(m._h, None, 1, 97 * 61, lrs.ctypes.data, None) == -1
    assert lib.cpt_mog2_apply(m._h, frames.data_ptr(), 1, 97 * 61, None, None) == -1
    assert lib.cpt_mog2_apply(None, frames.data_ptr(), 1, 97 * 61, lrs.ctypes.data, None) == -1
    assert lib.cpt_mog2_background(m._h, None) == -1
    assert lib.cpt_mog2_frames(None) == -1
    with pytest.raises(ValueError):
        m.apply(torch.zeros((61, 96), dtype=torch.uint8, device="cuda"), -1)
    ir = native.IrMotion(ctx, 97, 61, 3)
    model = native.Mog2(ctx, 97, 61)
    d_mask = torch.empty((61, 97), dtype=torch.uint8, device="cuda")
    bgr = np.zeros((61, 97, 3), np.uint8)
    params = native.CptIrMotionClipParams(12, 2, 30, 15, 10, 0)
    res = native.CptIrMotionClipResult()

    def step(slot_new, slot_oldest, clip=None, result=res):
        clip = clip or ir.clip_record(model, d_mask, 0, 1, False, 0)
        st = native.CptIrMotionClipStep(0, slot_new, slot_oldest, 1, 0)
        return lib.cpt_ir_motion_step(ctypes.byref(clip), bgr.ctypes.data, ctypes.byref(st), ctypes.byref(params), result)

    with pytest.raises(native.NativeError):
        ir.ring_slot(3)
    assert step(3, 0) == -1 and step(-1, 0) == -1 and step(0, 3) == -1  # ring slots
    assert step(1, 0, result=None) == -1                                 # no result record
    assert step(1, 0, clip=ir.clip_record(model, 0, 0, 1, False, 0)) == -1  # no mask buffer
    assert model.frames == 0
    # everything still works afterwards, on the same context
    assert m.frames == 0
    compare(ctx, mh.scene("walk", (61, 97), 12, seed=17), [-1.0] * 12, 1000)
    rng = np.random.default_rng(18)
    a, b = (rng.integers(0, 256, (61, 97, 3), dtype=np.uint8) for _ in range(2))
    ir.gray(a, 0, copy_out=False)
    gb = ir.gray(b, 1)
    assert np.array_equal(gb, cv2.cvtColor(b, cv2.COLOR_BGR2GRAY))
    # the per-frame MOG2 step's counts equal cpt_ir_motion_detect's on the same mask: a fresh model takes b as its background,
    # and its next frame a gives the mask
    params = native.CptIrMotionClipParams(12, 2, 30, 3, 3, 0)
    for bgr_t, slot in ((b, 1), (a, 0)):
        r = ir.step(ir.clip_record(model, d_mask, 0, 1, False, 0), bgr_t, native.CptIrMotionClipStep(0, slot, 1 - slot, 1, 0), params)
    mask = d_mask.cpu().numpy()
    assert mask.any() and not mask.all() and r.mask_pixels > 0
    assert (r.diff_pixels, r.mask_pixels) == ir.detect(0, 1, 12, 3, mask=mask)
