"""``IRMotionDetector`` and ``RollingBackground`` (piclassifier/irmotiondetector.py:11-160) for 640x480 IR cameras.

Per frame the reference converts BGR to grey, updates its background model, and erodes two binary images with a 15x15
(idle) or 10x10 (recording) box: ``absdiff(oldest grey, grey) > 12`` and the background model's foreground mask.  The grey
conversion, the difference mask, both erosions and the pixel counts run on the device (csrc/ir_kernels.cu), with the grey
ring resident in device memory.  The background model is OpenCV's MOG2: by default ``track.cliptracker.CVBackground``, cv2 on
the host, which needs the grey frame copied out and the mask copied back every frame.  ``MOG2Background`` (the same model
bit for bit, csrc/mog2.cuh) on the detector's engine keeps both on the device: ``process_frame`` is then one step of the
whole-recording call below (cpt_ir_motion_step), so per frame only the BGR frame goes in and the counts and the trigger
decision come out.  Any other object with ``update_background(gray, learning_rate=)`` / ``compute_filtered(None)`` /
``background`` can be passed as well.

With ``MOG2Background``, ``IRMotionDetector.process_frames`` and ``process_clips`` run whole recordings of many detectors
in one native call (cpt_ir_motion_clips): every frame's grey conversion, model update, erosion and trigger decision stay on
the device, so the next frame's learning rate and erosion box follow the previous frame's decision without a host round
trip.
"""
from collections import namedtuple
from typing import NamedTuple

import numpy as np

from .. import engine as _engine
from .. import native
from ..track.cliptracker import Background, CVBackground, MOG2Background, get_diff_back_filtered
from .motiondetector import MotionDetector, SlidingWindow


class RollingBackground(Background):
    """Running average over up to AVERAGE_OVER frames (irmotiondetector.py:11-47).  Plain array arithmetic."""

    AVERAGE_OVER = 1000

    def __init__(self, background_thresh=15):
        super().__init__()
        self._background = None
        self._frames = 0
        self.background_thresh = background_thresh

    def set_background(self, background, frames=1):
        self._background = np.float32(background)
        self._frames = frames

    def update_background(self, frame, filtered=None):
        if self._background is None:
            self._background = np.float32(np.array(frame, copy=True))
            return
        # (the reference compares against Background.AVERAGE_OVER, which does not exist, and assigns to a read-only
        # property: the intent -- an average over at most AVERAGE_OVER frames -- is what is kept)
        n = min(self._frames, RollingBackground.AVERAGE_OVER - 1)
        self._background = (self._background * n + frame) / (n + 1)
        self._frames += 1

    @property
    def background(self):
        return np.uint8(self._background)

    @property
    def frames(self):
        return min(self._frames, RollingBackground.AVERAGE_OVER)

    def compute_filtered(self, thermal, threshold=None):
        return get_diff_back_filtered(self.background, thermal, self.background_thresh)


WINDOW_SIZE = 50
MIN_FRAMES = 10 * 10  # 10 seconds
THRESHOLD = 12
TRIGGER_FRAMES = 2
MAX_TRIGGERED = 30
ERODE_IDLE = 15       # erosion box when not recording
ERODE_RECORDING = 10  # erosion box when recording
_PARAMS = native.CptIrMotionClipParams(THRESHOLD, TRIGGER_FRAMES, MAX_TRIGGERED, ERODE_IDLE, ERODE_RECORDING, 0)

# One planned device step: the ring slot the grey frame goes to, the oldest slot it is compared with, and whether the
# erosion and the trigger rule run (num_frames > MIN_FRAMES).
_Step = namedtuple("_Step", "slot oldest detect")


class IrMotionTrace(NamedTuple):
    """Per frame, what a caller of the ``process_frame`` loop reads after each frame."""

    movement_detected: np.ndarray  # bool, what process_frame returned
    triggered: np.ndarray          # int64
    diff_pixels: np.ndarray        # int64, eroded difference count before the min rule; -1 where no detection ran
    mask_pixels: np.ndarray        # int64, eroded foreground count before the min rule; -1 where no detection ran


class IRMotionDetector(MotionDetector):
    def __init__(self, thermal_config, headers, background=None, device=None):
        super().__init__(thermal_config, headers)
        self.num_preview_frames = thermal_config.recorder.preview_secs * headers.fps
        self.rgb_window = SlidingWindow(self.num_preview_frames, dtype=np.uint8)
        self.gray_window = SlidingWindow(self.num_preview_frames, dtype=np.uint8)  # holds ring slots; the pixels stay on the device
        self._background = background if background is not None else CVBackground()
        self.kernel_trigger = np.ones((ERODE_IDLE, ERODE_IDLE), "uint8")
        self.kernel_recording = np.ones((ERODE_RECORDING, ERODE_RECORDING), "uint8")
        self.movement_detected = False
        self.triggered = 0
        self.show = False
        self.prev_triggered = False
        self.processed = 0
        eng = _engine.get_engine(device)
        self._dev = native.IrMotion(eng.ctx, headers.res_x, headers.res_y, max(self.num_preview_frames, 1))
        self._device_background = isinstance(self._background, MOG2Background) and self._background.ctx is eng.ctx
        if self._device_background:
            eng.ctx.use_torch_stream()  # grey ring, model and erosion in one stream order from the first frame on

    def disconnected(self):
        self.rgb_window.reset()
        self.processed = 0

    @property
    def calibrating(self):
        return False

    @property
    def background(self):
        return self._background.background

    def get_kernel(self):
        return self.kernel_recording if self.movement_detected else self.kernel_trigger

    def preview_frames(self):
        return self.rgb_window.get_frames()[:-1]

    def get_recent_frame(self):
        return self.rgb_window.current

    def _check_frame(self, frame):
        shape = (self._dev.height, self._dev.width, 3)
        if np.asarray(frame).dtype != np.uint8 or np.shape(frame) != shape:
            raise ValueError("IR frames must be ({}, {}, 3) uint8".format(*shape[:2]))

    def _plan(self, frame, force_process):
        """Host half of ``process_frame`` before the device step: ``can_record()`` (called once), the ring cursors and
        ``num_frames``.  Returns the device step, or None for a frame outside the recording window, which only replaces the
        current frame."""
        if not (self.can_record() or force_process):
            self.rgb_window.update_current_frame(frame)
            self.num_frames += 1
            return None
        self.rgb_window.add(frame)
        # the grey ring lives on the device: the host window only tracks which slot is the oldest / the newest
        self.gray_window.add(None)
        step = _Step(self.gray_window.last_index, self.gray_window.oldest_index, self.num_frames > MIN_FRAMES)
        self.num_frames += 1
        return step

    def _apply(self, step, diff_erosion_pixels, erosion_pixels):
        """Host half of ``process_frame`` after the device step: the trigger rule on the two eroded counts."""
        if step is None or not step.detect:
            return
        # with the background frozen while motion lasts, a real change of the scene would keep the trigger up forever: the
        # frame difference bounds it
        if self.movement_detected:
            erosion_pixels = min(diff_erosion_pixels, erosion_pixels)
        self.prev_triggered = erosion_pixels > 0
        if erosion_pixels > 0:
            self.triggered = min(self.triggered + 1, MAX_TRIGGERED)
        else:
            self.triggered = max(self.triggered - 1, 0)
        if not self.movement_detected and self.triggered >= TRIGGER_FRAMES:
            self.movement_detected = True
        elif self.movement_detected and self.triggered <= 0:
            self.movement_detected = False

    def _apply_device(self, step, r, where=""):
        """``_apply`` on a device step's CptIrMotionClipResult ``r``; the device's trigger decision must agree."""
        diff, mask = (int(r.diff_pixels), int(r.mask_pixels)) if step.detect else (-1, -1)
        self._apply(step, diff, mask)
        if (self.movement_detected, self.triggered) != (bool(r.movement), int(r.triggered)):
            raise native.NativeError("{}the device's trigger decision differs from the host's".format(where))
        return diff, mask

    def _clip_record(self, first, n):
        """This detector's CptIrMotionClip of n device steps from step ``first``, on its MOG2Background's model and a new mask."""
        model, mask = self._background._steps(self._dev.height, self._dev.width, n)
        return self._dev.clip_record(model, mask, first, n, self.movement_detected, self.triggered)

    def process_frame(self, frame, force_process=False):
        """Returns True if there is motion (irmotiondetector.py:103-153)."""
        self._check_frame(frame)
        step = self._plan(frame, force_process)
        if step is None:
            self._apply(None, None, None)
        elif self._device_background:
            self._dev.ctx.use_torch_stream()
            r = self._dev.step(self._clip_record(0, 1), frame, native.CptIrMotionClipStep(0, step.slot, step.oldest, int(step.detect), 0),
                               _PARAMS)
            self._apply_device(step, r)
        else:
            gray = self._dev.gray(frame, step.slot)
            self._background.update_background(gray, learning_rate=0 if self.movement_detected else -1)
            counts = (None, None)
            if step.detect:
                counts = self._dev.detect(step.slot, step.oldest, THRESHOLD, self.get_kernel().shape[0], mask=self._background.compute_filtered(None))
            self._apply(step, *counts)
        return self.movement_detected

    def process_frames(self, frames, force_process=False):
        """``for f in frames: self.process_frame(f, force_process)`` in one native call (``process_clips`` with this
        detector alone).  Returns the per-frame ``IrMotionTrace``."""
        return process_clips([self], [frames], force_process)[0]

    @property
    def temp_thresh(self):
        return None


def _check_clips(detectors, frame_lists):
    """Everything ``process_clips`` rejects, checked before any state changes.  Returns per detector (frames for
    ``rgb_window``, frame addresses) and whether the frames are host memory."""
    import torch

    if len(detectors) != len(frame_lists):
        raise ValueError("{} detectors but {} frame lists".format(len(detectors), len(frame_lists)))
    if len({id(d) for d in detectors}) != len(detectors):
        raise ValueError("a detector appears more than once")
    frames_out, kinds = [], set()
    for det, frames in zip(detectors, frame_lists):
        if not isinstance(det, IRMotionDetector):
            raise TypeError("process_clips takes IRMotionDetector objects")
        d0 = detectors[0]
        if det._dev.ctx is not d0._dev.ctx or (det._dev.width, det._dev.height) != (d0._dev.width, d0._dev.height):
            raise ValueError("process_clips: the detectors must share one engine and one frame geometry")
        bg = det._background
        if not (isinstance(bg, MOG2Background) and bg.ctx is det._dev.ctx):
            raise ValueError("process_clips needs a MOG2Background on the detector's engine as background model (the same "
                             "masks as CVBackground, bit for bit): IRMotionDetector(..., background=MOG2Background())")
        if bg._model is not None and (bg._model.width, bg._model.height) != (det._dev.width, det._dev.height):
            raise ValueError("the detector's MOG2Background holds frames of another geometry")
        H, W = det._dev.height, det._dev.width
        if isinstance(frames, torch.Tensor):
            if not (frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and tuple(frames.shape[1:]) == (H, W, 3)
                    and frames.device.index == det._dev.ctx.device):
                raise ValueError("IR frames on the device must be one uint8 CUDA tensor [T][{}][{}][3] on the engine's device"
                                 .format(H, W))
            frames = frames.contiguous()
            views = list(frames.unbind(0))
            addresses = [frames.data_ptr() + t * H * W * 3 for t in range(len(views))]
            kinds.add("device")
        else:
            views = list(frames)
            for f in views:
                det._check_frame(f)
            arrays = [np.ascontiguousarray(f) for f in views]
            addresses = [a.ctypes.data for a in arrays]
            views = [(f, a) for f, a in zip(views, arrays)]  # the contiguous copies live until the call returns
            kinds.add("host")
        frames_out.append((views, addresses))
    if len({id(d._background) for d in detectors}) != len(detectors):
        raise ValueError("two detectors share one MOG2Background")
    if len(kinds) > 1:
        raise ValueError("process_clips takes host frames or device tensors, not both in one call")
    return frames_out, kinds == {"host"}


def process_clips(detectors, frame_lists, force_process=False):
    """Every frame of ``frame_lists[i]`` through ``detectors[i]``: the same state and per-frame results as calling
    ``process_frame`` on each frame in turn, in one native call for all detectors, with no host round trip per frame.

    Each detector needs a ``MOG2Background`` on its engine (ValueError otherwise, as for detectors that do not share one
    engine and geometry, or a detector given twice) and keeps its own configuration: ring length and MOG2 ``history`` /
    ``var_threshold``.  Frames are host uint8 [H][W][3] arrays, or one uint8 CUDA tensor [T][H][W][3] per detector, in which
    case ``rgb_window`` holds views of that tensor.  Every frame is checked before any state changes (ValueError as
    ``process_frame``).  Afterwards each detector, its grey ring and its MOG2Background (model, frame count, ``device_mask``)
    are as the ``process_frame`` loop would leave them.  Returns one ``IrMotionTrace`` per detector."""
    import torch

    detectors, frame_lists = list(detectors), [f if isinstance(f, torch.Tensor) else list(f) for f in frame_lists]
    frames, host = _check_clips(detectors, frame_lists)
    # plan every frame (advances each detector's host cursors)
    plans, steps, addresses, clips = [], [], [], []
    for det, (views, addrs) in zip(detectors, frames):
        first, plan = len(steps), []
        for view, address in zip(views, addrs):
            step = det._plan(view[0] if host else view, force_process)
            plan.append(step)
            if step is not None:
                steps.append(native.CptIrMotionClipStep(len(addresses), step.slot, step.oldest, int(step.detect), 0))
                addresses.append(address)
        plans.append(plan)
        if len(steps) > first:
            clips.append(det._clip_record(first, len(steps) - first))
    results = (native.CptIrMotionClipResult * max(1, len(steps)))()
    if clips:
        ctx = detectors[0]._dev.ctx
        ctx.use_torch_stream()
        params = native.CptIrMotionClipParams(THRESHOLD, TRIGGER_FRAMES, MAX_TRIGGERED, ERODE_IDLE, ERODE_RECORDING, int(host))
        table = np.array(addresses, dtype=np.uint64)
        ctx.ir_motion_clips((native.CptIrMotionClip * len(clips))(*clips), len(clips), table, len(table),
                            (native.CptIrMotionClipStep * len(steps))(*steps), len(steps), params, results)
    # the host half, frame by frame; the trigger rule runs again on the device's counts and must agree with its decisions
    traces, k = [], 0
    for i, (det, plan) in enumerate(zip(detectors, plans)):
        rows = []
        for t, step in enumerate(plan):
            diff = mask = -1
            if step is not None:
                diff, mask = det._apply_device(step, results[k], "detector {} frame {}: ".format(i, t))
                k += 1
            rows.append((det.movement_detected, det.triggered, diff, mask))
        cols = list(zip(*rows)) if rows else [()] * 4
        traces.append(IrMotionTrace(np.array(cols[0], dtype=bool), np.array(cols[1], dtype=np.int64), np.array(cols[2], dtype=np.int64),
                                    np.array(cols[3], dtype=np.int64)))
    return traces
