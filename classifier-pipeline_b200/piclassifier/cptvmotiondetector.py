"""``CPTVMotionDetector`` and ``is_affected_by_ffc`` (piclassifier/cptvmotiondetector.py:14-234)."""
from collections import namedtuple
from datetime import timedelta
from typing import NamedTuple

import numpy as np

from .. import native
from ..ml_tools.rectangle import Rectangle
from .motiondetector import MotionDetector, SlidingWindow, WeightedBackground

FFC_PERIOD = timedelta(seconds=9.9)
_NO_FRAME = -(2**31)  # frame reference of a cursor that is None (fails the native range check if the step reads it)

# One planned device step: flags (native.MOTION_*), ring slots of the new, oldest and oldest non-FFC frames, delta ring
# slots, the ring slots RunningMean starts from (None: no initialisation) and the trigger rule that applies.
_Step = namedtuple("_Step", "flags new oldest nonffc diff_new diff_old mean_slots reset detect")


class MotionTrace(NamedTuple):
    """Per frame, what a caller of the ``process_frame`` loop reads after each frame."""

    movement_detected: np.ndarray  # bool
    triggered: np.ndarray          # int64
    temp_thresh: np.ndarray        # float64
    processed: np.ndarray          # int64
    diff: np.ndarray               # int64, last_diff


def is_affected_by_ffc(cptv_frame):
    """A frame taken during / just after a flat-field correction (cptvmotiondetector.py:211-222).

    parity: with integer ``time_on`` / ``last_ffc_time`` (milliseconds from the CPTV decoder) the
    difference is compared with ``FFC_PERIOD.seconds`` == 9, i.e. nine *milliseconds*."""
    if hasattr(cptv_frame, "ffc_status") and cptv_frame.ffc_status in [1, 2]:
        return True
    if cptv_frame.time_on is None or cptv_frame.last_ffc_time is None:
        return False
    if isinstance(cptv_frame.time_on, int):
        return (cptv_frame.time_on - cptv_frame.last_ffc_time) < FFC_PERIOD.seconds
    return (cptv_frame.time_on - cptv_frame.last_ffc_time) < FFC_PERIOD


def since_ffc(cptv_frame):
    if hasattr(cptv_frame, "ffc_status") and cptv_frame.ffc_status in [1, 2]:
        return True
    if cptv_frame.time_on is None or cptv_frame.last_ffc_time is None:
        return False
    return cptv_frame.time_on - cptv_frame.last_ffc_time


class CPTVMotionDetector(MotionDetector):
    """Streaming motion trigger for Lepton frames (cptvmotiondetector.py:14-205).

    Same constructor, attributes and return values as the reference class.  The frame ring, the uint32
    running sum, the weighted background and the motion count live on the device; ``process_frame`` is one
    host->device frame copy, one fused kernel launch (csrc/motion_kernels.cu) and a 32-byte read-back.  The
    ring bookkeeping (``SlidingWindow`` cursors, FFC handling, trigger counting) stays on the host and keeps
    the frame objects for ``preview_frames`` / ``get_recent_frame``."""

    FFC_PERIOD = FFC_PERIOD
    BACKGROUND_WEIGHT_ADD = 0.1
    MEAN_FRAMES = 45

    def __init__(self, thermal_config, dynamic_thresh, headers, detect_after=None, device=None):
        super().__init__(thermal_config, headers)
        self.headers = headers
        if headers.model and headers.model.lower() == "lepton3.5":
            CPTVMotionDetector.BACKGROUND_WEIGHT_ADD = 1  # class attribute, as in the reference
        self.config = thermal_config.motion
        self.location_config = thermal_config.location
        self.num_preview_frames = thermal_config.recorder.preview_secs * headers.fps
        self.compare_gap = self.config.frame_compare_gap + 1
        edge = self.config.edge_pixels
        self.min_frames = thermal_config.recorder.min_secs * headers.fps
        self.max_frames = thermal_config.recorder.max_secs * headers.fps
        if not self.config.one_diff_only:
            self.diff_window = SlidingWindow(self.compare_gap, np.int32)
        self.running_mean = None  # becomes the device running sum (True once started)
        self.thermal_window = SlidingWindow(self.num_preview_frames + 1, "O")
        self.processed = 0
        self.thermal_thresh = 0
        self.crop_rectangle = Rectangle(edge, edge, headers.res_x - 2 * edge, headers.res_y - 2 * edge)
        self._background = WeightedBackground(edge, self.crop_rectangle, self.res_x, self.res_y,
                                              CPTVMotionDetector.BACKGROUND_WEIGHT_ADD, self.config.temp_thresh, device=device)
        self.movement_detected = False
        self.dynamic_thresh = dynamic_thresh
        self.triggered = 0
        self.ffc_affected = False
        self.detect_after = self.thermal_window.size * 2 if detect_after is None else detect_after
        self._ctx = self._background.ctx
        self._motion = native.Motion(self._ctx, self.thermal_window.size, self.MEAN_FRAMES,
                                     0 if self.config.one_diff_only else self.compare_gap, self._background.weight_slot)
        self._ring_refs = [-1 - s for s in range(self.thermal_window.size)]  # each ring slot as a frame reference
        self._clip = self._motion.clip_record(self._background.d_state, None, 0.0, 0, 0, 1)  # process_frame's detector record
        self._average = None
        self.last_diff = 0

    @property
    def _m(self):
        """Address of the detector's struct cpt_motion, whose leading members name its device buffers."""
        return self._motion.address

    @property
    def calibrating(self):
        return self.ffc_affected

    def preview_frames(self):
        return self.thermal_window.get_frames()[:-1]

    @property
    def temp_thresh(self):
        return self._background.average

    @property
    def background(self):
        return self._background.background

    def get_recent_frame(self):
        return self.thermal_window.current

    def disconnected(self):
        self.thermal_window.reset()
        if not self.config.one_diff_only:
            self.diff_window.reset()
        self.processed = 0

    def _pix(self, cptv_frame):
        pix = np.ascontiguousarray(cptv_frame.pix)
        if pix.dtype != np.uint16:
            raise TypeError("CPTVMotionDetector frames must be uint16")
        if pix.shape != (self.res_y, self.res_x):
            raise ValueError("frame shape {} does not match {}x{}".format(pix.shape, self.res_x, self.res_y))
        return pix

    def _plan(self, cptv_frame, force_process):
        """Host half of ``process_frame`` before the device step: FFC state, ``can_record()`` (called once), the
        ``SlidingWindow`` cursors and ``processed``.  Returns the device step, or None for a frame outside the recording
        window, which only replaces the ring's current frame."""
        prev_ffc = self.ffc_affected
        self.ffc_affected = is_affected_by_ffc(cptv_frame)
        self.num_frames += 1
        win = self.thermal_window
        if not (self.can_record() or force_process):
            win.update_current_frame(cptv_frame, self.ffc_affected)
            return None
        win.add(cptv_frame, self.ffc_affected)
        flags, mean_slots = 0, None
        if self.running_mean is None:
            n_stored = len(win.get_frames()[: self.MEAN_FRAMES])
            if n_stored == 1:
                flags |= native.MOTION_MEAN | native.MOTION_MEAN_RESTART
            else:
                # frames were only stored so far (outside the recording window): RunningMean(last_45)
                mean_slots = [(win.oldest_index + i) % win.size for i in range(n_stored)]
            self.running_mean = True
        else:
            flags |= native.MOTION_MEAN
        if not self.ffc_affected:
            flags |= native.MOTION_BACKGROUND
        reset = self.ffc_affected or prev_ffc
        detect = not reset and self.processed > self.detect_after
        diff_new = diff_old = -1
        if reset and prev_ffc:
            win.non_ffc_index = win.last_index
        if detect:
            flags |= native.MOTION_DETECT
            if self.config.warmer_only:
                flags |= native.MOTION_WARMER_ONLY
            if self.config.one_diff_only:
                flags |= native.MOTION_ONE_DIFF
            else:
                dw = self.diff_window
                if self.processed > 2 and dw.non_ffc_index is not None:
                    diff_old = dw.non_ffc_index
                dw.add(True, self.ffc_affected)
                diff_new = dw.last_index
        self.processed += 1
        return _Step(flags, win.last_index, win.oldest_index, win.non_ffc_index, diff_new, diff_old, mean_slots, reset, detect)

    def _apply(self, step, result):
        """Host half of ``process_frame`` after the device step (``result``: its cpt_motion_result): the background's
        average and the trigger counter."""
        if step is None:
            self.movement_detected = False
            return
        if step.flags & native.MOTION_BACKGROUND:
            self._background.invalidate(average=result.average)
        if step.reset:
            self.movement_detected = False
            self.triggered = 0
        elif step.detect:
            self.last_diff = int(result.diff)
            movement = self.last_diff > self.config.count_thresh
            self.triggered = self.triggered + 1 if movement else 0
            self.movement_detected = self.triggered >= self.config.trigger_frames

    def _init_average(self):
        init_avg = self._background._init_average
        return float(init_avg if init_avg is not None else 0.0)

    def process_frame(self, cptv_frame, force_process=False):
        pix = self._pix(cptv_frame)
        step = self._plan(cptv_frame, force_process)
        result = None
        if step is None:
            self._motion.store(pix, self.thermal_window.last_index)
        else:
            mean_rows = []
            record = _step_record(step, self._ring_refs, mean_rows)
            self._clip.init_average, self._clip.delta_thresh = self._init_average(), self.config.delta_thresh
            result = self._motion.step(self._clip, pix, record, mean_rows)
        self._apply(step, result)
        return self.movement_detected

    def process_frames(self, cptv_frames, force_process=False):
        """``for f in cptv_frames: self.process_frame(f, force_process)`` in one staged upload and one launch
        (``process_clips`` with this detector alone).  Returns the per-frame ``MotionTrace``."""
        return process_clips([self], [cptv_frames], force_process)[0]

    def skip_frame(self):
        return


def _step_record(step, ref, mean_rows):
    """The cpt_motion_clip_step of a planned step; ``ref[slot]`` is ring slot ``slot``'s frame reference (a row, or -1 - slot)."""
    mean_first, mean_slots = len(mean_rows), step.mean_slots or ()
    mean_rows += [ref[s] for s in mean_slots]  # the RunningMean start's frame references
    return (ref[step.new], ref[step.oldest], _NO_FRAME if step.nonffc is None else ref[step.nonffc], step.diff_new, step.diff_old,
            mean_first, len(mean_slots), step.flags)


class ClipSteps:
    """The device steps of many detectors over their frame lists, planned on the host by ``plan_clips``.

    Planning has already advanced each detector's host state (cursors, ``processed``, the frame objects of the ring);
    ``run`` does the device half and ``apply`` the rest of the host half.  Row ``offsets[i] + t`` of the staged frames is
    frame t of detector i."""

    def __init__(self, detectors, frame_lists, force_process):
        self.detectors = detectors
        self.plans = []
        self._processed = []  # per detector and frame: `processed` after the frame (planning runs ahead of apply)
        self.offsets = np.zeros(len(detectors) + 1, dtype=np.int64)
        steps, mean_rows, self._ring_rows = [], [], []
        self._clips = (native.CptMotionClip * len(detectors))()
        for i, (det, frames) in enumerate(zip(detectors, frame_lists)):
            win = det.thermal_window
            ref = list(det._ring_refs)  # what each ring slot holds: a row of this call, or itself
            ring_rows = np.full(win.size, -1, dtype=np.int32)
            first, plan, processed = len(steps), [], []
            for t, frame in enumerate(frames):
                row = int(self.offsets[i]) + t
                step = det._plan(frame, force_process)
                ref[win.last_index] = ring_rows[win.last_index] = row
                plan.append(step)
                processed.append(det.processed)
                if step is not None:
                    steps.append(_step_record(step, ref, mean_rows))
            self.plans.append(plan)
            self._processed.append(processed)
            self.offsets[i + 1] = self.offsets[i] + len(frames)
            self._ring_rows.append(ring_rows)
            self._clips[i] = det._motion.clip_record(det._background.d_state, ring_rows, det._init_average(), det.config.delta_thresh,
                                                     first, len(steps) - first)
        self.n_steps = len(steps)
        self._steps = (native.CptMotionClipStep * max(1, len(steps)))(*[native.CptMotionClipStep(*s) for s in steps])
        self._mean_rows = np.array(mean_rows, dtype=np.int32)
        self.results = (native.CptMotionResult * max(1, len(steps)))()

    @property
    def n_frames(self):
        return int(self.offsets[-1])

    def run(self, d_frames):
        """One ``cpt_motion_clips`` launch over ``d_frames`` (device uint16 [n_frames][H][W], any tensor or address)."""
        ctx = self.detectors[0]._ctx
        ctx.use_torch_stream()
        ctx.motion_clips(self._clips, len(self.detectors), d_frames, self.n_frames, self._steps, self.n_steps, self._mean_rows,
                         len(self._mean_rows), self.results)
        return self.results

    def apply(self):
        """The host half after the launch, frame by frame; one ``MotionTrace`` per detector."""
        traces, k = [], 0
        for i, (det, plan, processed) in enumerate(zip(self.detectors, self.plans, self._processed)):
            rows = []
            for t, step in enumerate(plan):
                result = None
                if step is not None:
                    result = self.results[k]
                    k += 1
                    if result.error:
                        raise native.NativeError("detector {} frame {}: running mean left the uint16 range (inconsistent ring / "
                                                 "mean window); the detector's state is not defined".format(i, t))
                det._apply(step, result)
                rows.append((det.movement_detected, det.triggered, float(det.temp_thresh), processed[t], det.last_diff))
            cols = list(zip(*rows)) if rows else [()] * 5
            traces.append(MotionTrace(np.array(cols[0], dtype=bool), np.array(cols[1], dtype=np.int64),
                                      np.array(cols[2], dtype=np.float64), np.array(cols[3], dtype=np.int64),
                                      np.array(cols[4], dtype=np.int64)))
        return traces


def _check_clips(detectors, frame_lists):
    if len(detectors) != len(frame_lists):
        raise ValueError("{} detectors but {} frame lists".format(len(detectors), len(frame_lists)))
    if len({id(d) for d in detectors}) != len(detectors):
        raise ValueError("a detector appears more than once")
    for det in detectors:
        if not isinstance(det, CPTVMotionDetector):
            raise TypeError("process_clips takes CPTVMotionDetector objects")
        d0 = detectors[0]
        if det._ctx is not d0._ctx or (det.res_x, det.res_y) != (d0.res_x, d0.res_y):
            raise ValueError("process_clips: the detectors must share one engine and one frame geometry")


def plan_clips(detectors, frame_lists, force_process=False):
    """Host half of ``process_clips`` up to the launch: plans every frame (this advances each detector's host state)
    and returns the ``ClipSteps`` to run on frames the caller stages itself, e.g. frames already on the device."""
    detectors, frame_lists = list(detectors), [list(f) for f in frame_lists]
    _check_clips(detectors, frame_lists)
    return ClipSteps(detectors, frame_lists, force_process)


def process_clips(detectors, frame_lists, force_process=False):
    """Every frame of ``frame_lists[i]`` through ``detectors[i]``: the same state and per-frame results as calling
    ``process_frame`` on each frame in turn, in one staged upload and one launch for all detectors.

    The detectors share one engine and geometry (else ValueError) and keep their own configuration.  Frames are
    checked before any state changes (TypeError / ValueError as ``process_frame``).  A step whose running mean leaves the
    uint16 range raises ``NativeError`` naming the detector and frame; that detector's state is then not defined.
    Returns one ``MotionTrace`` per detector."""
    import torch

    detectors, frame_lists = list(detectors), [list(f) for f in frame_lists]
    _check_clips(detectors, frame_lists)
    pix = [det._pix(f) for det, frames in zip(detectors, frame_lists) for f in frames]
    if not detectors:
        return []
    steps = ClipSteps(detectors, frame_lists, force_process)
    d_frames = None
    if pix:
        staged = np.stack(pix).view(np.int16)
        d_frames = torch.from_numpy(staged).to(detectors[0]._background.engine.device)
    steps.run(d_frames)
    return steps.apply()
