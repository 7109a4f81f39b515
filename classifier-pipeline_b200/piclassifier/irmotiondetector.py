"""``IRMotionDetector`` and ``RollingBackground`` (piclassifier/irmotiondetector.py:11-160) for 640x480 IR cameras.

Per frame the reference converts BGR to grey, updates its background model, and erodes two binary images with a 15x15
(idle) or 10x10 (recording) box: ``absdiff(oldest grey, grey) > 12`` and the background model's foreground mask.  The grey
conversion, the difference mask, both erosions and the pixel counts run on the device (csrc/ir_kernels.cu), with the grey
ring resident in device memory.  The background model is OpenCV's MOG2: by default ``track.cliptracker.CVBackground``, cv2 on
the host, which needs the grey frame copied out and the mask copied back every frame.  ``MOG2Background`` (the same model
bit for bit, csrc/mog2_kernels.cu) on the detector's engine keeps both on the device: the grey frame goes from its ring slot
into the model and the mask from the model into the erosion, so per frame only the BGR frame goes in and two counts come
out.  Any other object with ``update_background(gray, learning_rate=)`` / ``compute_filtered(None)`` / ``background`` can be
passed as well.
"""
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


class IRMotionDetector(MotionDetector):
    def __init__(self, thermal_config, headers, background=None, device=None):
        super().__init__(thermal_config, headers)
        self.num_preview_frames = thermal_config.recorder.preview_secs * headers.fps
        self.rgb_window = SlidingWindow(self.num_preview_frames, dtype=np.uint8)
        self.gray_window = SlidingWindow(self.num_preview_frames, dtype=np.uint8)  # holds ring slots; the pixels stay on the device
        self._background = background if background is not None else CVBackground()
        self.kernel_trigger = np.ones((15, 15), "uint8")   # erosion when not recording
        self.kernel_recording = np.ones((10, 10), "uint8")  # erosion when recording
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

    def process_frame(self, frame, force_process=False):
        """Returns True if there is motion (irmotiondetector.py:103-153)."""
        if self.can_record() or force_process:
            self.rgb_window.add(frame)
            # the grey ring lives on the device: the host window only tracks which slot is the oldest / the newest
            self.gray_window.add(None)
            slot = self.gray_window.last_index
            gray = self._dev.gray(frame, slot, copy_out=not self._device_background)
            if self.gray_window.oldest_index is None:
                return False
            learning_rate = 0 if self.movement_detected else -1
            if self._device_background:
                self._background.update_background_device(self._dev.ring_slot(slot), self._dev.width, self._dev.height, learning_rate)
            else:
                self._background.update_background(gray, learning_rate=learning_rate)
            if self.num_frames > MIN_FRAMES:
                k = self.get_kernel().shape[0]
                if self._device_background:
                    mask = dict(d_mask=self._background.device_mask)
                else:
                    mask = dict(mask=self._background.compute_filtered(None))
                diff_erosion_pixels, erosion_pixels = self._dev.detect(slot, self.gray_window.oldest_index, THRESHOLD, k, **mask)
                # with the background frozen while motion lasts, a real change of the scene would keep the trigger up
                # forever: the frame difference bounds it
                if self.movement_detected:
                    erosion_pixels = min(diff_erosion_pixels, erosion_pixels)
                self.prev_triggered = erosion_pixels > 0
                if erosion_pixels > 0:
                    self.triggered = min(self.triggered + 1, 30)
                else:
                    self.triggered = max(self.triggered - 1, 0)
                if not self.movement_detected and self.triggered >= TRIGGER_FRAMES:
                    self.movement_detected = True
                elif self.movement_detected and self.triggered <= 0:
                    self.movement_detected = False
        else:
            self.rgb_window.update_current_frame(frame)
        self.num_frames += 1
        return self.movement_detected

    @property
    def temp_thresh(self):
        return None
