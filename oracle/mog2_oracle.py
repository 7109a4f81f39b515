"""ctypes front-end of ``oracle/mog2_oracle.c``: OpenCV's MOG2 (detectShadows=False, one channel) restated in scalar C.
TEST INFRASTRUCTURE ONLY -- the product package never imports it.

``Mog2Oracle`` has cv2's surface: ``apply(frame, learning_rate)`` returns the foreground mask, ``background()`` is
``getBackgroundImage()``; ``stats`` accumulates which branches of the update ran (see the C file's header).
"""
import ctypes
import os
import subprocess

import numpy as np

from . import build as _build

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.path.join(HERE, "mog2_oracle.c")
LIB = os.path.join(_build.OUT_DIR, "libmog2_oracle.so")
STAT_NAMES = ("prune", "clamp_min", "clamp_max", "replace_weakest", "equal_swap", "five_modes", "new_mode", "background")
_lib = None


def build(force=False):
    os.makedirs(_build.OUT_DIR, exist_ok=True)
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= os.path.getmtime(SOURCE):
        return LIB
    tmp = LIB + ".{}.tmp".format(os.getpid())
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", tmp, SOURCE, "-lm"], check=True)
    os.replace(tmp, LIB)
    return LIB


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        P, F = ctypes.c_void_p, ctypes.c_float
        _lib.mog2_apply.argtypes = [P, ctypes.c_int, P, P, P, P] + [F] * 8 + [P]
        _lib.mog2_apply.restype = None
        _lib.mog2_background.argtypes = [ctypes.c_int, P, P, P, F, P]
        _lib.mog2_background.restype = None
    return _lib


def rates(learning_rate, nframes, history, complexity_reduction=0.05):
    """cv2's per-apply rule: (alphaT, prune) for the frame that makes the count ``nframes`` (already incremented)."""
    lr = learning_rate if (learning_rate >= 0 and nframes > 1) else 1.0 / min(2 * nframes, history)
    return np.float32(lr), np.float32(-lr * np.float64(np.float32(complexity_reduction)))


class Mog2Oracle:
    def __init__(self, shape, history=500, var_threshold=16.0, background_ratio=0.9, var_threshold_gen=9.0, var_init=15.0,
                 var_min=4.0, var_max=75.0, complexity_reduction=0.05):
        self.shape = tuple(shape)
        self.history = int(history)
        self.Tb, self.TB = np.float32(var_threshold), np.float32(background_ratio)
        self.Tg, self.var_init, self.var_min, self.var_max = (np.float32(v) for v in (var_threshold_gen, var_init, var_min, var_max))
        self.complexity_reduction = complexity_reduction
        self.nframes = 0
        self.stats = np.zeros(8, np.int64)
        self._init()

    def _init(self):
        n = self.shape[0] * self.shape[1]
        self.gmm = np.zeros((n, 5, 2), np.float32)
        self.mean = np.zeros((n, 5), np.float32)
        self.used = np.zeros(n, np.uint8)
        self.nframes = 0

    def apply(self, frame, learning_rate=-1.0):
        frame = np.ascontiguousarray(frame, dtype=np.uint8)
        assert frame.shape == self.shape
        if self.nframes == 0 or learning_rate >= 1:
            self._init()
        self.nframes += 1
        alpha, prune = rates(learning_rate, self.nframes, self.history, self.complexity_reduction)
        mask = np.empty(self.shape, np.uint8)
        p = lambda a: a.ctypes.data  # noqa: E731
        F = ctypes.c_float
        lib().mog2_apply(p(frame), frame.size, p(self.gmm), p(self.mean), p(self.used), p(mask), F(alpha), F(prune), F(self.Tb),
                         F(self.TB), F(self.Tg), F(self.var_init), F(self.var_min), F(self.var_max), p(self.stats))
        return mask

    def background(self):
        out = np.empty(self.shape, np.uint8)
        lib().mog2_background(out.size, self.gmm.ctypes.data, self.mean.ctypes.data, self.used.ctypes.data, ctypes.c_float(self.TB),
                              out.ctypes.data)
        return out

    def stat(self, name):
        return int(self.stats[STAT_NAMES.index(name)])
