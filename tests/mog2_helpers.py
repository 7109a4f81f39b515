"""Designed frame sequences and learning-rate schedules for the MOG2 tests (tests/test_mog2_oracle.py against cv2 on the host,
tests/test_mog2_gpu.py against cv2 and the C restatement on the device).  Each scene is built to reach one branch of the
update; ``BRANCHES`` names the counters of oracle/mog2_oracle.c that prove it does."""
import numpy as np


def _u8(a):
    return np.clip(np.rint(a), 0, 255).astype(np.uint8)


def scene(name, shape, frames, seed=0):
    """``frames`` uint8 frames of ``shape``."""
    rng = np.random.default_rng(seed)
    h, w = shape
    base = rng.integers(20, 230, shape).astype(np.float64)
    out = []
    for t in range(frames):
        if name == "constant":        # each pixel keeps its value: the variance falls to var_min
            f = base
        elif name == "noise":         # a new value every frame: five modes fill, the weakest is replaced, var_max on hits
            f = rng.integers(0, 256, shape)
        elif name == "flips":         # 0 / 255 per pixel
            f = np.where(rng.random(shape) < 0.5, 0, 255)
        elif name == "drift":         # slow drift plus sensor noise
            f = base + 0.4 * t + rng.normal(0, 2, shape)
        elif name == "walk":          # textured background, a bright block walks through
            f = base + rng.normal(0, 3, shape)
            y, x = (t * 3) % max(h - h // 4, 1), (t * 5) % max(w - w // 4, 1)
            f[y : y + h // 4, x : x + w // 4] += 70
        elif name == "mixed":         # cycles through the kinds above
            kind = t % 5
            f = (base, rng.integers(0, 256, shape), base + rng.integers(-2, 3, shape), np.where(rng.random(shape) < 0.5, 0, 255),
                 base.astype(np.int64) ^ (t & 7))[kind]
        elif name == "equal":         # two values alternating; with scene_rates' 0.5 then 0 the two modes keep equal weights
            f = np.where((np.arange(w)[None, :] + t) % 2 == 0, 60, 180) * np.ones(shape)
        elif name == "decay":         # a few frames of noise, then constant: the noise modes decay below -prune
            f = rng.integers(0, 256, shape) if t < 6 else base
        else:
            raise ValueError(name)
        out.append(_u8(f))
    return np.stack(out)


SCENES = ("constant", "noise", "flips", "drift", "walk", "mixed", "equal", "decay")

# the counters (oracle/mog2_oracle.c) each scene must move
BRANCHES = {
    "constant": ("clamp_min",),
    "noise": ("five_modes", "replace_weakest", "clamp_max"),
    "flips": ("new_mode",),
    "drift": ("new_mode",),
    "walk": ("new_mode",),
    "mixed": ("five_modes", "clamp_min"),
    "equal": ("equal_swap",),
    "decay": ("prune",),
}


def scene_rates(name, frames):
    """The learning rates a designed scene is run with: automatic, except for "equal", where one frame at 0.5 gives two
    modes of weight 0.5 and rate 0 keeps them so (a fitting mode then meets an equal weight above it and swaps)."""
    if name == "equal":
        return [-1.0, 0.5] + [0.0] * (frames - 2)
    return schedule("auto", frames)


def schedule(name, frames):
    """cv2 learningRate arguments per frame."""
    t = np.arange(frames)
    if name == "auto":
        return [-1.0] * frames
    if name == "recording":           # the IR detector freezes the model while motion lasts
        return [0.0 if 10 <= i < 25 or 40 <= i < 48 else -1.0 for i in t]
    if name == "reinit":              # 1 re-initialises the model mid-sequence
        return [1.0 if i in (0, 17, 31) else -1.0 for i in t]
    if name == "fractional":
        return [[0.3, 0.001, -1.0, 0.0, 0.999, 0.05][i % 6] for i in t]
    if name == "prune_boundary":      # prune computed with 0.05 in double instead of (double)0.05f differs at these rates
        return [[1.0 / 66, 0.010869565217391304, -1.0][i % 3] for i in t]
    raise ValueError(name)


SCHEDULES = ("auto", "recording", "reinit", "fractional", "prune_boundary")
