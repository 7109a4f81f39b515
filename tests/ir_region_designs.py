"""Material for the batched IR regions (track/irtrackextractor.py detect_ir_regions_batch / ir_clip_regions): seeded grey IR
clips, designed 480x640 frames that each aim at one case of the components passes, and the per-frame composition with
live cv2 that the device is held equal to."""
import numpy as np

W, H = 640, 480
INT_MAX = 2**31 - 1


def ir_gray_clip(seed, frames, shape=(H, W), objects=3):
    """Grey uint8 frames: a textured static scene, sensor noise and a few warm objects moving across it."""
    rng = np.random.default_rng(seed)
    h, w = shape
    cell = max(1, min(h, w) // 16)
    scene = rng.integers(30, 140, (h // cell + 1, w // cell + 1)).repeat(cell, 0).repeat(cell, 1)[:h, :w].astype(np.int16)
    obj = [(rng.uniform(0, w), rng.uniform(0, h), rng.uniform(-6, 6) * w / 640, rng.uniform(-4, 4) * h / 480,
            int(rng.integers(max(2, w // 40), max(3, w // 8))), int(rng.integers(max(2, h // 40), max(3, h // 8))), int(rng.integers(50, 110)))
           for _ in range(objects)]
    out = np.empty((frames, h, w), np.uint8)
    for t in range(frames):
        f = scene + rng.integers(-3, 4, (h, w))
        for x0, y0, vx, vy, ow, oh, heat in obj:
            x, y = int(x0 + vx * t) % w, int(y0 + vy * t) % h
            f[y : y + oh, x : x + ow] += heat
        out[t] = np.clip(f, 0, 255)
    return out


def cv2_components(gray, threshold=0):
    """detect_objects_ir with live cv2: open with the tuple kernel, threshold, connectedComponentsWithStats."""
    import cv2

    opened = cv2.morphologyEx(gray, cv2.MORPH_OPEN, (15, 15))
    _, mask = cv2.threshold(opened, threshold, 255, cv2.THRESH_BINARY)
    n, labels, stats, _ = cv2.connectedComponentsWithStats(mask)
    return n, labels, stats


def cv2_regions(gray, scale=None, threshold=0):
    """(n, labels, stats, merged) of one frame: cv2's components, then merge_components on the rows without the background."""
    from classifier_pipeline_b200.track.irtrackextractor import merge_components

    n, labels, stats = cv2_components(gray, threshold)
    merged = np.array(merge_components(list(stats[1:]), scale=scale), np.int32).reshape(-1, 5)
    return n, labels, stats, merged


def cv2_masks(frames, learning_rates, history=1000, var_threshold=16):
    import cv2

    m = cv2.createBackgroundSubtractorMOG2(history=history, varThreshold=var_threshold, detectShadows=False)
    return np.stack([m.apply(f, None, float(lr)) for f, lr in zip(frames, learning_rates)])


def lifted(mask):
    """Grey input whose open is ``mask`` (0 / 1) away from the top rows: every column run of two or more rows is moved up
    one row, because the open turns input rows a..b into rows a+1..b."""
    out = np.zeros_like(mask, dtype=np.uint8)
    out[:-1] = mask[1:] * 255
    return out


def designs():
    """name -> 480x640 uint8 frame."""
    d = {"empty": np.zeros((H, W), np.uint8), "all_foreground": np.full((H, W), 255, np.uint8)}
    # one-row features: a single row survives no open (a lone row y gives O[y] = O[y+1] = 0)
    f = np.zeros((H, W), np.uint8)
    f[10, 5:600] = 255
    f[200, :] = 255
    f[300, 100:101] = 255
    f[479, 40:90] = 255
    d["one_row"] = f
    # objects in rows 0-1 and on all four edges (rows 0 and 1 of the open both take input row 0)
    f = np.zeros((H, W), np.uint8)
    f[0, 100:140] = 255            # row 0 only: becomes rows 0-1
    f[0:6, 300:310] = 255
    f[1, 500:520] = 255            # row 1 only: removed
    f[470:480, 200:260] = 255      # bottom edge
    f[100:140, 0:3] = 255          # left edge
    f[150:190, 636:640] = 255      # right edge
    f[0:4, 0:4] = 255              # corners
    f[0:4, 636:640] = 255
    f[476:480, 0:4] = 255
    f[476:480, 636:640] = 255
    d["edges"] = f
    # the raster-first pixel (3, 10) lies in block (1, 5); the pixel (0, 11) puts the component's least block at (0, 5)
    m = np.zeros((H, W), np.uint8)
    m[10:14, 3] = 1
    m[11:14, 0:3] = 1
    d["first_pixel_off_block"] = lifted(m)
    # blocks that interleave in block-raster order: Q's first pixel (14, 21) comes after S's (20, 20) in raster order but
    # Q's block (7, 10) comes before S's (10, 10); P and R interleave with them over block rows 10-14
    m = np.zeros((H, W), np.uint8)
    m[20:30, 10] = 1   # P
    m[21:25, 14] = 1   # Q
    m[23:27, 12] = 1   # R
    m[20:24, 20] = 1   # S
    for k in range(12):  # a row of the same pattern further down, shifted by one column each time
        m[60 + 3 * k : 64 + 3 * k, 30 + 5 * k] = 1
        m[61 + 3 * k : 64 + 3 * k, 32 + 5 * k] = 1
    d["interleaved_blocks"] = lifted(m)
    d["dot_grid"] = dot_grid()
    return d


def dot_grid():
    """Rows 0::3 and 1::3 set on even columns: the open leaves rows 3k+1, 3k+2 (and row 0, joined to rows 1-2) on each even
    column, 160 x 320 = 51 200 components."""
    f = np.zeros((H, W), np.uint8)
    for r0 in (0, 1):
        f[r0::3, 0::2] = 255
    return f


DOT_GRID_COMPONENTS = 51200


def merge_limits_cases():
    """(scale, (min_mass, min_size, max_gap)) with Python's semantics: int() truncates, a falsy scale keeps the defaults."""
    return [(None, (40, 16, 40)), (0, (40, 16, 40)), (1, (40, 16, 40)), (0.5, (20, 8, 20.0)), (1.5, (60, 24, 60.0)),
            (0.33, (13, 5, 40 * 0.33)), (2.7, (108, 43, 40 * 2.7))]
