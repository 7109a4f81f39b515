"""BGR scenes for IRMotionDetector over whole recordings (tests/test_ir_motion_clips_gpu.py), and the detector restated on
cv2 alone (cv2.cvtColor, cv2.createBackgroundSubtractorMOG2, cv2.erode), which tests/test_ir_clip_scenes.py uses to check
that each designed scene reaches the case it is named for."""
import numpy as np

MIN_FRAMES, THRESHOLD, TRIGGER_FRAMES, MAX_TRIGGERED = 100, 12, 2, 30


def scene(seed, frames, shape=(120, 160), boxes=(), patches=()):
    """uint8 BGR frames [frames][H][W][3]: a static textured scene with sensor noise of +-3.
    boxes: (t0, t1, size, speed) -- a size x size box 90 brighter, moving right by `speed` pixels per frame for t0 <= t < t1.
    patches: (t0, size) -- from frame t0 on, a fixed size x size patch 80 brighter."""
    rng = np.random.default_rng(seed)
    h, w = shape
    cell = 8 if min(h, w) >= 32 else 1
    scene0 = rng.integers(30, 120, ((h + cell - 1) // cell, (w + cell - 1) // cell, 3)).repeat(cell, 0).repeat(cell, 1)[:h, :w].astype(np.int16)
    out = np.empty((frames, h, w, 3), np.uint8)
    for t in range(frames):
        f = scene0 + rng.integers(-3, 4, (h, w, 3))
        for t0, t1, size, speed in boxes:
            if t0 <= t < t1:
                x0 = (4 + (t - t0) * speed) % max(1, w - size)
                y0 = (h - size) // 3
                f[y0 : y0 + size, x0 : x0 + size] += 90
        for t0, size in patches:
            if t >= t0:
                f[h - size - 4 : h - 4, w - size - 4 : w - 4] += 80
        out[t] = np.clip(f, 0, 255)
    return out


# name: (frames, boxes, patches)
DESIGNS = {
    # a box appears at frame 110: the second frame with foreground starts the recording
    "trigger": (130, [(110, 122, 24, 6)], []),
    # a patch arrives during a recording: the frozen model keeps it foreground, and the frame difference ends the recording
    # while the mask count is still positive
    "freeze": (175, [(105, 125, 24, 6)], [(112, 30)]),
    # a box that moves for 45 frames: triggered saturates at 30, then counts down to 0
    "saturate": (200, [(105, 150, 24, 5)], []),
    # a big box starts a recording, a 12 x 12 box keeps it going under the 10 x 10 box, and after the recording the same
    # small box is eroded away by the 15 x 15 box
    "box_switch": (240, [(105, 112, 24, 6), (112, 150, 12, 3), (200, 230, 12, 3)], []),
    # detection starts at num_frames == MIN_FRAMES + 1, with a moving box in the frame difference from the start
    "min_frames": (104, [(0, 104, 24, 2)], []),
}


def design(name, seed=0, shape=(120, 160)):
    frames, boxes, patches = DESIGNS[name]
    return scene(seed, frames, shape, boxes, patches)


def cv2_trace(frames, ring=10, history=1000, var_threshold=16, inside=None, force=False):
    """IRMotionDetector.process_frame on every frame, restated on cv2: per frame (movement_detected, triggered, eroded
    difference count, eroded mask count), the counts -1 where no detection ran."""
    import cv2

    mog = cv2.createBackgroundSubtractorMOG2(history=history, varThreshold=var_threshold, detectShadows=False)
    grays, last, oldest = [None] * ring, None, None
    movement, trig, num, rows = False, 0, 0, []
    for t, f in enumerate(frames):
        d = m = -1
        if inside is None or inside[t] or force:
            if last is None:
                last = oldest = 0
            else:
                nxt = (last + 1) % ring
                if nxt == oldest:
                    oldest = (oldest + 1) % ring
                last = nxt
            g = cv2.cvtColor(np.ascontiguousarray(f), cv2.COLOR_BGR2GRAY)
            grays[last] = g
            mask = mog.apply(g, None, 0 if movement else -1)
            if num > MIN_FRAMES:
                k = np.ones((10, 10) if movement else (15, 15), np.uint8)
                delta = cv2.threshold(cv2.absdiff(grays[oldest], g), THRESHOLD, 255, cv2.THRESH_BINARY)[1]
                d, m = int((cv2.erode(delta, k) > 0).sum()), int((cv2.erode(mask, k) > 0).sum())
                e = min(d, m) if movement else m
                trig = min(trig + 1, MAX_TRIGGERED) if e > 0 else max(trig - 1, 0)
                if not movement and trig >= TRIGGER_FRAMES:
                    movement = True
                elif movement and trig <= 0:
                    movement = False
        num += 1
        rows.append((movement, trig, d, m))
    return np.array(rows, dtype=np.int64).reshape(-1, 4)


def check_design(name, tr):
    """Assert that trace rows (movement, triggered, diff, mask) reach the case `name` is designed for."""
    mov, trig, diff, mask = tr[:, 0].astype(bool), tr[:, 1], tr[:, 2], tr[:, 3]
    if name == "trigger":
        a = int(np.argmax(mask > 0))
        assert mask[a] > 0 and not mov[:a + 1].any() and trig[a] == 1 and mov[a + 1] and trig[a + 1] == TRIGGER_FRAMES
    elif name == "freeze":
        ends = [t for t in range(1, len(mov)) if mov[t - 1] and not mov[t]]
        assert ends, "no recording ended"
        e = ends[0]
        # the recording ends on the frame difference: the mask still shows the patch that arrived during the recording
        assert diff[e] == 0 and mask[e] > 0 and (mask[e:] > 0).all()
    elif name == "saturate":
        assert trig.max() == MAX_TRIGGERED
        top = int(np.flatnonzero(trig == MAX_TRIGGERED)[-1])
        assert np.array_equal(trig[top : top + MAX_TRIGGERED + 1], np.arange(MAX_TRIGGERED, -1, -1))
    elif name == "box_switch":
        # recording while the small box moves (counted under the 10 x 10 box) ...
        assert mov[115:150].all() and (diff[116:150] > 0).all() and (mask[115:150] > 0).any()
        # ... the recording ends, and the same small box later is eroded away under the 15 x 15 box
        assert not mov[195:].any() and (diff[205:230] == 0).all() and (mask[205:230] == 0).all()
    elif name == "min_frames":
        assert (diff[: MIN_FRAMES + 1] == -1).all() and (mask[: MIN_FRAMES + 1] == -1).all() and diff[MIN_FRAMES + 1] > 0
    else:
        raise ValueError(name)
