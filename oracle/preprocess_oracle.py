"""CPU restatement (numpy) of the classifier-input preprocessing path, K9/K10.  TEST INFRASTRUCTURE ONLY.

Restates, with the reference file:line each function follows:
  * ``cv2.resize`` INTER_LINEAR / INTER_NEAREST on float32 (third-party OpenCV 4.x, call site
    ml_tools/imageprocessing.py:77-82);
  * ``resize_and_pad`` (ml_tools/imageprocessing.py:11-70);
  * ``normalize`` (ml_tools/imageprocessing.py:151-169);
  * ``preprocess_frame`` (ml_tools/preprocess.py:56-113) as called by
    ``Interpreter.preprocess_segments`` (ml_tools/interpreter.py:365-474) with ``get_limits``
    (ml_tools/interpreter.py:315-363), default HyperParams (diff_norm on, thermal_diff_norm off);
  * ``preprocess_movement`` / ``square_clip`` (ml_tools/preprocess.py:151-202,
    ml_tools/imageprocessing.py:85-104).
Pinned by tests/test_preprocess_oracle.py against fixtures generated from the reference itself
(tests/golden/pre_*.npz, tests/golden/make_golden_preprocess.py) and against the installed cv2
where available.
"""
import numpy as np

INTER_NEAREST = 0
INTER_LINEAR = 1


def linear_taps(dn, sn, thin):
    """Source taps of cv2.resize INTER_LINEAR along one axis for destination indices 0..dn-1: (i0, i1, w), the
    fp32 weight w of the second tap, before any edge rule.  Two coordinate rules, measured against cv2 4.13 (x86):
      * not thin (both source sides > 1, IPP's linear resize): f = (d + 0.5) * (sn / dn) - 0.5 in double, the
        ratio taken directly (not as 1 / (dn / sn): that misplaces coordinates that land exactly on an integer),
        product and difference rounded separately; i0 = floor(f), w = fp32(f - i0);
      * thin (a source side is 1, OpenCV's own resizeGeneric_): f = fp32((d + 0.5) * (1 / (dn / sn)) - 0.5), the
        coordinate rounded to fp32 before the floor; i0 = floor(f), w = f - i0 in fp32."""
    d = np.arange(dn, dtype=np.float64) + 0.5
    if thin:
        f = (d * (1.0 / (dn / sn)) - 0.5).astype(np.float32)
        i0 = np.floor(f).astype(np.int64)
        w = f - i0.astype(np.float32)
    else:
        f = d * (sn / dn) - 0.5
        i0 = np.floor(f).astype(np.int64)
        w = (f - i0).astype(np.float32)
    return i0, i0 + 1, w


def clamp_taps(i0, i1, w, sn, zero_weight):
    """The edge rule: taps outside [0, sn-1] are clamped; with zero_weight an index clamped at either end also
    gets weight 0 (i0 < 0 -> (0, 1, 0); i0 >= sn-1 -> (sn-1, sn-1, 0)), without it the weight is kept."""
    w = w.copy()
    if zero_weight:
        w[(i0 < 0) | (i0 >= sn - 1)] = 0
        i0 = np.clip(i0, 0, sn - 1)
        return i0, np.minimum(i0 + 1, sn - 1), w
    return np.clip(i0, 0, sn - 1), np.clip(i1, 0, sn - 1), w


def resize_linear(src, dw, dh):
    """cv2.resize(float32, (dw, dh), INTER_LINEAR), bit for bit with cv2 4.13 on x86 (IPP build).  Half-pixel
    centres; horizontal pass (fp32 rows) then vertical pass.  Measured with live cv2 (tests/test_resize_cv2.py):
      * identity (dw, dh) == (sw, sh): a copy;
      * both source sides > 1 (IPP): taps of linear_taps(thin=False) in both directions, clamped with the weight
        zeroed at both ends in both directions, each pair as fma(b - a, w, a) (the fp32 difference, then one fused
        multiply-add).  One side unchanged, integer up- and downscales and exact 2x downscales all take this form:
        there is no INTER_AREA switch for fp32 here;
      * a source side of 1, 1x1 included (OpenCV's generic path): taps of linear_taps(thin=True); horizontally the
        index is clamped with the weight zeroed, vertically only the row index is clamped and the weight is kept;
        each pair as fl(a * fl(1 - w)) + fl(b * w), two rounded products and a rounded sum, no fused multiply-add.
        So a 1-row source resized to dh rows gives rows that differ from the source row by ULPs."""
    src = np.asarray(src, np.float32)
    sh, sw = src.shape
    if (dw, dh) == (sw, sh):
        return src.copy()
    thin = sw == 1 or sh == 1
    x0, x1, wx = clamp_taps(*linear_taps(dw, sw, thin), sw, zero_weight=True)
    y0, y1, wy = clamp_taps(*linear_taps(dh, sh, thin), sh, zero_weight=not thin)

    def lerp(a, b, w):
        if thin:
            return a * (np.float32(1) - w) + b * w  # (fp32 numpy: each product and the sum rounded)
        return fma32(b - a, np.broadcast_to(w, a.shape), a)

    rows = lerp(src[:, x0], src[:, x1], wx[None, :])  # (sh, dw)
    return lerp(rows[y0], rows[y1], wy[:, None])


def fma32(x, y, z):
    """fp32 fma(x, y, z) with one rounding, elementwise.  The product of two fp32 values is exact in fp64; the fp64
    sum is turned into its round-to-odd value (TwoSum gives the exact error), whose rounding to fp32 is the correct
    rounding of the exact x * y + z -- a plain fp64 sum would round twice."""
    p = np.asarray(x, np.float32).astype(np.float64) * np.asarray(y, np.float32).astype(np.float64)
    z = np.asarray(z, np.float32).astype(np.float64)
    s = p + z
    t = s - p
    err = (p - (s - t)) + (z - t)
    even = (s.view(np.int64) & 1) == 0
    s = np.where((err != 0) & even, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def resize_nearest(src, dw, dh):
    """cv2.resize INTER_NEAREST: src index = min(floor(dst * src/dst), src-1)."""
    src = np.asarray(src)
    sh, sw = src.shape
    # OpenCV: ifx = 1 / (dsize / ssize) in double; sx = min(cvFloor(dx * ifx), ssize - 1)
    xs = np.minimum(np.floor(np.arange(dw) * (1.0 / (dw / sw))).astype(np.int64), sw - 1)
    ys = np.minimum(np.floor(np.arange(dh) * (1.0 / (dh / sh))).astype(np.int64), sh - 1)
    return src[ys][:, xs].astype(np.float32)


def resized_size(w, h, dim):
    """imageprocessing.py:24-31: aspect-preserving target size, numpy round (half to even), clamped to [1, dim]."""
    scale = min(dim[0] / h, dim[1] / w)
    width = int(np.round(np.float64(w) * scale))
    height = int(np.round(np.float64(h) * scale))
    return min(max(width, 1), dim[0]), min(max(height, 1), dim[1])


def paste_offsets(fw, fh, dim, region, crop, keep_edge=True):
    """imageprocessing.py:44-59 with edge_offset == (0, 0, 0, 0): centred, or anchored to the side of the
    crop rectangle the region touches.  region / crop are (x, y, w, h)."""
    ox = (dim[1] - fw) // 2
    oy = (dim[0] - fh) // 2
    if keep_edge and crop is not None:
        rx, ry, rw, rh = region
        cx, cy, cw, ch = crop
        if rx <= cx:
            ox = min(0, dim[1] - fw)
        elif rx + rw >= cx + cw:
            ox = max(dim[1] - fw, 0)
        if ry <= cy:
            oy = min(0, dim[0] - fh)
        elif ry + rh >= cy + ch:
            oy = max(dim[0] - fh, 0)
    return ox, oy


def resize_and_pad(frame, dim, region, crop, keep_edge=True, pad=None, interpolation=INTER_LINEAR):
    frame = np.asarray(frame)
    h, w = frame.shape
    fw, fh = resized_size(w, h, dim)
    if pad is None:
        pad = frame.min()
    out = np.full(dim, pad, dtype=np.float32)
    small = resize_linear(frame, fw, fh) if interpolation == INTER_LINEAR else resize_nearest(frame, fw, fh)
    ox, oy = paste_offsets(fw, fh, dim, region, crop, keep_edge)
    out[oy : oy + fh, ox : ox + fw] = small
    return out


def normalize(data, mn=None, mx=None, new_max=1):
    """imageprocessing.py:151-169.  Returns (array, ok)."""
    data = np.asarray(data)
    if data.size == 0:
        return np.zeros(data.shape), False
    mx = np.amax(data) if mx is None else mx
    mn = np.amin(data) if mn is None else mn
    if mx == mn:
        if mx == 0:
            return np.zeros(data.shape), False
        return data / mx, True
    return new_max * (np.float32(data) - mn) / (mx - mn), True


def track_limits(filtered, regions):
    """get_limits with diff_norm: (min, max) of region.subimage(filtered) over the track's non-blank regions;
    the max starts at 0.  regions: rows [frame, x, y, w, h, blank, ...]; filtered indexed by frame number."""
    lo, hi = None, np.float32(0)
    for frame, x, y, w, h, blank in (r[:6] for r in reversed(regions)):
        if blank or w <= 0 or h <= 0 or frame < 0 or frame >= len(filtered):
            continue
        sub = np.float32(filtered[frame][y : y + h, x : x + w])
        lo = sub.min() if lo is None or sub.min() < lo else lo
        hi = sub.max() if sub.max() > hi else hi
    return lo, hi


def thermal_limits(thermal, regions):
    """get_limits with thermal_diff_norm (interpreter.py:338-345): (min, max) of frame.thermal - np.median(frame.thermal)
    over the WHOLE frame of every non-blank region of the track (float32 arithmetic, as float_arrays() makes the frames)."""
    lo = hi = None
    for frame, x, y, w, h, blank in (r[:6] for r in reversed(regions)):
        if blank or w <= 0 or h <= 0 or frame < 0 or frame >= len(thermal):
            continue
        t = np.float32(thermal[frame])
        d = t - np.median(t)
        lo = d.min() if lo is None or d.min() < lo else lo
        hi = d.max() if hi is None or d.max() > hi else hi
    return lo, hi


def preprocess_track(thermal, filtered, regions, crop, segments, dim=(32, 32), frames_per_row=5, seed=None, preprocess_fn=None,
                     diff_norm=True, thermal_diff_norm=False):
    """Interpreter.preprocess_segments for one track.  thermal (T,H,W) uint16, filtered (T,H,W) float32
    (frame index == frame number), regions rows [frame, x, y, w, h, blank], segments = list of frame-number
    arrays.  Returns float32 (n_segments, dim*rows, dim*rows, 2)."""
    by_frame = {int(r[0]): r for r in regions}
    unique = []
    for seg in segments:
        for f in seg:
            if int(f) not in unique:
                unique.append(int(f))
    medians = {}
    clip_at_zero = True
    for f in unique:
        _, x, y, w, h = by_frame[f][:5]
        medians[f] = np.median(thermal[f])
        if clip_at_zero:
            sub = np.float32(thermal[f][y : y + h, x : x + w]) - medians[f]
            if np.median(sub) <= 0:
                clip_at_zero = False
    # interpreter.py:405-408: limits only when one of the two options asks for them; preprocess.py:92-113: without filtered
    # limits BOTH channels are normalised per tile (Frame.normalize), and thermal limits only switch the clip off
    lo, hi = track_limits(filtered, regions) if diff_norm else (None, None)
    tlim = thermal_limits(thermal, regions) if thermal_diff_norm else None
    tiles = {}
    for f in unique:
        _, x, y, w, h = (int(v) for v in by_frame[f][:5])
        region = (x, y, w, h)
        t = resize_and_pad(np.float32(thermal[f][y : y + h, x : x + w]), dim, region, crop, keep_edge=True)
        fl = resize_and_pad(np.float32(filtered[f][y : y + h, x : x + w]), dim, region, crop, keep_edge=True, pad=0)
        t = t - np.float32(medians[f]) if float(medians[f]) == np.float32(medians[f]) else (t - medians[f])
        t = np.float32(t)
        if tlim is None and clip_at_zero:
            t = np.clip(t, 0, None)
        if diff_norm:
            fl, _ = normalize(fl, lo, hi, new_max=255)
            if tlim is not None:
                t, _ = normalize(t, tlim[0], tlim[1], new_max=255)
            else:
                t, _ = normalize(t, new_max=255)
        else:
            fl, _ = normalize(fl, new_max=255)
            t, _ = normalize(t, new_max=255)
        tiles[f] = (np.float32(t), np.float32(fl))
    out = []
    for seg in segments:
        samples = list(range(len(seg)))
        n = frames_per_row * 5
        if len(seg) < n:
            rng = np.random.default_rng(seed)
            samples.extend(rng.choice(samples, n - len(seg)))
            samples.sort()
        image = np.zeros((frames_per_row * dim[0], frames_per_row * dim[1], 2), np.float32)
        i = 0
        for row in range(frames_per_row):
            for col in range(frames_per_row):
                t, fl = tiles[int(seg[samples[i]])]
                image[row * dim[0] : (row + 1) * dim[0], col * dim[1] : (col + 1) * dim[1], 0] = t
                image[row * dim[0] : (row + 1) * dim[0], col * dim[1] : (col + 1) * dim[1], 1] = fl
                i += 1
        if preprocess_fn == "inc3":
            image = image / np.float32(127.5) - np.float32(1.0)
        out.append(image)
    return np.float32(out)
