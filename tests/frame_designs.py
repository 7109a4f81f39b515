"""Designed clips for the per-frame mask and component stage (no GPU needed).

A design is a clip of two frames: a constant background frame (also the clip's init frame), then
``background + amplitude * pattern`` with a 0/1 pattern.  Its last frame is the frame under test: its filtered image is
exactly ``amplitude * pattern``.  (The quad-byte designs are longer: see ``quad_bound_design``.)  The amplitude is tuned so that the frame's mapped threshold ``ith`` lands in a chosen
range, which fixes how far the 5x5 blur spreads the pattern:
  * ``ith`` 0 (DILATE): the mask is the pattern grown by two pixels on every side;
  * ``ith`` 30..35 (POINTS): an isolated pattern pixel, or pixels three apart, stay single mask pixels;
  * ``ith`` 80..88 (LINES): a vertical pattern line stays one pixel wide, and lines three apart stay apart.
The close (``C[y] = M[y-1] | (M[y] & M[y-2])``) then moves the mask down a row.  A design is only trusted through its
reach: the functions below measure, from the C oracle's outputs alone, which side of each kernel switch the frame is on,
and ``tests/test_frame_designs.py`` asserts every design's claim.

The constants mirror what the kernels switch on: ``csrc/cptrack_kernels.cuh`` (bands, lean tables, slots, list cap, quad
byte bias) and ``csrc/strip_sweep.cu`` (the reference lag).
"""
from collections import namedtuple

import numpy as np

from oracle import oracle as orc

# csrc/cptrack_kernels.cuh
kBandRows = 24         # hot rows one band of frame_regions_kernel covers
kBandHalo = 4          # rows of normalised values a blur output can reach
kLeanSlots = 32        # components the in-CTA stage (components_lean) numbers; more: frame_components_kernel
kLeanParents = 1024    # its run ids: rows of the extent * runs per row
kRunsPerRow = 80
CPT_MAX_COMPONENTS = 255
kListCap = 1024        # marked 8-pixel groups the single kernel puts on its work lists; more: every group
kQuadRefBias = 64
# csrc/strip_sweep.cu
kRefLag = 8            # a frame's quad bytes are stored against its strip's minimum this many frames earlier
kRefDefault = kQuadRefBias

H, W = 120, 160
BACKGROUND = 3000
BT = 20
DILATE, POINTS, LINES = (0, 0), (30, 35), (80, 88)

Design = namedtuple("Design", "name frames bt claim")


def strip_rows(height, width):
    """First row of every strip of the strip sweep, and the end (cptrack.cu: strips of whole rows, at most 1920 pixels)."""
    rmax = max(1920 // width, 1)
    n = (height + rmax - 1) // rmax
    return [s * height // n for s in range(n + 1)]


# ---------------------------------------------------------------------------------------------------------------- making
def _frames(pattern, amp):
    bg = np.full(pattern.shape, BACKGROUND, np.uint16)
    return np.stack([bg, (BACKGROUND + amp * pattern.astype(np.int64)).astype(np.uint16)])


def _ith(pattern, amp, bt=BT):
    f = _frames(pattern, amp)
    _, th, _, _, _ = orc.normalise_frame(f[1], f[0].astype(np.int32), float(BACKGROUND), bt)
    return int(np.floor(th))


def tune(pattern, ith_range, bt=BT):
    """The least amplitude whose frame has lo <= ith <= hi (ith falls as the amplitude grows)."""
    lo, hi = ith_range
    a, b = 1, 65535 - BACKGROUND
    if _ith(pattern, b, bt) > hi:
        raise ValueError("no amplitude brings ith down to %d" % hi)
    while a < b:
        m = (a + b) // 2
        if _ith(pattern, m, bt) <= hi:
            b = m
        else:
            a = m + 1
    if _ith(pattern, a, bt) < lo:
        raise ValueError("ith jumps past [%d, %d]" % (lo, hi))
    return a


def design(name, pattern, mode, claim, bt=BT):
    return Design(name, _frames(pattern, tune(pattern, mode, bt)), bt, claim)


def points(coords, h=H, w=W):
    p = np.zeros((h, w), np.uint8)
    for y, x in coords:
        p[y, x] = 1
    return p


def grid(n, y0=2, x0=1, pitch=3, h=H, w=W, stagger=False):
    """n single pixels three apart, row by row; stagger: every other pixel one row lower, so that in each block row the
    lower pixel can come first in OpenCV label order."""
    out = []
    y = y0
    while len(out) < n:
        if y + 1 >= h - 1:
            raise ValueError("grid does not fit")
        for x in range(x0, w - 1, pitch):
            if len(out) == n:
                break
            out.append((y + (1 if stagger and (x // pitch) % 2 == 0 else 0), x))
        y += pitch + (1 if stagger else 0)
    return points(out, h, w)


# ----------------------------------------------------------------------------------------------------------------- reach
def run_oracle(d, max_comp=CPT_MAX_COMPONENTS):
    h, w = d.frames.shape[1:]
    p = orc.make_params(W=w, H=h, edge=1, background_thresh=d.bt, weight_add=0.1, max_comp=max_comp)
    return orc.extract_clip(d.frames, d.frames[0], p)


def closed_mask(o, t=1):
    return o["labels"][t] > 0


def runs_per_row(mask):
    m = mask.astype(np.int8)
    starts = np.diff(np.concatenate([np.zeros((m.shape[0], 1), np.int8), m], axis=1), axis=1) == 1
    return starts.sum(axis=1)


def row_extent(mask):
    rows = np.nonzero(mask.any(axis=1))[0]
    return (int(rows[0]), int(rows[-1])) if len(rows) else None


def frame_scalars(frames, o, t=1):
    """(ith, ac, gmn, gmx, fth) of frame t as frame_scalars_of computes them; fth None: no usable bound."""
    pix = frames[t]
    ac = int(np.rint(pix.astype(np.float64).mean() - o["avg"][t]))  # (rint: half to even, as Python's round)
    gmx, gmn = int(o["norm"][t, 0]), int(o["norm"][t, 1])
    ith = int(np.floor(o["thresh"][t]))
    fth = None
    if gmx != gmn and 255 * (gmx - gmn) < (1 << 24) and 0 <= ith < 255:
        fth = -(-(ith + 1) * (gmx - gmn) // 255) + ac + gmn
    return ith, ac, gmn, gmx, fth


def hot_rows(frames, o, t=1):
    """Rows that hold a pixel with F >= fth (F: the oracle's filtered image)."""
    fth = frame_scalars(frames, o, t)[4]
    if fth is None:
        return np.arange(frames.shape[1])
    return np.nonzero((o["filtered"][t] >= fth).any(axis=1))[0]


def bands(rows):
    """frame_regions_kernel's bands: kBandRows rows from the first hot row not yet covered on; [(lo, hi)] hot rows."""
    out, rows = [], list(rows)
    while rows:
        lo = rows[0]
        inb = [r for r in rows if r < lo + kBandRows]
        out.append((lo, inb[-1]))
        rows = rows[len(inb):]
    return out


def lean_rpr(frames, o, t=1):
    """Runs per row of components_lean's run table: min(80, 1024 / rows), rows = the mask's possible extent grown by the close."""
    rows = hot_rows(frames, o, t)
    h = frames.shape[1]
    c0, c1 = max(int(rows[0]) - 2, 0), min(int(rows[-1]) + 3, h - 1)
    return min(kRunsPerRow, kLeanParents // (c1 - c0 + 1))


def strip_dq(frames, o, t=1):
    """Per strip, fth - ref: ref is the strip's filtered minimum kRefLag frames earlier plus kQuadRefBias (strip_folder)."""
    fth = frame_scalars(frames, o, t)[4]
    rows = strip_rows(*frames.shape[1:])
    out = []
    for s in range(len(rows) - 1):
        if t >= kRefLag:
            ref = int(o["filtered"][t - kRefLag][rows[s]:rows[s + 1]].min())
            ref = max(min(ref, 1 << 20), -(1 << 20)) + kQuadRefBias
        else:
            ref = kRefDefault
        out.append(None if fth is None else fth - ref)
    return out


def marked_groups(frames, o, t=1, edge=1):
    """Lower bound on the single kernel's list_u length: the groups within 4 rows / 2 quads of an exact hot quad."""
    fth = frame_scalars(frames, o, t)[4]
    h, w = frames.shape[1:]
    if fth is None:
        return 0
    hotq = (o["filtered"][t] >= fth).reshape(h, w // 4, 4).any(axis=2)
    hotq[:edge] = False
    hotq[h - edge:] = False
    n = 0
    for r in range(h):
        near = hotq[max(r - 4, 0): r + 5].any(axis=0)
        mk = near.copy()
        for s in (1, 2):
            mk[s:] |= near[:-s]
            mk[:-s] |= near[s:]
        n += int(mk.reshape(-1, 2).any(axis=1).sum())
    return n


def strips_of_rows(rows, height, width):
    sr = strip_rows(height, width)
    return sorted({int(np.searchsorted(sr, r, side="right")) - 1 for r in rows})


def crosses_words(mask):
    """Per 32-pixel word boundary xb of the row: (a run covers xb - 1 and xb, a pixel links across xb only diagonally)."""
    out = []
    for xb in range(32, mask.shape[1], 32):
        a, b = mask[:, xb - 1], mask[:, xb]
        diag = (b[1:] & a[:-1] & ~b[:-1] & ~a[1:]) | (a[1:] & b[:-1] & ~a[:-1] & ~b[1:])
        out.append((bool((a & b).any()), bool(diag.any())))
    return out


def reach(d, o=None, t=None):
    """Everything the claims are written against, for the design's frame under test (its last frame)."""
    o = run_oracle(d) if o is None else o
    t = len(d.frames) - 1 if t is None else t
    m = closed_mask(o, t)
    ith, ac, gmn, gmx, fth = frame_scalars(d.frames, o, t)
    hr = hot_rows(d.frames, o, t)
    return dict(
        ncomp=int(o["ncomp"][t]), ith=ith, fth=fth, flat=gmx == gmn, extent=row_extent(m),
        max_runs=int(runs_per_row(m).max()), hot_rows=hr, bands=bands(hr) if fth is not None else None,
        rpr=lean_rpr(d.frames, o, t) if len(hr) else None, dq=strip_dq(d.frames, o, t),
        marked=marked_groups(d.frames, o, t), mask=m, labels=o["labels"][t],
        hot_strips=strips_of_rows(hr, *d.frames.shape[1:]) if fth is not None else None, words=crosses_words(m),
    )


# --------------------------------------------------------------------------------------------------------------- designs
def _vline(p, x, y0, y1):
    p[y0:y1 + 1, x] = 1
    return p


def comb(teeth, y0, y1, x0=1, pitch=3, h=H, w=W):
    """teeth one-pixel vertical lines three apart on rows y0..y1-1, joined by a line on row y1: one component whose rows
    hold `teeth` runs."""
    p = np.zeros((h, w), np.uint8)
    xs = [x0 + pitch * k for k in range(teeth)]
    for x in xs:
        _vline(p, x, y0, y1)
    p[y1, xs[0]:xs[-1] + 1] = 1
    return p


def quad_bound_design(name, strip, dq, bt=1000, amp=4000, h=H, w=W):
    """Strip `strip` is the only hot strip of the frame under test and its fth - ref is dq.

    kRefLag + 2 frames: a constant frame, a pulse that raises the whole strip by U, kRefLag - 1 constant frames, then the frame
    under test.  The pulse is kRefLag frames before the frame under test, so the strip's quad bytes there are stored
    against ref = U + kQuadRefBias (the pulse's pixels stay out of the background: it comes back to the constant level).
    The frame under test holds, inside the strip, one bright pixel that sets the range and a plateau whose level is the
    frame's own fth: its normalised value is ith + 1, so the plateau is foreground, and its quads' byte is fth - ref = dq
    itself, the value the byte compare decides on."""
    rows = strip_rows(h, w)
    y0, y1 = rows[strip], rows[strip + 1]
    test = np.zeros((h, w), np.int64)
    test[y0 + (y1 - y0) // 2, w - 20] = amp
    level = amp // 4
    for _ in range(10):
        test[y0 + 2:y1 - 2, 40:64] = level
        pair = np.stack([np.full((h, w), BACKGROUND, np.uint16), (BACKGROUND + test).astype(np.uint16)])
        o = run_oracle(Design(name, pair, bt, None))
        fth = frame_scalars(pair, o, 1)[4]
        if fth == level:
            break
        level = fth
    else:
        raise ValueError("plateau level does not settle")
    pulse = fth - kQuadRefBias - dq
    if not 0 < pulse < 65535 - BACKGROUND:
        raise ValueError("dq %d is out of reach" % dq)
    bg = np.full((h, w), BACKGROUND, np.uint16)
    up = bg.copy()
    up[y0:y1] += np.uint16(pulse)
    frames = np.stack([bg, up] + [bg] * (kRefLag - 1) + [pair[1]])
    return Design(name, frames, bt, lambda r: r["dq"][strip] == dq and r["hot_strips"] == [strip] and r["ncomp"] >= 1)


def designs():
    """All designs at 160x120.  Each claim is a predicate on reach()."""
    out = []
    # ---- in-CTA component table (kLeanSlots), compact extent
    for n in (31, 32, 33):
        out.append(design("lean_%d" % n, grid(n, y0=50, pitch=4), POINTS,
                          lambda r, n=n: r["ncomp"] == n and r["rpr"] == kRunsPerRow))
    # ---- run table: rpr = min(80, 1024 / rows); rows of rpr and rpr + 1 runs, one component each so that only the run table
    # decides.  A 20-row extent (rpr 51) and a full-height one (rpr 8)
    for k in (0, 1):
        p = comb(51 + k, 50, 64)
        out.append(design("runs_short_%s" % ("rpr" if k == 0 else "rpr_plus1"), p, LINES,
                          lambda r, k=k: r["rpr"] == 51 and r["max_runs"] == 51 + k and r["ncomp"] <= kLeanSlots))
        p = points([(2, 2), (117, 2)] + [(60, 10 + 6 * i) for i in range(8 + k)])
        out.append(design("runs_tall_%s" % ("rpr" if k == 0 else "rpr_plus1"), p, POINTS,
                          lambda r, k=k: r["rpr"] == 8 and r["max_runs"] == 8 + k and r["ncomp"] <= kLeanSlots))
    # ---- full slot table (CPT_MAX_COMPONENTS), staggered so that OpenCV order is not raster order of first pixels
    for n in (254, 255, 256, 600):
        out.append(design("slots_%d" % n, grid(n, stagger=True), POINTS, lambda r, n=n: r["ncomp"] == n))
    # ---- bands: hot rows spanning kBandRows and kBandRows + 1 rows; a second hot group 1..6 rows after a full band; a
    # component across a band boundary; a full-height object (five bands)
    for span in (kBandRows, kBandRows + 1):
        out.append(design("band_span_%d" % span, points([(30, 20), (30 + span - 1, 60)]), POINTS,
                          lambda r, span=span: len(r["bands"]) == (1 if span == kBandRows else 2)))
    for gap in range(1, 7):
        p = points([(30, 20), (30 + kBandRows - 1, 60), (30 + kBandRows - 1 + gap, 100)])
        out.append(design("band_gap_%d" % gap, p, POINTS,
                          lambda r, gap=gap: len(r["bands"]) == 2 and r["bands"][1][0] - r["bands"][0][1] == gap))
    out.append(design("band_crossing", _vline(np.zeros((H, W), np.uint8), 70, 20, 60), LINES,
                      lambda r: len(r["bands"]) == 2 and r["ncomp"] == 1))
    p = _vline(np.zeros((H, W), np.uint8), 80, 0, H - 1)
    p[40, 20] = p[90, 140] = 1
    out.append(design("band_full_height", p, DILATE, lambda r: len(r["bands"]) >= 5 and r["extent"] == (0, H - 1)))
    # ---- frame edges: objects on rows 0, 1, H-2, H-1, column 0 and in the last quad
    p = points([(0, 10), (1, 30), (H - 2, 50), (H - 1, 70), (40, 0), (70, W - 1), (100, W - 3)])
    out.append(design("edges_points", p, POINTS, lambda r: r["mask"][0].any() and r["mask"][:, 0].any() and r["mask"][:, W - 1].any()))
    p = points([(0, 10), (0, W - 1), (H - 1, 0), (H - 1, 60), (60, 0), (61, W - 1)])
    out.append(design("edges_blocks", p, DILATE,
                      lambda r: r["mask"][0].any() and r["mask"][H - 1].any() and r["mask"][:, 0].any() and r["mask"][:, W - 1].any()))
    # ---- word boundaries: runs across x = 32k, and chains that touch only diagonally across x = 32k (both directions)
    p = np.zeros((H, W), np.uint8)
    for i, xb in enumerate((32, 64, 96, 128)):
        p[10 + 8 * i, xb - 1] = 1                              # (DILATE: a run xb - 3 .. xb + 1)
        # squares that meet corner to corner: (xb - 1, y) and (xb, y + 1)
        p[50, xb - 3] = p[55, xb + 2] = 1                      # down-right across the boundary: needB for the lower square
        p[80 + i % 2, xb + 2] = p[85 + i % 2, xb - 3] = 1      # down-left: needC
    out.append(design("word_boundaries", p, DILATE, lambda r: r["ncomp"] == 12))
    p = np.zeros((H, W), np.uint8)
    for xb in (32, 64, 96, 128):
        p[30, xb - 1] = p[31, xb] = 1     # diagonal pixels across the boundary: one component
        p[60, xb] = p[61, xb - 1] = 1
    out.append(design("word_diagonal_points", p, POINTS, lambda r: r["ncomp"] == 8))
    # ---- label order: in each block row a component whose first pixel is on the lower row but further left comes first;
    # U-shapes whose arms join below
    p = np.zeros((H, W), np.uint8)
    for k in range(6):
        y = 11 + 12 * k               # (mask rows y + 1 = 2j and y + 2 = 2j + 1: one block row)
        p[y, 60 + 6 * k] = 1          # first in raster order, right
        p[y + 1, 20 + 4 * k] = 1      # one row lower, left: the smaller key
    out.append(design("label_order_rows", p, POINTS, lambda r: r["ncomp"] == 12))
    p = np.zeros((H, W), np.uint8)
    for x0, top_l, top_r in ((20, 30, 20), (70, 20, 30), (120, 25, 25)):
        _vline(p, x0, top_l, 60)
        _vline(p, x0 + 24, top_r, 60)
        p[60, x0:x0 + 25] = 1
        _vline(p, x0 + 12, top_l + 8, top_l + 14)    # a component inside the U
    out.append(design("label_order_u_shapes", p, LINES, lambda r: r["ncomp"] == 6))
    # ---- quad-byte bounds: dq = fth - ref around the dense switch (dq < -127) and the saturated bytes (dq >= 127), in a
    # middle strip; and a hot strip that is only the first or only the last strip
    for dq in (-129, -128, -127, -126, 126, 127, 128, 400):
        out.append(quad_bound_design("quad_dq_%s" % str(dq).replace("-", "m"), 4, dq))
    n_strips = len(strip_rows(H, W)) - 1
    out.append(quad_bound_design("quad_first_strip", 0, -127))
    out.append(quad_bound_design("quad_last_strip", n_strips - 1, 127))
    # ---- no foreground: a range below bt (ith >= 255), a constant offset (gmx == gmn)
    out.append(Design("no_fg_low_range", _frames(grid(40, y0=40), 8), BT, lambda r: r["ith"] >= 255 and r["ncomp"] == 0))
    out.append(Design("no_fg_offset", _frames(np.ones((H, W), np.uint8), 50), BT, lambda r: r["flat"] and r["ncomp"] == 0))
    # ---- the single kernel's work lists: well under and well over kListCap marked groups
    out.append(design("list_under", points([(40, 40), (80, 120)]), POINTS, lambda r: r["marked"] < kListCap // 2))
    p = points([(y, x) for y in range(3, H - 2, 8) for x in range(4, W - 4, 16)])
    out.append(design("list_over", p, POINTS, lambda r: r["marked"] > 2 * kListCap and r["ncomp"] == 150))
    return out


def small_designs(h, w):
    """A few designs at another geometry (edges, word boundaries, over 255 components)."""
    out = []
    p = points([(0, 3), (1, w // 2), (h - 2, 5), (h - 1, w - 1), (h // 2, 0), (h // 2 + 3, w - 2)], h, w)
    out.append(design("edges_%dx%d" % (w, h), p, POINTS,
                      lambda r: r["mask"][0].any() and r["mask"][1].any() and r["mask"][h - 1].any() and r["mask"][:, 0].any()
                      and r["mask"][:, w - 4:].any()))
    p = np.zeros((h, w), np.uint8)
    for xb in range(32, w, 32):
        p[4, xb - 1] = 1                                         # (DILATE: a run xb - 3 .. xb + 1)
        p[h // 3, xb - 3] = p[h // 3 + 5, xb + 2] = 1            # squares that meet corner to corner across xb
        p[2 * h // 3, xb + 2] = p[2 * h // 3 + 5, xb - 3] = 1    # ... the other diagonal
    out.append(design("words_%dx%d" % (w, h), p, DILATE, lambda r: len(r["words"]) == (w - 1) // 32 and all(a and b for a, b in r["words"])))
    out.append(design("slots_300_%dx%d" % (w, h), grid(300, y0=1, h=h, w=w, stagger=True), POINTS, lambda r: r["ncomp"] == 300))
    return out
