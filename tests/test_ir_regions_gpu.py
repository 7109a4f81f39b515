"""Components and rectangle merging of whole IR clips on the device (cpt_detect_objects_batch, cpt_ir_merge_components,
track.irtrackextractor.detect_ir_regions_batch / ir_clip_regions) against the per-frame composition with live cv2 (MOG2,
open, threshold, connectedComponentsWithStats) followed by merge_components.  Everything bit-exact."""
import os

import numpy as np
import pytest

from tests import helpers, ir_helpers
from tests import ir_region_designs as ird

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _ctx():
    from classifier_pipeline_b200 import engine

    eng = engine.get_engine()
    eng.ctx.use_torch_stream()
    return eng


def native_batch(frames, max_components, scale=None, threshold=0):
    """One cpt_detect_objects_batch + cpt_ir_merge_components call: host (counts, stats rows, labels, merged rows,
    merged counts), with the rows cut to each frame's count."""
    import torch

    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.track.irtrackextractor import merge_limits

    eng = _ctx()
    d = torch.from_numpy(np.ascontiguousarray(frames)).to(eng.device)
    n, h, w = d.shape
    i32 = dict(dtype=torch.int32, device=eng.device)
    counts, stats = torch.empty(n, **i32), torch.empty((n, max_components + 1, 5), **i32)
    cents, labels = torch.empty((n, max_components + 1, 2), dtype=torch.float64, device=eng.device), torch.empty((n, h, w), **i32)
    eng.ctx.detect_objects_batch(d, n, w, h, threshold, native.DETECT_OPEN_GRAY, max_components, counts, stats, cents, labels)
    mcounts, merged = torch.empty(n, **i32), torch.empty((n, max_components, 5), **i32)
    eng.ctx.ir_merge_components(stats, counts, n, max_components, *merge_limits(scale), merged, mcounts)
    counts, stats, cents, labels = counts.cpu().numpy(), stats.cpu().numpy(), cents.cpu().numpy(), labels.cpu().numpy()
    mcounts, merged = mcounts.cpu().numpy(), merged.cpu().numpy()
    rows = [stats[t, : min(counts[t], max_components + 1)] for t in range(n)]
    cent = [cents[t, : min(counts[t], max_components + 1)] for t in range(n)]
    return counts, rows, cent, labels, [merged[t, : max(mcounts[t], 0)] for t in range(n)], mcounts


def assert_frame(got_n, got_labels, got_stats, got_merged, gray, scale=None, what=""):
    n, labels, stats, merged = ird.cv2_regions(gray, scale=scale)
    assert got_n == n, what
    if got_labels is not None:
        assert np.array_equal(got_labels, labels), what
    assert np.array_equal(got_stats, stats), what
    assert np.array_equal(np.asarray(got_merged).reshape(-1, 5), merged), what


SCHEDULE = "schedule"


@pytest.mark.parametrize("shape,frames,seed,lr", [((480, 640), 40, 0, -1), ((120, 160), 60, 1, -1), ((61, 97), 60, 2, -1),
                                                   ((120, 160), 70, 3, SCHEDULE)])
def test_clip_regions_match_cv2(shape, frames, seed, lr):
    """ir_clip_regions == per frame: cv2 MOG2 -> open -> threshold -> components -> merge_components; the labels of the
    same masks through detect_ir_regions_batch too."""
    from classifier_pipeline_b200.track.cliptracker import MOG2Background
    from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions_batch, ir_clip_regions

    clip = ird.ir_gray_clip(seed, frames, shape)
    if lr == SCHEDULE:  # automatic, then rate 0 over a span, a re-initialisation, automatic again
        lr = np.full(frames, -1.0)
        lr[20:35] = 0
        lr[40] = 1
        lr[50:55] = 0.3
    lrs = np.full(frames, float(lr)) if np.isscalar(lr) else lr
    masks = ird.cv2_masks(clip, lrs)
    stats, merged = ir_clip_regions(clip, MOG2Background(), learning_rate=lr)
    st2, mg2, labels = detect_ir_regions_batch(masks, labels=True)
    assert len(stats) == len(merged) == frames
    busy = kept = 0
    for t in range(frames):
        n, lab, st, mg = ird.cv2_regions(masks[t])
        assert np.array_equal(stats[t], st) and np.array_equal(merged[t], mg), t
        assert np.array_equal(st2[t], st) and np.array_equal(mg2[t], mg) and np.array_equal(labels[t], lab), t
        busy += n > 2
        kept += len(mg) > 0
    assert busy > frames // 4  # the clip is not trivial: several components on many frames
    assert kept > frames // 4 or shape[0] < 120  # at 61x97 the objects are smaller than the merge's filter keeps
    # device input: the masks stay on the device
    import torch

    stats_d, merged_d = ir_clip_regions(torch.from_numpy(clip).cuda(), MOG2Background(), learning_rate=lr)
    assert all(np.array_equal(a, b) for a, b in zip(stats_d, stats)) and all(np.array_equal(a, b) for a, b in zip(merged_d, merged))


def test_batch_equals_single_image_and_golden():
    from classifier_pipeline_b200.ml_tools.imageprocessing import detect_objects_ir
    from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions, detect_ir_regions_batch

    gold = np.load(os.path.join(helpers.GOLDEN, "ir.npz"))
    frames = np.stack([ir_helpers.ir_filtered(s) for s in range(4)])
    stats, merged, labels = detect_ir_regions_batch(frames, labels=True)
    for s in range(4):
        assert len(stats[s]) == int(gold["ir{}_n".format(s)])
        assert np.array_equal(labels[s], gold["ir{}_labels".format(s)])
        assert np.array_equal(stats[s], gold["ir{}_stats".format(s)])
        assert np.array_equal(merged[s], gold["ir{}_merged".format(s)])
        lab1, mg1 = detect_ir_regions(frames[s])
        _, _, st1 = detect_objects_ir(frames[s], threshold=0)
        assert np.array_equal(labels[s], lab1) and np.array_equal(stats[s], st1)
        assert np.array_equal(merged[s], np.array(mg1).reshape(-1, 5))


def test_designed_frames_in_one_batch():
    names = list(ird.designs())
    frames = np.stack([ird.designs()[k] for k in names])
    counts, stats, cents, labels, merged, mcounts = native_batch(frames, 60000)
    for t, name in enumerate(names):
        assert_frame(counts[t], labels[t], stats[t], merged[t], frames[t], what=name)
        n, _, _, c = cv2.connectedComponentsWithStats(cv2.threshold(cv2.morphologyEx(frames[t], cv2.MORPH_OPEN, (15, 15)), 0, 255,
                                                                                  cv2.THRESH_BINARY)[1])
        assert np.array_equal(cents[t], c, equal_nan=True), name
    fg = names.index("all_foreground")
    assert stats[fg][0].tolist() == [-1, ird.INT_MAX, 0, 0, 0] and np.isnan(cents[fg][0]).all()
    assert counts[names.index("dot_grid")] - 1 == ird.DOT_GRID_COMPONENTS


def test_dot_grid_at_and_below_its_count():
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions_batch

    grid = ird.dot_grid()
    frames = np.stack([grid, ir_helpers.ir_filtered(0), grid])
    n_true = ird.DOT_GRID_COMPONENTS + 1
    _, labels_cv, stats_cv, _ = ird.cv2_regions(grid)
    for mc in (ird.DOT_GRID_COMPONENTS, ird.DOT_GRID_COMPONENTS - 1):
        counts, stats, _, labels, merged, mcounts = native_batch(frames, mc)
        assert counts[0] == counts[2] == n_true
        assert np.array_equal(labels[0], labels_cv) and np.array_equal(labels[2], labels_cv)
        assert np.array_equal(stats[0], stats_cv[: mc + 1])  # the first max_components components, in label order
        assert_frame(counts[1], labels[1], stats[1], merged[1], frames[1], what="frame after the grid")
        if mc == ird.DOT_GRID_COMPONENTS:
            assert mcounts[0] == 0  # every dot is filtered out
        else:
            assert mcounts[0] == mcounts[2] == -1  # truncated lists are never merged
    with pytest.raises(native.NativeError, match="frame 0"):
        detect_ir_regions_batch(frames)


# ---- merge lists straight into the merge kernel ----

def merge_on_device(lists, scale=None, max_components=None):
    import torch

    from classifier_pipeline_b200.track.irtrackextractor import merge_limits

    eng = _ctx()
    mc = max_components or max(1, max(len(r) for r in lists))
    stats = np.zeros((len(lists), mc + 1, 5), np.int32)
    counts = np.array([len(r) + 1 for r in lists], np.int32)
    for t, r in enumerate(lists):
        if len(r):
            stats[t, 1 : len(r) + 1] = r
    d_stats, d_counts = torch.from_numpy(stats).to(eng.device), torch.from_numpy(counts).to(eng.device)
    merged = torch.full((len(lists), mc, 5), -7, dtype=torch.int32, device=eng.device)
    mcounts = torch.empty(len(lists), dtype=torch.int32, device=eng.device)
    eng.ctx.ir_merge_components(d_stats, d_counts, len(lists), mc, *merge_limits(scale), merged, mcounts)
    merged, mcounts = merged.cpu().numpy(), mcounts.cpu().numpy()
    return [merged[t, : mcounts[t]] for t in range(len(lists))]


def python_merge(rows, scale=None):
    from classifier_pipeline_b200.track.irtrackextractor import merge_components

    return np.array(merge_components([np.array(r, np.int32) for r in rows], scale=scale), np.int32).reshape(-1, 5)


def random_rows(rng, n, span=(640, 480), size=60):
    x, y = rng.integers(0, span[0], n), rng.integers(0, span[1], n)
    w, h = rng.integers(1, size, n), rng.integers(1, size, n)
    area = np.maximum(1, (rng.random(n) * w * h).astype(np.int64))
    return np.stack([x, y, w, h, area], 1).astype(np.int32)


def designed_lists():
    lists = {
        "empty": np.zeros((0, 5), np.int32),
        # equal areas: the stable sort keeps label order among them
        "equal_areas": np.array([[0, 0, 10, 10, 100], [200, 0, 10, 10, 100], [30, 0, 10, 10, 100], [230, 0, 10, 10, 100],
                                 [400, 300, 10, 10, 100], [60, 0, 9, 9, 100]], np.int32),
        # equal x: pairs with the same x are never compared, even when they overlap
        "equal_x": np.array([[50, 50, 20, 20, 400], [50, 60, 20, 20, 300], [50, 300, 20, 20, 200], [75, 55, 5, 5, 90],
                             [50, 85, 10, 10, 100]], np.int32),
        # a chain: each rectangle is within the gap of the next only, so merges restart the scan repeatedly
        "chain": np.array([[i * 45, (i % 3) * 7, 12, 12, 50 + (i * 37) % 90] for i in range(14)], np.int32),
        # the filter: mass just over and at min_mass, sides just over and at min_size
        "filter": np.array([[0, 0, 1, 1, 41], [100, 0, 1, 1, 40], [200, 0, 17, 17, 5], [300, 0, 16, 17, 5], [400, 0, 17, 16, 5]],
                           np.int32),
    }
    # squared gaps of 1597 (1599 is not a sum of two squares), 1600 and 1601 against max_gap 40
    for name, (dx, dy) in {"d2_1597": (34, 21), "d2_1600": (40, 0), "d2_1601": (40, 1)}.items():
        lists[name] = np.array([[0, 0, 10, 10, 100], [10 + dx, 10 + dy if dy else 0, 10, 10, 90]], np.int32)
    return lists


def test_merge_designed_lists():
    lists = designed_lists()
    assert (lambda r: ((r[1][0] - 10) ** 2 + (r[1][1] - 10) ** 2))(lists["d2_1601"]) == 1601
    assert len(python_merge(lists["d2_1597"])) == 1 and len(python_merge(lists["d2_1600"])) == 2
    assert len(python_merge(lists["chain"])) < len(lists["chain"]) - 3
    got = merge_on_device(list(lists.values()))
    for (name, rows), g in zip(lists.items(), got):
        assert np.array_equal(g, python_merge(rows)), name


@pytest.mark.parametrize("scale", [None, 0.5, 1.5])
def test_merge_random_lists(scale):
    rng = np.random.default_rng(7 if scale is None else int(scale * 10))
    lists = [random_rows(rng, int(rng.integers(0, 60)), size=50) for _ in range(60)]
    got = merge_on_device(lists, scale=scale)
    merges = 0
    for t, (rows, g) in enumerate(zip(lists, got)):
        want = python_merge(rows, scale)
        assert np.array_equal(g, want), t
        merges += len(want) < len(rows)
    assert merges > 10


def test_merge_long_lists():
    """Lists of hundreds of rectangles: the filter, the sort, the scan and the compaction each take many 32-wide passes."""
    from classifier_pipeline_b200.track.irtrackextractor import merge_limits

    rng = np.random.default_rng(11)
    lists = []
    for k in range(3):
        far = random_rows(rng, 260, span=(20000, 20000), size=40)
        cluster = random_rows(rng, 40, span=(300, 300), size=40)
        rows = np.concatenate([far, cluster])
        rows[::7, 4] = rows[3, 4]  # many equal areas
        lists.append(rng.permutation(rows))
    mm, ms, _ = merge_limits()
    for rows in lists:
        assert ((rows[:, 4] > mm) | ((rows[:, 2] > ms) & (rows[:, 3] > ms))).sum() > 4 * 32
    got = merge_on_device(lists, max_components=400)
    for rows, g in zip(lists, got):
        want = python_merge(rows)
        assert np.array_equal(g, want)
        assert len(want) > 64 and len(want) < ((rows[:, 4] > mm) | ((rows[:, 2] > ms) & (rows[:, 3] > ms))).sum()


# ---- call shapes ----

def test_calls_longer_than_a_chunk_and_big_then_small():
    """640x480 frames take about 3.4 MB of scratch each, so 100 frames span two chunks of the 256 MB bound."""
    from classifier_pipeline_b200.track.irtrackextractor import detect_ir_regions, detect_ir_regions_batch

    clip = ird.ir_gray_clip(5, 100)
    masks = ird.cv2_masks(clip, np.full(100, -1.0))
    stats, merged, labels = detect_ir_regions_batch(masks, labels=True)
    for t in range(100):
        assert_frame(len(stats[t]), labels[t], stats[t], merged[t], masks[t], what=t)
    small = ird.ir_gray_clip(6, 3, (61, 97))
    st_s, mg_s, lab_s = detect_ir_regions_batch(small, labels=True)
    for t in range(3):
        assert_frame(len(st_s[t]), lab_s[t], st_s[t], mg_s[t], small[t], what=("small", t))
        lab1, mg1 = detect_ir_regions(small[t])
        assert np.array_equal(lab1, lab_s[t]) and np.array_equal(np.array(mg1).reshape(-1, 5), mg_s[t])
    st_e, mg_e = detect_ir_regions_batch(np.zeros((0, 61, 97), np.uint8))
    assert st_e == [] and mg_e == []


def test_rejected_inputs_leave_the_context_usable():
    import torch

    from classifier_pipeline_b200 import native

    eng = _ctx()
    lib, h = eng.ctx.lib, eng.ctx._h
    d = torch.zeros((2, 8, 8), dtype=torch.uint8, device=eng.device)
    counts = torch.empty(2, dtype=torch.int32, device=eng.device)
    stats = torch.empty((2, 5, 5), dtype=torch.int32, device=eng.device)
    merged = torch.empty((2, 4, 5), dtype=torch.int32, device=eng.device)
    p = lambda t: t.data_ptr()  # noqa: E731
    ok = (h, p(d), 2, 8, 8, 0.0, native.DETECT_OPEN_GRAY, 4, p(counts), p(stats), None, None)

    def det(**kw):
        args = list(ok)
        for k, v in kw.items():
            args[["h", "frames", "n", "w", "h_", "thr", "steps", "mc", "counts", "stats", "cents", "labels"].index(k)] = v
        return lib.cpt_detect_objects_batch(*args)

    assert det(h=None) == -1 and det(frames=None) == -1 and det(counts=None) == -1 and det(stats=None) == -1
    assert det(n=-1) == -1 and det(w=0) == -1 and det(h_=0) == -1 and det(w=1 << 14, h_=1 << 13) == -1 and det(mc=0) == -1
    assert det(steps=native.DETECT_CLOSE) == -3 and det(steps=native.DETECT_OPEN_GRAY | native.DETECT_OTSU) == -3
    assert det(steps=native.DETECT_MASK_ONLY) == -3
    assert det(n=0) == 0 and det(steps=0) == 0
    m = lambda **kw: lib.cpt_ir_merge_components(kw.get("h", h), kw.get("stats", p(stats)), kw.get("counts", p(counts)), kw.get("n", 2),  # noqa: E731
                                                kw.get("mc", 4), 40, 16, 40.0, kw.get("merged", p(merged)), kw.get("mcounts", p(counts)))
    assert m(h=None) == -1 and m(stats=None) == -1 and m(counts=None) == -1 and m(merged=None) == -1 and m(mcounts=None) == -1
    assert m(n=-1) == -1 and m(mc=0) == -1 and m(n=0) == 0
    # still usable
    frames = np.stack([ir_helpers.ir_filtered(1)])
    counts_, stats_, _, labels_, merged_, _ = native_batch(frames, 8192)
    assert_frame(counts_[0], labels_[0], stats_[0], merged_[0], frames[0])


def test_all_foreground_single_image():
    """cv2 reports the empty background row of an all-foreground image as [-1, INT_MAX, 0, 0, 0] with a NaN centroid."""
    from classifier_pipeline_b200.ml_tools.imageprocessing import detect_objects, detect_objects_ir

    for shape in ((1, 1), (61, 97), (480, 640)):
        img = np.full(shape, 255, np.uint8)
        n, labels, stats = detect_objects_ir(img, threshold=0)
        want_n, want_labels, want_stats = ird.cv2_components(img)
        assert n == want_n == 2 and np.array_equal(labels, want_labels) and np.array_equal(stats, want_stats), shape
        n, labels, stats, cents = detect_objects(img.astype(np.float64), threshold=0, kernel=(3, 3))
        assert stats[0].tolist() == [-1, ird.INT_MAX, 0, 0, 0] and np.isnan(cents[0]).all(), shape
