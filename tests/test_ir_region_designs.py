"""The designed frames of tests/ir_region_designs.py reach what they claim, checked with cv2 alone (no GPU), and the host
derives merge_components' limits from ``scale`` with Python's semantics."""
import numpy as np
import pytest

from tests import ir_region_designs as ird

cv2 = pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def frames():
    return ird.designs()


def block_key(x, y):
    return (y >> 1) * ((ird.W + 1) >> 1) + (x >> 1)


def first_blocks(labels, n):
    """Least 2x2 block key and raster-first pixel of every label 1..n-1."""
    keys, first = {}, {}
    ys, xs = np.nonzero(labels)
    for y, x in zip(ys, xs):  # raster order
        lab = int(labels[y, x])
        first.setdefault(lab, (int(x), int(y)))
        keys[lab] = min(keys.get(lab, 1 << 62), block_key(int(x), int(y)))
    return keys, first


def test_empty_and_all_foreground(frames):
    n, _, stats = ird.cv2_components(frames["empty"])
    assert n == 1 and stats[0].tolist() == [0, 0, ird.W, ird.H, ird.W * ird.H]
    n, _, stats = ird.cv2_components(frames["all_foreground"])
    assert n == 2 and stats[0].tolist() == [-1, ird.INT_MAX, 0, 0, 0]
    assert stats[1].tolist() == [0, 0, ird.W, ird.H, ird.W * ird.H]


def test_one_row_features_vanish(frames):
    assert frames["one_row"].any()
    assert ird.cv2_components(frames["one_row"])[0] == 1


def test_edges(frames):
    n, labels, stats = ird.cv2_components(frames["edges"])
    rows = stats[1:]
    assert (rows[:, 0] == 0).any() and (rows[:, 1] == 0).any()
    assert (rows[:, 0] + rows[:, 2] == ird.W).any() and (rows[:, 1] + rows[:, 3] == ird.H).any()
    # a feature in input row 0 only survives as rows 0-1; one in input row 1 only is removed
    assert any(r[1] == 0 and r[3] == 2 and r[0] == 100 for r in rows.tolist())
    assert not labels[:, 500:520].any()
    assert labels[0, 0] and labels[0, ird.W - 1] and labels[ird.H - 1, 0] and labels[ird.H - 1, ird.W - 1]


def test_first_pixel_off_block(frames):
    n, labels, _ = ird.cv2_components(frames["first_pixel_off_block"])
    assert n == 2
    keys, first = first_blocks(labels, n)
    assert first[1] == (3, 10) and block_key(*first[1]) != keys[1] and keys[1] == block_key(0, 11)


def test_interleaved_blocks(frames):
    n, labels, _ = ird.cv2_components(frames["interleaved_blocks"])
    assert n == 1 + 4 + 24
    keys, first = first_blocks(labels, n)
    labs = sorted(keys)
    # OpenCV numbers by least block key, and that order differs from the raster order of the first pixels
    assert [keys[lab] for lab in labs] == sorted(keys.values())
    assert sorted(labs, key=lambda lab: (first[lab][1], first[lab][0])) != labs
    assert labels[21, 14] < labels[20, 20]  # Q before S
    # block rows of P, Q, R, S interleave: every block row 10..12 holds blocks of at least three of them
    for br in (10, 11, 12):
        assert len({int(v) for v in np.unique(labels[2 * br : 2 * br + 2, 8:24]) if v}) >= 3


def test_dot_grid(frames):
    n, _, stats = ird.cv2_components(frames["dot_grid"])
    assert n - 1 == ird.DOT_GRID_COMPONENTS
    assert stats[1].tolist() == [0, 0, 1, 3, 3]  # row 0 joins rows 1-2


@pytest.mark.parametrize("scale,want", ird.merge_limits_cases())
def test_merge_limits(scale, want):
    from classifier_pipeline_b200.track.irtrackextractor import merge_limits

    got = merge_limits(scale)
    assert got == want and [type(v) for v in got[:2]] == [int, int]
