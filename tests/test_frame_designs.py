"""The designed clips of tests/frame_designs.py without a GPU: every design reaches the side of the kernel switch it claims
(measured on the C oracle's outputs), and on every designed frame the oracle's mask chain equals OpenCV's."""
import numpy as np
import pytest

from tests import frame_designs as fd

DESIGNS = fd.designs() + fd.small_designs(40, 152) + fd.small_designs(64, 80)
IDS = [d.name for d in DESIGNS]


@pytest.mark.parametrize("d", DESIGNS, ids=IDS)
def test_design_reaches_its_switch(d):
    r = fd.reach(d)
    assert d.claim(r), {k: v for k, v in r.items() if k not in ("mask", "labels", "hot_rows")}


def test_both_sides_of_every_switch_are_designed():
    r = {d.name: fd.reach(d) for d in DESIGNS}
    assert [r["lean_%d" % n]["ncomp"] for n in (31, 32, 33)] == [31, 32, 33]
    for name in ("runs_short", "runs_tall"):
        fits, over = r[name + "_rpr"], r[name + "_rpr_plus1"]
        assert fits["max_runs"] == fits["rpr"] and over["max_runs"] == over["rpr"] + 1
        assert fits["ncomp"] <= fd.kLeanSlots and over["ncomp"] <= fd.kLeanSlots
    assert r["runs_tall_rpr"]["extent"][0] <= 3 and r["runs_tall_rpr"]["extent"][1] >= 116
    assert [r["slots_%d" % n]["ncomp"] for n in (254, 255, 256, 600)] == [254, 255, 256, 600]
    assert len(r["band_span_24"]["bands"]) == 1 and len(r["band_span_25"]["bands"]) == 2
    assert sorted(b["bands"][1][0] - b["bands"][0][1] for k, b in r.items() if k.startswith("band_gap_")) == [1, 2, 3, 4, 5, 6]
    assert len(r["band_full_height"]["bands"]) >= 5
    m = r["edges_points"]["mask"] | r["edges_blocks"]["mask"]
    assert m[0].any() and m[1].any() and m[-2].any() and m[-1].any() and m[:, 0].any() and m[:, -4:].any()
    assert r["no_fg_low_range"]["ith"] >= 255 and r["no_fg_offset"]["flat"]
    assert r["list_under"]["marked"] < fd.kListCap // 2 and r["list_over"]["marked"] > 2 * fd.kListCap
    assert sorted(r[k]["dq"][4] for k in r if k.startswith("quad_dq_")) == [-129, -128, -127, -126, 126, 127, 128, 400]
    assert r["quad_first_strip"]["hot_strips"] == [0] and r["quad_last_strip"]["hot_strips"] == [len(fd.strip_rows(fd.H, fd.W)) - 2]


def test_word_boundary_designs_cross_every_word():
    # a run across xb - 1 | xb, and somewhere a pixel whose only link is diagonal across the boundary, at every xb
    d = next(d for d in DESIGNS if d.name == "word_boundaries")
    assert fd.reach(d)["words"] == [(True, True)] * 4


def test_label_order_designs_rank_a_lower_row_first():
    """In label_order_rows, each pair's lower, left component has the smaller label although its first pixel comes later in
    raster order."""
    d = next(d for d in DESIGNS if d.name == "label_order_rows")
    lab = fd.reach(d)["labels"].astype(np.int32)
    later_first = 0
    for lbl in range(1, lab.max() + 1):
        ys, xs = np.nonzero(lab == lbl)
        first = (ys.min(), xs[ys == ys.min()].min())
        for other in range(lbl + 1, lab.max() + 1):
            oy, ox = np.nonzero(lab == other)
            if (oy.min(), ox[oy == oy.min()].min()) < first:
                later_first += 1
    assert later_first == 6


@pytest.mark.parametrize("d", DESIGNS, ids=IDS)
def test_oracle_mask_chain_equals_opencv(d):
    """blur5 / threshold_close / cc8 of the oracle against OpenCV on the designed frame (int32 labels: more than 255 components
    are compared too)."""
    cv2 = pytest.importorskip("cv2")
    from oracle import oracle as orc

    o = fd.run_oracle(d)
    t = len(d.frames) - 1
    u, th = o["u"][t], float(o["thresh"][t])
    blurred = orc.blur5(u)
    assert np.array_equal(blurred, cv2.GaussianBlur(u, (5, 5), 0))
    _, m = cv2.threshold(cv2.GaussianBlur(u, (5, 5), 0), th, 255, cv2.THRESH_BINARY)
    m = cv2.morphologyEx(m, cv2.MORPH_CLOSE, (5, 5))
    mask = orc.threshold_close(blurred, th)
    assert np.array_equal(mask * 255, m)
    n, labels, comp = orc.cc8(mask)
    n2, l2, s2, c2 = cv2.connectedComponentsWithStats(m, ltype=cv2.CV_32S)
    assert n + 1 == n2 and n == o["ncomp"][t]
    assert np.array_equal(labels, l2)
    s, c = orc.stats_centroids_from_comp(comp)
    assert np.array_equal(s, s2[1:])
    assert np.array_equal(c, c2[1:])
    assert np.array_equal(np.minimum(labels, 255).astype(np.uint8), o["labels"][t])
