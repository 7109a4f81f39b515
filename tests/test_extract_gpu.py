"""Parity of the CUDA extraction kernel (through the C ABI) with the C oracle and with the
reference's golden fixtures.  Bit-exact: filtered frames (hence every per-frame background),
normalisation scalars, thresholds, label images, component stats, final WeightedBackground
state.  Tolerance class: per-region variance (fp64 sums on both sides, one-pass on the device;
rel 1e-6) and vs the reference's fp32 np.var (rel 2e-4)."""
import numpy as np
import pytest

from tests import helpers

pytestmark = pytest.mark.gpu

RAW = ["possum_raw", "hedgehog_raw", "synth0_raw", "synth1_raw", "synth2_raw", "synth3_raw"]


@pytest.fixture(scope="module")
def extractor():
    from classifier_pipeline_b200.batch import BatchExtractor

    return BatchExtractor(device=0, max_regions=32)


def _run_device(extractor, init, tracked, bt, weight_add, flags=None, keep_state=True):
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips

    frames = np.concatenate([init[None], tracked])
    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    slot = extractor.ctx.weight_table(weight_add, max_frames=4096)
    clips = linear_clips([len(tracked)], bt, slot, flags=native.CLIP_UPDATE_BACKGROUND if flags is None else flags)
    clips["frame_offset"] = 1
    clips["init_offset"] = 0
    clips["out_offset"] = 0
    # (with or without a state record the launch takes the split plan -- sweep kernel + per-frame kernels -- unless the
    # `plan` fixture forces the single persistent kernel)
    out = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=keep_state, out={})
    torch.cuda.synchronize()
    return out


def _compare_with_oracle(extractor, out, o, T, slot_weight_add, with_state=True):
    regions = extractor.regions_numpy(out["regions"])[:T]
    info = extractor.info_numpy(out["info"])[:T]
    assert np.array_equal(out["filtered"][:T].cpu().numpy(), o["filtered"])
    assert np.array_equal(info["background_average"], o["avg"])
    assert np.array_equal(info["threshold"], o["thresh"])
    assert np.array_equal(info["norm_max"].astype(np.float32), o["norm"][:, 0])
    assert np.array_equal(info["norm_min"].astype(np.float32), o["norm"][:, 1])
    assert np.array_equal(info["n_components"], o["ncomp"])
    assert np.array_equal(out["labels"][:T].cpu().numpy(), o["labels"])
    for t in range(T):
        n = int(o["ncomp"][t])
        r = regions[t, :n]
        got = np.stack([r["x"], r["y"], r["width"], r["height"], r["area"], r["sum_x"], r["sum_y"], r["key"]], axis=1)
        assert np.array_equal(got, o["comp"][t, :n]), t
        np.testing.assert_allclose(r["pixel_variance"], o["var"][t, :n], rtol=1e-6, atol=1e-6)
    if not with_state:
        return
    st = extractor.ctx.state_read(out["state"], 0)
    assert np.array_equal(st["background"], o["final_bg"])
    assert st["average"] == o["final_avg"]
    slot = extractor.ctx.weight_table(slot_weight_add, max_frames=4096)
    weights = np.array([extractor.ctx.weight_value(slot, int(k)) for k in range(int(st["weight_count"].max()) + 1)])
    assert np.array_equal(weights[st["weight_count"]], o["final_weight"])
    assert st["frames_seen"] == T


@pytest.fixture(params=["split", "single"])
def plan(request, extractor):
    """Both launch plans of DESIGN.md section 3.1: batch launches that keep the filtered images take the split plan unless the
    ctx is told to run the single persistent kernel."""
    extractor.ctx.force_single_kernel(request.param == "single")
    yield request.param
    extractor.ctx.force_single_kernel(False)


@pytest.mark.parametrize("name", RAW)
def test_kernel_matches_oracle_and_reference(extractor, name, plan):
    from oracle import oracle as orc

    d, meta = helpers.load_golden(name)
    init, tracked = helpers.clip_input(name)
    T = len(tracked)
    p = orc.make_params(background_thresh=meta["background_thresh"], weight_add=meta["weight_add"], max_comp=32)
    o = orc.extract_clip(tracked, init, p)
    out = _run_device(extractor, init, tracked, meta["background_thresh"], meta["weight_add"])
    _compare_with_oracle(extractor, out, o, T, meta["weight_add"])
    # and directly against what the reference produced
    assert np.array_equal(out["labels"][:T].cpu().numpy(), d["labels"])
    bg = helpers.golden_background(d)
    assert np.array_equal(out["filtered"][:T].cpu().numpy(), (tracked.astype(np.int64) - bg).astype(np.float32))
    regions = extractor.regions_numpy(out["regions"])[:T]
    for t, (gs, gc) in enumerate(helpers.golden_components(d)):
        r = regions[t, : len(gs)]
        assert np.array_equal(np.stack([r["x"], r["y"], r["width"], r["height"], r["area"]], axis=1), gs)
        cents = np.stack([r["sum_x"] / r["area"].astype(np.float64), r["sum_y"] / r["area"].astype(np.float64)], axis=1)
        assert np.array_equal(cents, gc)
    for row in d["regions"]:
        t, rid, var = int(row[0]), int(row[7]), row[6]
        assert regions[t, rid]["pixel_variance"] == pytest.approx(var, rel=2e-4, abs=1e-4)


@pytest.mark.parametrize("name", RAW)
def test_split_path_matches_oracle_and_reference(extractor, name):
    """The same clips through the split path (no state record: extract_sweep_kernel + frame_regions_kernel +
    frame_components_kernel + region_variance_kernel)."""
    from oracle import oracle as orc

    d, meta = helpers.load_golden(name)
    init, tracked = helpers.clip_input(name)
    T = len(tracked)
    p = orc.make_params(background_thresh=meta["background_thresh"], weight_add=meta["weight_add"], max_comp=32)
    o = orc.extract_clip(tracked, init, p)
    out = _run_device(extractor, init, tracked, meta["background_thresh"], meta["weight_add"], keep_state=False)
    _compare_with_oracle(extractor, out, o, T, meta["weight_add"], with_state=False)
    assert np.array_equal(out["labels"][:T].cpu().numpy(), d["labels"])
    bg = helpers.golden_background(d)
    assert np.array_equal(out["filtered"][:T].cpu().numpy(), (tracked.astype(np.int64) - bg).astype(np.float32))


def test_split_and_single_kernel_paths_agree_on_a_ragged_batch(extractor):
    """Both launch plans, same ragged batch (empty clip, one-frame clip, clips around the 45-frame window, unused output
    frames between clips): every output identical, variances included."""
    import torch
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.synthetic import clip_model, make_clip

    lengths = [50, 0, 17, 64, 1, 46, 45, 90, 2, 131]
    pix = [make_clip(40 + i, frames=max(n, 1))[0][:n] for i, n in enumerate(lengths)]
    frames = np.concatenate([p for p in pix if len(p)])
    bts = np.array([clip_model(40 + i)[2] for i in range(len(lengths))])
    slots = np.array([extractor.ctx.weight_table(clip_model(40 + i)[3], max_frames=4096) for i in range(len(lengths))])
    clips = linear_clips(lengths, bts, slots)
    clips["out_offset"] += 3 * np.arange(len(lengths))  # gaps: output frames no clip writes
    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    outs = []
    try:
        for single in (True, False):
            extractor.ctx.force_single_kernel(single)
            o = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=True, out={})
            torch.cuda.synchronize()
            outs.append(o)
    finally:
        extractor.ctx.force_single_kernel(False)
    a, b = outs
    # the saved per-clip records: background, counters (crop view), sliding sums, average, last filtered image
    npx = 160 * 120
    for i in range(len(lengths)):
        sa, sb = extractor.ctx.state_read(a["state"], i, sliding_sum=True), extractor.ctx.state_read(b["state"], i, sliding_sum=True)
        for f in ("background", "weight_count", "sliding_sum"):
            assert np.array_equal(sa[f], sb[f]), (i, f)
        assert sa["average"] == sb["average"] and sa["frames_seen"] == sb["frames_seen"], i
        if lengths[i]:
            fa_, fb_ = a["state"][i, 64 + 8 * npx :], b["state"][i, 64 + 8 * npx :]
            assert torch.equal(fa_, fb_), i
    ia, ib = extractor.info_numpy(a["info"]), extractor.info_numpy(b["info"])
    ra, rb = extractor.regions_numpy(a["regions"]), extractor.regions_numpy(b["regions"])
    fa, fb = a["filtered"].cpu().numpy(), b["filtered"].cpu().numpy()
    la, lb = a["labels"].cpu().numpy(), b["labels"].cpu().numpy()
    seen = 0
    for i, n in enumerate(lengths):
        o0 = int(clips["out_offset"][i])
        sl = slice(o0, o0 + n)
        assert np.array_equal(fa[sl], fb[sl]) and np.array_equal(la[sl], lb[sl]), i
        for f in ("threshold", "norm_min", "norm_max", "avg_change", "filtered_min", "filtered_max", "n_components", "thermal_sum", "background_average"):
            assert np.array_equal(ia[f][sl], ib[f][sl]), (i, f)
        for t in range(o0, o0 + n):
            k = min(int(ia["n_components"][t]), extractor.max_regions)
            seen += k
            for f in ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key", "pixel_variance"):
                assert np.array_equal(ra[t, :k][f], rb[t, :k][f]), (i, t, f)
    assert seen > 50


def test_batch_of_ragged_clips_matches_single_clip_runs(extractor, plan):
    """Clips are independent: a ragged batch (incl. an empty clip) equals per-clip oracle runs."""
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.synthetic import clip_model, make_clip
    from oracle import oracle as orc

    lengths = [50, 0, 17, 64, 1, 46, 45, 90]
    pix = [make_clip(10 + i, frames=max(n, 1))[0][:n] for i, n in enumerate(lengths)]
    frames = np.concatenate([p for p in pix if len(p)])
    bts = [clip_model(10 + i)[2] for i in range(len(lengths))]
    was = [clip_model(10 + i)[3] for i in range(len(lengths))]
    slots = [extractor.ctx.weight_table(w, max_frames=4096) for w in was]
    clips = linear_clips(lengths, np.array(bts), np.array(slots))
    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    out = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=True)
    torch.cuda.synchronize()
    regions = extractor.regions_numpy(out["regions"])
    info = extractor.info_numpy(out["info"])
    labels = out["labels"].cpu().numpy()
    filtered = out["filtered"].cpu().numpy()
    for i, n in enumerate(lengths):
        if n == 0:
            continue
        o0 = int(clips["out_offset"][i])
        p = orc.make_params(background_thresh=bts[i], weight_add=was[i], max_comp=32)
        o = orc.extract_clip(pix[i], pix[i][0], p)
        assert np.array_equal(filtered[o0 : o0 + n], o["filtered"]), i
        assert np.array_equal(labels[o0 : o0 + n], o["labels"]), i
        assert np.array_equal(info["n_components"][o0 : o0 + n], o["ncomp"]), i
        assert np.array_equal(info["threshold"][o0 : o0 + n], o["thresh"]), i
        for t in range(n):
            k = int(o["ncomp"][t])
            r = regions[o0 + t, :k]
            got = np.stack([r["x"], r["y"], r["width"], r["height"], r["area"], r["sum_x"], r["sum_y"], r["key"]], axis=1)
            assert np.array_equal(got, o["comp"][t, :k])
        st = extractor.ctx.state_read(out["state"], i)
        assert np.array_equal(st["background"], o["final_bg"]), i


def test_resume_equals_one_shot(extractor):
    """Streaming: running a clip in pieces with CPT_CLIP_RESUME reproduces the one-shot run."""
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.synthetic import make_clip

    pix, _ = make_clip(21, frames=120)
    d_frames = torch.from_numpy(pix.view(np.int16)).cuda().view(torch.uint16)
    slot = extractor.ctx.weight_table(1.0, max_frames=4096)
    clips = linear_clips([120], 50, slot)
    ref = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=True, out={})
    torch.cuda.synchronize()
    ref_regions = extractor.regions_numpy(ref["regions"]).copy()
    ref_labels = ref["labels"].cpu().numpy()
    state = None
    got_regions, got_labels = [], []
    pos = 0
    for piece in (1, 44, 3, 60, 12):
        c = linear_clips([piece], 50, slot, flags=native.CLIP_UPDATE_BACKGROUND | (native.CLIP_RESUME if pos else 0))
        c["frame_offset"] = 0
        c["init_offset"] = 0
        c["first_frame"] = pos
        c["ring_frames"] = 120  # frame t lives at slot t % 120 == t
        c["out_offset"] = 0
        o = extractor.extract_device(d_frames, c, keep_filtered=True, keep_labels=True, keep_state=True, d_state=state, out={})
        torch.cuda.synchronize()
        state = o["state"]
        got_regions.append(extractor.regions_numpy(o["regions"])[:piece].copy())
        got_labels.append(o["labels"][:piece].cpu().numpy())
        pos += piece
    got_regions = np.concatenate(got_regions)
    assert np.array_equal(np.concatenate(got_labels), ref_labels)
    for f in ("x", "y", "width", "height", "area", "sum_x", "sum_y"):
        # only compare live entries
        info = extractor.info_numpy(ref["info"])
        for t in range(120):
            n = min(int(info["n_components"][t]), extractor.max_regions)
            assert np.array_equal(got_regions[t, :n][f], ref_regions[t, :n][f])
    for t in range(120):
        n = min(int(extractor.info_numpy(ref["info"])["n_components"][t]), extractor.max_regions)
        assert np.array_equal(got_regions[t, :n]["pixel_variance"], ref_regions[t, :n]["pixel_variance"])


def test_host_staged_call_matches_device_call(extractor):
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.synthetic import make_clip

    pix = np.concatenate([make_clip(30 + i, frames=40)[0] for i in range(5)])
    slot0 = extractor.ctx.weight_table(0.1, max_frames=4096)
    slot1 = extractor.ctx.weight_table(1.0, max_frames=4096)
    clips = linear_clips([40] * 5, np.array([20, 50, 20, 50, 20]), np.array([slot0, slot1, slot0, slot1, slot0]))
    clips["flags"][3] |= native.CLIP_DENOISE  # (one clip of the default configuration: its chunk runs the denoise passes)
    d_frames = torch.from_numpy(pix.view(np.int16)).cuda().view(torch.uint16)
    dev = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, out={})
    torch.cuda.synchronize()
    host = extractor.extract_host(pix, clips, keep_filtered=True, keep_labels=True, chunk_clips=2)
    assert np.array_equal(host["labels"], dev["labels"].cpu().numpy())
    assert np.array_equal(host["filtered"], dev["filtered"].cpu().numpy())
    info_d = extractor.info_numpy(dev["info"])
    assert np.array_equal(host["info"]["n_components"], info_d["n_components"])
    assert np.array_equal(host["info"]["threshold"], info_d["threshold"])
    rd = extractor.regions_numpy(dev["regions"])
    for t in range(200):
        n = min(int(info_d["n_components"][t]), extractor.max_regions)
        for f in ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key"):
            assert np.array_equal(host["regions"][t, :n][f], rd[t, :n][f])
        assert np.array_equal(host["regions"][t, :n]["pixel_variance"], rd[t, :n]["pixel_variance"])


def test_extreme_frames(extractor):
    """Constant frames (degenerate normalisation), saturated values and dense noise masks."""
    import torch
    from classifier_pipeline_b200.batch import linear_clips
    from oracle import oracle as orc

    rng = np.random.default_rng(99)
    T = 12
    cases = {
        "constant": np.full((T, 120, 160), 3000, np.uint16),
        "zeros": np.zeros((T, 120, 160), np.uint16),
        "saturated": rng.choice(np.array([0, 65535], np.uint16), size=(T, 120, 160)),
        "noise": rng.integers(2000, 2400, size=(T, 120, 160)).astype(np.uint16),
        "steps": (np.arange(T)[:, None, None] * 300 + rng.integers(0, 30, size=(T, 120, 160))).astype(np.uint16),
    }
    slot = extractor.ctx.weight_table(0.1, max_frames=4096)
    for name, pix in cases.items():
        clips = linear_clips([T], 20, slot)
        d_frames = torch.from_numpy(pix.view(np.int16)).cuda().view(torch.uint16)
        out = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=True, out={})
        torch.cuda.synchronize()
        p = orc.make_params(background_thresh=20, weight_add=0.1, max_comp=255)
        o = orc.extract_clip(pix, pix[0], p)
        info = extractor.info_numpy(out["info"])[:T]
        assert np.array_equal(out["filtered"][:T].cpu().numpy(), o["filtered"]), name
        assert np.array_equal(info["threshold"], o["thresh"]), name
        assert np.array_equal(info["n_components"], o["ncomp"]), name
        if o["ncomp"].max() <= 255:
            assert np.array_equal(out["labels"][:T].cpu().numpy(), o["labels"]), name
        st = extractor.ctx.state_read(out["state"], 0)
        assert np.array_equal(st["background"], o["final_bg"]), name


@pytest.mark.parametrize("name", ["possum_nlm", "hedgehog_nlm", "synth4_nlm"])
def test_denoise_pipeline_matches_oracle_and_reference(extractor, name):
    """TrackingConfig.denoise=True (the reference's default): normalise -> cv2.fastNlMeansDenoising -> blur ->
    threshold -> close -> components as device passes; labels / stats bit-exact vs the oracle and the reference."""
    from classifier_pipeline_b200 import native
    from oracle import oracle as orc

    d, meta = helpers.load_golden(name)
    init, tracked = helpers.clip_input(name)
    T = len(tracked)
    p = orc.make_params(background_thresh=meta["background_thresh"], weight_add=meta["weight_add"], max_comp=32, denoise=True)
    o = orc.extract_clip(tracked, init, p)
    out = _run_device(extractor, init, tracked, meta["background_thresh"], meta["weight_add"],
                      flags=native.CLIP_UPDATE_BACKGROUND | native.CLIP_DENOISE)
    _compare_with_oracle(extractor, out, o, T, meta["weight_add"])
    assert np.array_equal(out["labels"][:T].cpu().numpy(), d["labels"])
    regions = extractor.regions_numpy(out["regions"])[:T]
    for t, (gs, gc) in enumerate(helpers.golden_components(d)):
        r = regions[t, : len(gs)]
        assert np.array_equal(np.stack([r["x"], r["y"], r["width"], r["height"], r["area"]], axis=1), gs)


def test_mixed_batch_denoise_and_plain(extractor):
    """Clips with and without CPT_CLIP_DENOISE in one launch."""
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import linear_clips
    from classifier_pipeline_b200.synthetic import clip_model, make_clip
    from oracle import oracle as orc

    lengths = [30, 24, 30]
    pix = [make_clip(40 + i, frames=n)[0] for i, n in enumerate(lengths)]
    frames = np.concatenate(pix)
    bts = [clip_model(40 + i)[2] for i in range(3)]
    was = [clip_model(40 + i)[3] for i in range(3)]
    slots = [extractor.ctx.weight_table(w, max_frames=4096) for w in was]
    clips = linear_clips(lengths, np.array(bts), np.array(slots))
    clips["flags"][1] |= native.CLIP_DENOISE
    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    out = extractor.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, out={})
    torch.cuda.synchronize()
    labels = out["labels"].cpu().numpy()
    info = extractor.info_numpy(out["info"])
    regions = extractor.regions_numpy(out["regions"])
    for i, n in enumerate(lengths):
        o0 = int(clips["out_offset"][i])
        o = orc.extract_clip(pix[i], pix[i][0], orc.make_params(background_thresh=bts[i], weight_add=was[i], max_comp=32, denoise=(i == 1)))
        assert np.array_equal(labels[o0 : o0 + n], o["labels"]), i
        assert np.array_equal(info["n_components"][o0 : o0 + n], o["ncomp"]), i
        for t in range(n):
            k = int(o["ncomp"][t])
            np.testing.assert_allclose(regions[o0 + t, :k]["pixel_variance"], o["var"][t, :k], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("geom", [(80, 64, 1), (128, 96, 1), (152, 40, 1), (160, 120, 0)])
@pytest.mark.parametrize("single", [False, True])
def test_other_geometries_match_the_oracle(geom, single):
    """The generic (rolled, unbalanced) sweep, generic staging chunks and generic hot-row extraction: frames that are not
    160x120 with a 1-pixel border, under both launch plans."""
    import torch
    from classifier_pipeline_b200.batch import BatchExtractor, linear_clips
    from classifier_pipeline_b200.synthetic import make_clip
    from oracle import oracle as orc

    W, H, edge = geom
    ex = BatchExtractor(device=0, width=W, height=H, edge_pixels=edge, max_regions=32)
    ex.ctx.force_single_kernel(single)
    lengths = [60, 3, 47]
    pix = [make_clip(70 + i, frames=n, width=W, height=H)[0] for i, n in enumerate(lengths)]
    slot = ex.ctx.weight_table(0.1, max_frames=1024)
    clips = linear_clips(lengths, 20, slot)
    d_frames = torch.from_numpy(np.concatenate(pix).view(np.int16)).cuda().view(torch.uint16)
    out = ex.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, keep_state=True, out={})
    torch.cuda.synchronize()
    regions = ex.regions_numpy(out["regions"])
    info = ex.info_numpy(out["info"])
    filtered = out["filtered"].cpu().numpy()
    labels = out["labels"].cpu().numpy()
    p = orc.make_params(W=W, H=H, edge=edge, background_thresh=20, weight_add=0.1, max_comp=32)
    seen = 0
    for i, n in enumerate(lengths):
        o0 = int(clips["out_offset"][i])
        o = orc.extract_clip(pix[i], pix[i][0], p)
        assert np.array_equal(filtered[o0 : o0 + n], o["filtered"]), i
        assert np.array_equal(labels[o0 : o0 + n], o["labels"]), i
        assert np.array_equal(info["n_components"][o0 : o0 + n], o["ncomp"]), i
        assert np.array_equal(info["threshold"][o0 : o0 + n], o["thresh"]), i
        for t in range(n):
            k = int(o["ncomp"][t])
            seen += k
            r = regions[o0 + t, :k]
            got = np.stack([r["x"], r["y"], r["width"], r["height"], r["area"], r["sum_x"], r["sum_y"], r["key"]], axis=1)
            assert np.array_equal(got, o["comp"][t, :k])
            np.testing.assert_allclose(r["pixel_variance"], o["var"][t, :k], rtol=1e-6, atol=1e-6)
        st = ex.ctx.state_read(out["state"], i)
        assert np.array_equal(st["background"], o["final_bg"]), i
    assert seen > 0
