"""Order statistics on the device against numpy, on inputs chosen to land on each side of every switch in the kernels:
median.cuh's 2048-bin histogram and two-pass radix paths (whole frames in cpt_frame_medians, crops in both medians passes
and the clip_thermals_at_zero decision), the thermal_diff_norm limits on wide-range frames, and the fp32 extrema of
cpt_minmax_f32 and the preprocessing limits pass on signed zeros, infinities, subnormals and lengths around a warp, a CTA
and the grid-stride loop."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GEOMETRIES = [(160, 120), (152, 40), (80, 64)]


def _dev_u16(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint16).view(np.int16)).cuda().view(torch.uint16)


def _dev_bytes(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def _frames_for_medians(rng, npx):
    """name -> uint16 (npx,): both sides of the histogram / radix switch and the bucket edges of the radix passes."""
    f = {}
    base = 3000
    a = rng.integers(base, base + 2048, npx)
    a[:2] = base, base + 2047
    f["range_2047"] = a  # the last histogram case
    b = a.copy()
    b[1] = base + 2048
    f["range_2048"] = b  # the first radix case
    f["uniform_0_65535"] = rng.integers(0, 65536, npx)
    f["half_255_half_256"] = rng.permutation(np.repeat([255, 256], npx // 2))
    w = f["half_255_half_256"].copy()  # the same middle ranks on the radix path: they sit in high-byte buckets 0 and 1
    w[np.flatnonzero(w == 255)[0]], w[np.flatnonzero(w == 256)[0]] = 0, 65535
    f["half_255_half_256_wide"] = w
    hi = rng.integers(0, 65536, npx)
    hi[rng.random(npx) < 0.8] = 65535  # both ranks in bucket 255, the exit value of both radix loops
    f["mostly_65535"] = hi
    lo = rng.integers(0, 65536, npx)
    lo[rng.random(npx) < 0.8] = 0
    f["mostly_0"] = lo
    f["constant"] = np.full(npx, 2900)
    c = np.full(npx, 2900)
    c[int(rng.integers(npx))] = 60000
    f["constant_wide_outlier"] = c
    c = np.full(npx, 2900)
    c[int(rng.integers(npx))] = 2901
    f["constant_narrow_outlier"] = c
    t = rng.integers(0, 65536, npx)
    t[rng.random(npx) < 0.4] = 31000
    f["ties_wide"] = t
    t = rng.integers(5000, 6500, npx)
    t[rng.random(npx) < 0.4] = 5700
    f["ties_narrow"] = t
    for name, v, lo_v, hi_v in (("adjacent_wide", 40000, 0, 65535), ("adjacent_narrow", 5000, 4000, 6000),
                                ("adjacent_bucket_edge", 0x7FFF, 0, 65535)):
        half = npx // 2
        below = rng.integers(lo_v, v + 1, half)
        above = rng.integers(v + 1, hi_v + 1, npx - half)
        below[0], above[0] = v, v + 1  # the two middle ranks: v and v + 1
        f[name] = rng.permutation(np.concatenate([below, above]))
    return {k: v.astype(np.uint16) for k, v in f.items()}


@pytest.mark.parametrize("W,H", GEOMETRIES)
def test_frame_medians_equal_numpy(W, H):
    import torch

    from classifier_pipeline_b200 import engine

    rng = np.random.default_rng(W * 1000 + H)
    cases = _frames_for_medians(rng, W * H)
    names = list(cases)
    frames = np.stack([cases[n].reshape(H, W) for n in names])
    ptp = frames.reshape(len(frames), -1).max(1).astype(np.int64) - frames.reshape(len(frames), -1).min(1)
    assert (ptp < 2048).any() and (ptp >= 2048).any()
    eng = engine.get_engine(None, W, H, 1)
    eng.ctx.use_torch_stream()
    d_med = torch.empty(len(frames), dtype=torch.float32, device="cuda")
    eng.ctx.frame_medians(_dev_u16(torch, frames), len(frames), d_med)
    got = d_med.cpu().numpy().astype(np.float64)
    want = np.array([np.median(f.astype(np.float64)) for f in frames])
    bad = [(n, g, w) for n, g, w in zip(names, got, want) if g != w]
    assert not bad, bad
    assert want[names.index("half_255_half_256_wide")] == 255.5 and want[names.index("adjacent_wide")] == 40000.5


# ---------------------------------------------------------------- crop medians and clip_thermals_at_zero
W0, H0 = 160, 120


def _crop_cases(rng):
    """(frames uint16 (n, H, W), samples [(frame, x, y, w, h)]): one sample per track."""
    npx = W0 * H0
    frames, samples = [], []

    def add(frame, rects):
        frames.append(frame.reshape(H0, W0).astype(np.uint16))
        samples.extend((len(frames) - 1,) + tuple(r) for r in rects)

    def rects(k):
        out = [(int(rng.integers(0, W0)), int(rng.integers(0, H0)), 1, 1), (0, 0, W0, H0)]
        for _ in range(k):
            w, h = int(rng.integers(1, 60)), int(rng.integers(1, 50))
            out += [(int(rng.integers(0, W0 - w + 1)), int(rng.integers(0, H0 - h + 1)), w, h),
                    (int(rng.integers(0, W0 - w + 1)), int(rng.integers(0, H0)), w, 1),
                    (int(rng.integers(0, W0)), int(rng.integers(0, H0 - h + 1)), 1, h)]
        return out

    # narrow frames (histogram path), wide frames (radix path, also for the crops: their own range is >= 2048)
    for f in _frames_for_medians(rng, npx).values():
        add(f, rects(2))
    add(rng.integers(0, 65536, npx), [(10, 10, 7, 5), (3, 4, 8, 6), (0, 0, 1, 2), (50, 60, 2, 1), (20, 30, 33, 17)])
    # crop median == frame median (clip turns off) and == frame median + 0.5 (clip stays on), narrow and wide
    for spread in (300, 20000):
        m = 30000
        for odd in (True, False):
            f = rng.integers(m - spread, m + spread + 1, npx)
            f[rng.random(npx) < 0.4] = m  # the frame median is m
            x, y, w, h = 40, 30, 7, (5 if odd else 6)
            n = w * h
            below = rng.integers(m - spread, m, n // 2 - (0 if odd else 1))
            above = rng.integers(m + 1, m + spread + 1, n // 2 - (0 if odd else 1))
            mid = [m] if odd else [m, m + 1]
            crop = rng.permutation(np.concatenate([below, mid, above]))
            f.reshape(H0, W0)[y : y + h, x : x + w] = crop.reshape(h, w)
            add(f, [(x, y, w, h)])
    return np.stack(frames), samples


@pytest.mark.parametrize("kernel", ["sample_median", "sample_crop_median"])
def test_crop_medians_and_clip_decision_equal_numpy(kernel):
    """sample.median and each track's clip_at_zero against np.median(frame) and the rule of interpreter.py:393-399,
    np.median(np.float32(sub) - median) <= 0 switches the clip off; one sample per track."""
    import torch

    from classifier_pipeline_b200 import engine, native
    from classifier_pipeline_b200.batch import BatchPreprocessor

    frames, samples = _crop_cases(np.random.default_rng(17))
    smp = np.zeros(len(samples), native.SAMPLE_DTYPE)
    for i, (f, x, y, w, h) in enumerate(samples):
        smp[i] = (f, x, y, w, h, i, 0.0)
    want_median = np.array([np.median(frames[f].astype(np.float64)) for f in smp["frame"]])
    want_clip = np.array([0 if np.median(np.float32(frames[f][y : y + h, x : x + w]) - m) <= 0 else 1
                          for (f, x, y, w, h), m in zip(samples, want_median)])
    crop_ptp = np.array([int(frames[f][y : y + h, x : x + w].max()) - int(frames[f][y : y + h, x : x + w].min()) for f, x, y, w, h in samples])
    assert (want_clip == 0).any() and (want_clip == 1).any() and (crop_ptp >= 2048).sum() >= 10
    # the last four samples are the boundary constructions: crop median == frame median, then frame median + 0.5
    crop_med = np.array([np.median(frames[f][y : y + h, x : x + w].astype(np.float64)) for f, x, y, w, h in samples])
    assert list(crop_med[-4:] - want_median[-4:]) == [0, 0.5, 0, 0.5] and list(want_clip[-4:]) == [0, 1, 0, 1]

    eng = engine.get_engine(None, W0, H0, 1)
    eng.ctx.use_torch_stream()
    d_thermal = _dev_u16(torch, frames)
    d_smp = _dev_bytes(torch, smp)
    d_tracks = torch.empty((len(smp), native.TRACK_NORM_DTYPE.itemsize), dtype=torch.uint8, device="cuda")
    eng.ctx.preprocess_limits(None, None, 0, d_tracks, len(smp))  # (resets the track rows)
    if kernel == "sample_median":
        eng.ctx.preprocess_medians(d_thermal, d_smp, len(smp), d_tracks)
    else:
        d_med = torch.empty(len(frames), dtype=torch.float32, device="cuda")
        eng.ctx.frame_medians(d_thermal, len(frames), d_med)
        eng.ctx.preprocess_medians(d_thermal, d_smp, len(smp), d_tracks, d_frame_medians=d_med)
    got = d_smp.cpu().numpy().view(native.SAMPLE_DTYPE)
    tracks = BatchPreprocessor.tracks_numpy(d_tracks)
    assert np.array_equal(got["median"].astype(np.float64), want_median)
    bad = [(samples[i], want_median[i], crop_med[i]) for i in np.flatnonzero(tracks["clip_at_zero"] != want_clip)]
    assert not bad, bad


@pytest.mark.parametrize("kernel", ["frames", "frame_stats"])
def test_thermal_limits_on_wide_range_frames_equal_oracle(kernel):
    """get_limits with thermal_diff_norm (interpreter.py:338-345): min / max of frame.thermal - median over every region's
    whole frame, read from the frames (track_thermal_limits_kernel) or from the frame extrema and medians
    (track_thermal_limits_stats_kernel), exactly as the oracle computes them."""
    import torch

    from classifier_pipeline_b200 import engine, native
    from classifier_pipeline_b200.batch import BatchPreprocessor
    from oracle import preprocess_oracle as po

    rng = np.random.default_rng(23)
    frames = np.stack([v.reshape(H0, W0) for v in _frames_for_medians(rng, W0 * H0).values()])
    n_frames = len(frames)
    tracks = []
    for ti in range(12):
        fr = np.sort(rng.choice(n_frames, int(rng.integers(1, 6)), replace=False))
        tracks.append(np.array([[f, 5, 6, 10 + ti, 8, int(k > 0 and rng.random() < 0.2)] for k, f in enumerate(fr)], np.int64))
    tracks.append(np.array([[f, 1, 1, 4, 4, 0] for f in range(n_frames)], np.int64))  # every frame
    rows = [(ti, r) for ti, regs in enumerate(tracks) for r in regs if not r[5]]
    lim = np.zeros(len(rows), native.SAMPLE_DTYPE)
    for i, (ti, r) in enumerate(rows):
        lim[i] = (r[0], r[1], r[2], r[3], r[4], ti, 0.0)

    eng = engine.get_engine(None, W0, H0, 1)
    eng.ctx.use_torch_stream()
    d_thermal = _dev_u16(torch, frames)
    d_lim = _dev_bytes(torch, lim)
    d_tracks = torch.empty((len(tracks), native.TRACK_NORM_DTYPE.itemsize), dtype=torch.uint8, device="cuda")
    eng.ctx.preprocess_limits(None, None, 0, d_tracks, len(tracks))
    if kernel == "frames":
        eng.ctx.preprocess_thermal_limits(d_thermal, d_lim, len(lim), d_tracks, len(tracks))
    else:
        d_med = torch.empty(n_frames, dtype=torch.float32, device="cuda")
        eng.ctx.frame_medians(d_thermal, n_frames, d_med)
        info = np.zeros(n_frames, native.INFO_DTYPE)
        info["thermal_min"] = frames.reshape(n_frames, -1).min(1)
        info["thermal_max"] = frames.reshape(n_frames, -1).max(1)
        eng.ctx.preprocess_thermal_limits(d_thermal, d_lim, len(lim), d_tracks, len(tracks), d_frame_medians=d_med,
                                          d_frame_info=_dev_bytes(torch, info))
    got = BatchPreprocessor.tracks_numpy(d_tracks)
    assert (got["has_thermal_limits"] == 1).all()
    for ti, regs in enumerate(tracks):
        lo, hi = po.thermal_limits(frames, regs)
        assert (float(got["thermal_min"][ti]), float(got["thermal_max"][ti])) == (float(lo), float(hi)), ti


# ---------------------------------------------------------------- fp32 extrema
def _extrema_cases(rng, num_sms):
    f32 = np.float32
    tiny = np.finfo(np.float32).smallest_subnormal
    fmax = np.finfo(np.float32).max
    cases = {
        "neg3_negzero": f32([-3, -0.0]),
        "negzero_only": np.full(40, -0.0, f32),
        "negzero_one": f32([-0.0]),
        "zeros_mixed": f32([0.0, -0.0, -0.0, 0.0, -0.0]),
        "negzero_warp_vs_negative_warp": np.concatenate([np.full(32, -0.0, f32), np.full(32, -5.0, f32)]),
        "negative_warp_vs_negzero_warp": np.concatenate([np.full(256 * 3, -5.0, f32), np.full(256 * 5, -0.0, f32)]),
        "negatives_and_negzero_spread": np.where(rng.random(5000) < 0.01, f32(-0.0), -rng.random(5000).astype(f32) - f32(1)),
        "pos_and_negzero": f32([2.5, -0.0, 1.0]),
        "inf": f32([1.0, np.inf, -np.inf, -2.0]),
        "flt_max": f32([fmax, -fmax, 0.0]),
        "subnormals": f32([tiny, -tiny, 3 * tiny, -7 * tiny]),
        "subnormal_negzero": f32([-0.0, tiny]),
        "neg_subnormal_negzero": f32([-0.0, -tiny]),
    }
    for n in (1, 31, 32, 33, 255, 256, 257, 4 * num_sms * 256 * 2 + 77):
        a = rng.normal(0, 100, n).astype(f32)
        cases["n{}".format(n)] = a
        b = a.copy()
        b[0], b[-1] = f32(-1e6), f32(1e6)
        cases["n{}_first_min_last_max".format(n)] = b
        c = a.copy()
        c[-1], c[0] = f32(-1e6), f32(1e6)
        cases["n{}_first_max_last_min".format(n)] = c
        cases["n{}_all_negative".format(n)] = -np.abs(a) - f32(1)
    return cases


def test_minmax_f32_equals_numpy():
    import torch

    from classifier_pipeline_b200 import engine

    eng = engine.get_engine()
    eng.ctx.use_torch_stream()
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    bad = []
    for name, a in _extrema_cases(np.random.default_rng(31), num_sms).items():
        d_out = torch.empty(2, dtype=torch.float32, device="cuda")
        eng.ctx.minmax_f32(torch.from_numpy(a).cuda(), a.size, d_out)
        mn, mx = d_out.cpu().numpy()
        # by value: where numpy's extremum is -0.0, +0.0 is accepted too (-FLT_MAX never is)
        if not (mn == np.min(a) and mx == np.max(a)):
            bad.append((name, a.size, float(mn), float(np.min(a)), float(mx), float(np.max(a))))
    assert not bad, bad


def test_normalize_with_signed_zeros_equals_oracle():
    """imageprocessing.normalize finds its extrema with cpt_minmax_f32: a -0.0 maximum must not come back as -FLT_MAX."""
    from classifier_pipeline_b200.ml_tools import imageprocessing as ip
    from oracle import preprocess_oracle as po

    rng = np.random.default_rng(37)
    arrays = [np.float32([-3, -0.0]), np.float32([[-3, -0.0], [-1.5, -2.0]]),
              np.concatenate([np.full(32, -0.0, np.float32), np.full(32, -5.0, np.float32)]),
              np.where(rng.random((120, 160)) < 0.05, np.float32(-0.0), -rng.random((120, 160)).astype(np.float32) * 50),
              np.float32([0.0, -0.0, 7.0])]
    for a in arrays:
        got, (ok, mx, mn) = ip.normalize(a, new_max=255)
        want, _ = po.normalize(a, new_max=255)
        assert ok and mx == np.max(a) and mn == np.min(a)
        assert got.dtype == want.dtype
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-5)
        assert got.min() >= 0 and got.max() <= 255


def test_track_filtered_limits_with_negative_and_signed_zero_crops():
    """track_limits_kernel (float CAS atomics) against get_limits on tracks whose filtered crops are all negative (the
    maximum stays at its start value 0) or hold -0.0."""
    import torch

    from classifier_pipeline_b200 import engine, native
    from classifier_pipeline_b200.batch import BatchPreprocessor
    from oracle import preprocess_oracle as po

    rng = np.random.default_rng(41)
    n_frames = 6
    filtered = -rng.random((n_frames, H0, W0)).astype(np.float32) * 300 - np.float32(1)
    filtered[2, 10:40, 10:50] = -0.0
    filtered[3, 60:70, 60:90] = np.where(rng.random((10, 30)) < 0.5, np.float32(-0.0), np.float32(-4.0))
    filtered[4] = -0.0
    tracks = [
        np.array([[0, 5, 5, 30, 20, 0], [1, 100, 50, 40, 40, 0]], np.int64),   # all negative
        np.array([[2, 10, 10, 40, 30, 0]], np.int64),                          # all -0.0
        np.array([[3, 60, 60, 30, 10, 0], [1, 0, 0, 1, 1, 0]], np.int64),      # -0.0 and negatives
        np.array([[2, 5, 5, 20, 20, 0], [0, 3, 3, 2, 2, 0]], np.int64),        # -0.0 in one region, negatives in another
        np.array([[4, 0, 0, W0, H0, 0], [5, 0, 0, W0, H0, 1]], np.int64),      # a whole -0.0 frame; a blank region
    ]
    rows = [(ti, r) for ti, regs in enumerate(tracks) for r in regs if not r[5]]
    lim = np.zeros(len(rows), native.SAMPLE_DTYPE)
    for i, (ti, r) in enumerate(rows):
        lim[i] = (r[0], r[1], r[2], r[3], r[4], ti, 0.0)
    eng = engine.get_engine(None, W0, H0, 1)
    eng.ctx.use_torch_stream()
    d_tracks = torch.empty((len(tracks), native.TRACK_NORM_DTYPE.itemsize), dtype=torch.uint8, device="cuda")
    eng.ctx.preprocess_limits(torch.from_numpy(filtered).cuda(), _dev_bytes(torch, lim), len(lim), d_tracks, len(tracks))
    got = BatchPreprocessor.tracks_numpy(d_tracks)
    assert (got["has_limits"] == 1).all()
    for ti, regs in enumerate(tracks):
        lo, hi = po.track_limits(filtered, regs)
        assert got["filtered_min"][ti] == lo and got["filtered_max"][ti] == hi, (ti, got[ti], lo, hi)
