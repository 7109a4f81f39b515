"""CPTV v2 decode on the device (cpt_cptv_decode) == the host decoder, for the reference's clips and for
synthetic streams of every bit width; parse_clip on files goes through it."""
import os

import numpy as np
import pytest

from tests import helpers
from tests.cptv_writer import write_cptv
from tests.test_cptv import random_walk_clip

pytestmark = pytest.mark.gpu


def _device_decode(paths):
    from classifier_pipeline_b200 import engine
    from classifier_pipeline_b200.cptv import CptvReader, decode_clips_device

    eng = engine.get_engine()
    d_frames, first, frames = decode_clips_device(eng, [CptvReader(p) for p in paths])
    return d_frames.cpu().numpy(), first, frames


def test_reference_clips_match_host_decoder():
    from classifier_pipeline_b200.cptv import read_clip

    paths = [os.path.join(helpers.GOLDEN, "clips", n + ".cptv") for n in ("possum", "hedgehog")]
    pix, first, meta = _device_decode(paths)
    for i, p in enumerate(paths):
        _, frames = read_clip(p)
        assert first[i + 1] - first[i] == len(frames)
        assert np.array_equal(pix[first[i] : first[i + 1]], np.array([f.pix for f in frames]))
        assert [m.background_frame for m in meta[i]] == [f.background_frame for f in frames]
        assert [m.time_on for m in meta[i]] == [f.time_on for f in frames]


def test_every_bit_width(tmp_path):
    paths, clips = [], []
    for k, (step, force) in enumerate([(0, None), (1, None), (3, None), (40, None), (700, None), (20000, None), (2, 13), (5, 16), (1, 9)]):
        rng = np.random.default_rng(100 + k)
        frames = random_walk_clip(rng, 5 + k % 3, step)
        path = tmp_path / "c{}.cptv".format(k)
        write_cptv(path, frames, force_bit_width=force)
        paths.append(path)
        clips.append(frames)
    pix, first, _ = _device_decode(paths)
    for i, frames in enumerate(clips):
        assert np.array_equal(pix[first[i] : first[i + 1]], frames), i


def _packed_inputs(paths):
    """(stream, table, clip_first, decoded clips) of CPTV files for cpt_extract_batch_cptv_host."""
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.cptv import CptvReader, read_clip

    streams, rows, first, decoded = [], [], [0], []
    base = 0
    for p in paths:
        buf, table, _ = CptvReader(p).index_frames()
        rows += [(base + off, w, 0) for off, w in table]
        streams.append(buf)
        base += len(buf)
        first.append(first[-1] + len(table))
        decoded.append(read_clip(p)[1])
    stream = np.frombuffer(b"".join(streams) + b"\0\0\0\0", dtype=np.uint8).copy()
    return stream, np.array(rows, dtype=native.CPTV_FRAME_DTYPE), np.array(first, dtype=np.int64), decoded


def test_packed_host_call_matches_raw_host_call():
    """cpt_extract_batch_cptv_host (packed payloads over PCIe, decoded on the device) == cpt_extract_batch_host on the
    frames the host decoder produces, for the reference's two clips (possum starts with a background frame the clip
    skips) -- regions, thresholds and counts identical."""
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import BatchExtractor, linear_clips

    ex = BatchExtractor(device=0, max_regions=16)
    paths = [os.path.join(helpers.GOLDEN, "clips", n + ".cptv") for n in ("possum", "hedgehog")]
    stream, table, first, decoded = _packed_inputs(paths)
    slot = ex.ctx.weight_table(0.1, max_frames=1024)
    skip = [1 if frames[0].background_frame else 0 for frames in decoded]
    lengths = [len(frames) - s for frames, s in zip(decoded, skip)]
    clips = linear_clips(lengths, 20, slot)
    raw = np.concatenate([np.array([f.pix for f in frames]) for frames in decoded])
    clips["init_offset"] = first[:-1]
    clips["frame_offset"] = first[:-1] + np.array(skip)
    want = ex.extract_host(raw, clips, chunk_clips=1, out={})
    got = ex.extract_host_packed(stream, table, first, clips, chunk_clips=1, out={})
    total = int(sum(lengths))
    for f in ("n_components", "threshold", "norm_min", "norm_max", "avg_change", "background_average"):
        assert np.array_equal(got["info"][f][:total], want["info"][f][:total]), f
    assert int(want["info"]["n_components"][:total].sum()) > 50
    for t in range(total):
        n = min(int(want["info"]["n_components"][t]), 16)
        for f in ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key"):
            assert np.array_equal(got["regions"][t, :n][f], want["regions"][t, :n][f]), (t, f)
        assert np.array_equal(got["regions"][t, :n]["pixel_variance"], want["regions"][t, :n]["pixel_variance"]), t


def test_packed_synthetic_batch_and_malformed_table():
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.batch import BatchExtractor, linear_clips
    from classifier_pipeline_b200.synthetic import MODELS, make_clips_torch, pack_clips_torch

    ex = BatchExtractor(device=0, max_regions=16)
    C, T = 5, 60
    d_frames, models = make_clips_torch(C, T, torch.device("cuda", 0))
    d_frames.view(torch.int16)[3, 10:12, 40:60, 50:80] += 900  # a step large enough to need 16-bit deltas in those frames
    stream, table, first = pack_clips_torch(d_frames)
    assert set(table["bit_width"]) == {8, 16}
    slots = [ex.ctx.weight_table(m[3], max_frames=1024) for m in MODELS]
    clips = linear_clips([T] * C, np.array([MODELS[m][2] for m in models]), np.array([slots[m] for m in models]))
    raw = d_frames.view(torch.int16).reshape(-1, 120, 160).cpu().numpy().view(np.uint16)
    want = ex.extract_host(raw, clips, chunk_clips=2, out={})
    got = ex.extract_host_packed(stream, table, first, clips, chunk_clips=2, out={})
    assert np.array_equal(got["info"]["n_components"], want["info"]["n_components"])
    assert np.array_equal(got["info"]["threshold"], want["info"]["threshold"])
    assert np.array_equal(got["info"]["thermal_sum"], want["info"]["thermal_sum"])
    for t in range(C * T):
        n = min(int(want["info"]["n_components"][t]), 16)
        for f in ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key"):
            assert np.array_equal(got["regions"][t, :n][f], want["regions"][t, :n][f]), (t, f)
        assert np.array_equal(got["regions"][t, :n]["pixel_variance"], want["regions"][t, :n]["pixel_variance"]), t
    # a payload that runs past the end of the stream is refused before anything is launched
    bad = table.copy()
    bad["payload_offset"][7] = stream.size - 100
    with pytest.raises(native.NativeError):
        ex.extract_host_packed(stream, bad, first, clips, chunk_clips=2, out={})
    bad = table.copy()
    bad["bit_width"][3] = 0
    with pytest.raises(native.NativeError):
        ex.extract_host_packed(stream, bad, first, clips, chunk_clips=2, out={})
