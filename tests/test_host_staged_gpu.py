"""The two host-staged calls (cpt_extract_batch_host: uint16 frames; cpt_extract_batch_cptv_host: packed CPTV payloads)
share one chunked, double-buffered pipeline and grow the context's staging and scratch buffers on demand.  Both must
equal the device-resident call for every chunking, one context must give over a sequence of differently shaped calls
what fresh contexts give, and a rejected input must leave the context usable."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# frame table rows per clip: with 1, 2 or 3 clips per chunk a later chunk spans more frames than the first one (the split
# plan's buffers grow in the middle of a call) and the last chunk is ragged
ROWS = [12, 40, 9, 64, 25, 80, 31]
DENOISE = (1, 5)  # a small and then a larger chunk with CPT_CLIP_DENOISE: the denoise buffers grow in the middle of a call
LEADING = {2: 1, 4: 3}  # clip -> frames between its init frame (the clip's first row) and its first tracked frame
MAX_REGIONS = 16
INFO_FIELDS = ("background_average", "threshold", "norm_min", "norm_max", "avg_change", "filtered_min", "filtered_max",
               "n_components", "thermal_sum")
REGION_FIELDS = ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key")


def _context():
    """A fresh context with the weight tables of both synthetic clip models in slots 0 and 1."""
    from classifier_pipeline_b200.batch import BatchExtractor
    from classifier_pipeline_b200.synthetic import MODELS

    ex = BatchExtractor(device=0, max_regions=MAX_REGIONS)
    assert [ex.ctx.weight_table(m[3], max_frames=4096) for m in MODELS] == [0, 1]
    return ex


def _inputs(rows, first_index=0, denoise=(), leading=None):
    """Seeded synthetic clips laid out back to back: (frames uint16 (sum(rows), H, W), (stream, table, clip_first) of the
    same frames packed, clip records addressing frames by row)."""
    import torch
    from classifier_pipeline_b200 import native
    from classifier_pipeline_b200.synthetic import clip_model, make_clip, pack_clips_torch

    leading = leading or {}
    pix = [make_clip(first_index + i, frames=n)[0] for i, n in enumerate(rows)]
    streams, tables, base = [], [], 0
    for p in pix:
        stream, table, _ = pack_clips_torch(torch.from_numpy(p.view(np.int16)).cuda().view(torch.uint16)[None])
        table["payload_offset"] += base
        # (a copy without the slack bytes past the clip's last payload: a view would not keep the pinned memory alive)
        streams.append(np.array(stream[:-4]))
        tables.append(table)
        base += len(streams[-1])
    stream = np.concatenate(streams + [np.zeros(4, np.uint8)])
    first = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    lead = np.array([leading.get(i, 0) for i in range(len(rows))], np.int64)
    n_frames = np.asarray(rows, np.int64) - lead
    clips = np.zeros(len(rows), native.CLIP_DTYPE)
    clips["init_offset"] = first[:-1]
    clips["frame_offset"] = first[:-1] + lead
    clips["out_offset"] = np.concatenate([[0], np.cumsum(n_frames)[:-1]])
    clips["n_frames"] = n_frames
    clips["background_thresh"] = [clip_model(first_index + i)[2] for i in range(len(rows))]
    clips["weight_table"] = [(first_index + i) % 2 for i in range(len(rows))]  # (the slot of clip_model(i) in _context)
    clips["flags"] = native.CLIP_UPDATE_BACKGROUND
    for i in denoise:
        clips["flags"][i] |= native.CLIP_DENOISE
    return np.concatenate(pix), (stream, np.concatenate(tables), first), clips


def _device_call(ex, frames, clips):
    import torch

    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    out = ex.extract_device(d_frames, clips, keep_filtered=True, keep_labels=True, out={})
    torch.cuda.synchronize()
    return dict(regions=ex.regions_numpy(out["regions"]), info=ex.info_numpy(out["info"]), filtered=out["filtered"].cpu().numpy(),
                labels=out["labels"].cpu().numpy())


def _assert_same(got, want, clips):
    total = int((clips["out_offset"] + clips["n_frames"]).max())
    for f in INFO_FIELDS:
        assert np.array_equal(got["info"][f][:total], want["info"][f][:total]), f
    for key in ("filtered", "labels"):
        if got.get(key) is not None:
            assert np.array_equal(got[key][:total], want[key][:total]), key
    n = np.minimum(want["info"]["n_components"][:total], MAX_REGIONS)
    live = np.arange(MAX_REGIONS)[None, :] < n[:, None]
    g, w = got["regions"][:total][live], want["regions"][:total][live]
    assert live.any()
    for f in REGION_FIELDS:
        assert np.array_equal(g[f], w[f]), f
    assert np.array_equal(g["pixel_variance"], w["pixel_variance"])


@pytest.fixture(scope="module")
def batch():
    """The ROWS batch and what the device-resident call returns for it (on a context of its own, so that the host calls
    below start from empty buffers)."""
    frames, packed, clips = _inputs(ROWS, denoise=DENOISE, leading=LEADING)
    return frames, packed, clips, _device_call(_context(), frames, clips)


@pytest.mark.parametrize("chunk_clips", [0, 1, 2, 3, len(ROWS), len(ROWS) + 1])
def test_host_calls_match_the_device_call(batch, chunk_clips):
    frames, packed, clips, want = batch
    raw = _context().extract_host(frames, clips, keep_filtered=True, keep_labels=True, chunk_clips=chunk_clips, out={})
    _assert_same(raw, want, clips)
    got = _context().extract_host_packed(*packed, clips, chunk_clips=chunk_clips, out={})
    _assert_same(got, want, clips)


def test_one_context_over_a_sequence_of_calls(batch):
    """Small, large, small; raw without the filtered / label images, then with them; packed after raw on the same staging
    buffers: every call equals the same call on a fresh context."""
    frames, packed, clips, _ = batch
    small = _inputs([10, 22, 15], first_index=20, leading={1: 2})
    large = (frames, packed, clips)

    def raw(ex, inputs, chunk, keep):
        return ex.extract_host(inputs[0], inputs[2], keep_filtered=keep, keep_labels=keep, chunk_clips=chunk, out={})

    def pk(ex, inputs, chunk, keep):
        return ex.extract_host_packed(*inputs[1], inputs[2], chunk_clips=chunk, out={})

    ex = _context()
    for call, inputs, chunk, keep in [(raw, small, 2, False), (raw, large, 3, False), (raw, small, 1, False), (raw, small, 2, True),
                                      (raw, large, 2, True), (pk, large, 3, False), (pk, small, 1, False), (raw, large, 2, True)]:
        _assert_same(call(ex, inputs, chunk, keep), call(_context(), inputs, chunk, keep), inputs[2])


def test_rejected_inputs_leave_the_context_usable(batch):
    from classifier_pipeline_b200 import native

    frames, packed, clips, want = batch
    ex = _context()
    resume = clips.copy()
    resume["flags"][3] |= native.CLIP_RESUME
    with pytest.raises(native.NativeError):
        ex.extract_host(frames, resume, chunk_clips=2, out={})
    with pytest.raises(native.NativeError):
        ex.extract_host_packed(*packed, resume, chunk_clips=2, out={})
    # a clip whose outputs run past the output buffers
    total = int(clips["n_frames"].sum())
    regions = native.pinned_empty((total - 1, MAX_REGIONS), native.REGION_DTYPE)
    info = native.pinned_empty((total - 1,), native.INFO_DTYPE)
    with pytest.raises(native.NativeError):
        ex.ctx.extract_batch_host(frames, clips, total - 1, regions, info, chunk_clips=2)
    _assert_same(ex.extract_host(frames, clips, keep_filtered=True, keep_labels=True, chunk_clips=2, out={}), want, clips)
    _assert_same(ex.extract_host_packed(*packed, clips, chunk_clips=2, out={}), want, clips)
