"""The per-frame mask and component stage against the C oracle on the designed clips of tests/frame_designs.py, which put
frames on both sides of each of its switches: the in-CTA component table and run table of frame_regions_kernel, its bands,
the fallback kernel's full slot table (more than 255 components included), frame edges, word boundaries, label order,
frames without foreground and the single kernel's work-list cap.  Bit-exact: filtered images, thresholds, component counts,
labels and region records; variances rtol 1e-6."""
import numpy as np
import pytest

from tests import frame_designs as fd

pytestmark = pytest.mark.gpu

DESIGNS = fd.designs()
FIELDS = ("x", "y", "width", "height", "area", "sum_x", "sum_y", "key")


def _clips(ex, designs, repeat=1):
    from classifier_pipeline_b200.batch import linear_clips

    ds = list(designs) * repeat
    slot = ex.ctx.weight_table(0.1, max_frames=1024)
    clips = linear_clips([len(d.frames) for d in ds], np.array([d.bt for d in ds]), slot)
    return ds, np.concatenate([d.frames for d in ds]), clips


def _device(ex, frames, clips, single, keep_filtered=True):
    import torch

    d_frames = torch.from_numpy(frames.view(np.int16)).cuda().view(torch.uint16)
    ex.ctx.force_single_kernel(single)
    try:
        out = ex.extract_device(d_frames, clips, keep_filtered=keep_filtered, keep_labels=True, out={})
        torch.cuda.synchronize()
    finally:
        ex.ctx.force_single_kernel(False)
    return dict(filtered=out["filtered"].cpu().numpy() if keep_filtered else None, labels=out["labels"].cpu().numpy(),
                info=ex.info_numpy(out["info"]).copy(), regions=ex.regions_numpy(out["regions"]).copy())


def _compare(got, ds, clips, max_regions):
    for i, d in enumerate(ds):
        o = fd.run_oracle(d, max_comp=max_regions)
        o0, n = int(clips["out_offset"][i]), len(d.frames)
        sl = slice(o0, o0 + n)
        assert np.array_equal(got["filtered"][sl], o["filtered"]), d.name
        assert np.array_equal(got["info"]["threshold"][sl], o["thresh"]), d.name
        assert np.array_equal(got["info"]["n_components"][sl], o["ncomp"]), d.name
        assert np.array_equal(got["labels"][sl], o["labels"]), d.name
        for t in range(n):
            k = min(int(o["ncomp"][t]), max_regions)
            r = got["regions"][o0 + t, :k]
            assert np.array_equal(np.stack([r[f] for f in FIELDS], axis=1), o["comp"][t, :k]), (d.name, t)
            np.testing.assert_allclose(r["pixel_variance"], o["var"][t, :k], rtol=1e-6, atol=1e-6, err_msg=d.name)


@pytest.fixture(scope="module", params=[32, 255])
def extractor(request):
    from classifier_pipeline_b200.batch import BatchExtractor

    return BatchExtractor(device=0, max_regions=request.param)


@pytest.mark.parametrize("single", [False, True], ids=["split", "single"])
def test_designs_match_the_oracle(extractor, single):
    ds, frames, clips = _clips(extractor, DESIGNS)
    _compare(_device(extractor, frames, clips, single), ds, clips, extractor.max_regions)


def test_lean_designs_with_fewer_region_slots_than_components():
    """32 components with 16 region slots: the in-CTA stage ranks all 32 and stores the first 16."""
    from classifier_pipeline_b200.batch import BatchExtractor

    ex = BatchExtractor(device=0, max_regions=16)
    ds, frames, clips = _clips(ex, [d for d in DESIGNS if d.name.startswith("lean_")])
    for single in (False, True):
        _compare(_device(ex, frames, clips, single), ds, clips, 16)


def test_both_plans_agree_on_the_designs(extractor):
    """The split plan against the single kernel with the filtered images kept (which leaves the variances of all frames but
    the first to region_variance_kernel) and without them (regions only: the single kernel computes every variance)."""
    ds, frames, clips = _clips(extractor, DESIGNS)
    a = _device(extractor, frames, clips, False)
    for keep_filtered in (True, False):
        b = _device(extractor, frames, clips, True, keep_filtered=keep_filtered)
        assert not keep_filtered or np.array_equal(a["filtered"], b["filtered"])
        assert np.array_equal(a["labels"], b["labels"]), keep_filtered
        for f in ("threshold", "n_components", "norm_min", "norm_max", "avg_change"):
            assert np.array_equal(a["info"][f], b["info"][f]), (keep_filtered, f)
        for t in range(len(frames)):
            k = min(int(a["info"]["n_components"][t]), extractor.max_regions)
            for f in FIELDS + ("pixel_variance",):
                assert np.array_equal(a["regions"][t, :k][f], b["regions"][t, :k][f]), (keep_filtered, t, f)


def test_host_staged_chunks_and_a_larger_second_call(extractor):
    """extract_host with one and three clips per chunk, so that fallback frames fall in several chunks; then a call twice the
    size on the same context, which grows its scratch buffers."""
    ds, frames, clips = _clips(extractor, DESIGNS)
    for chunk in (1, 3):
        host = extractor.extract_host(frames, clips, keep_filtered=True, keep_labels=True, chunk_clips=chunk)
        _compare(host, ds, clips, extractor.max_regions)
    ds2, frames2, clips2 = _clips(extractor, DESIGNS, repeat=2)
    host = extractor.extract_host(frames2, clips2, keep_filtered=True, keep_labels=True, chunk_clips=3)
    _compare(host, ds2, clips2, extractor.max_regions)


@pytest.mark.parametrize("geom", [(152, 40), (80, 64)], ids=["152x40", "80x64"])
@pytest.mark.parametrize("single", [False, True], ids=["split", "single"])
def test_other_geometries_match_the_oracle(geom, single):
    """152 pixels: a row of 38 quads, not whole words of quad bytes (the byte-wise path).  80x64: a two-word row."""
    from classifier_pipeline_b200.batch import BatchExtractor

    W, H = geom
    ex = BatchExtractor(device=0, width=W, height=H, edge_pixels=1, max_regions=255)
    ds, frames, clips = _clips(ex, fd.small_designs(H, W))
    _compare(_device(ex, frames, clips, single), ds, clips, 255)
