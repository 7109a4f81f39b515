"""The C-ABI library loads and exports every symbol include/cptrack.h declares (no GPU needed)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    g.build()
    from classifier_pipeline_b200 import native

    return native.load()


def header_symbols():
    text = open(os.path.join(ROOT, "include", "cptrack.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cpt_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(lib):
    from classifier_pipeline_b200 import native

    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), s
    assert sorted(native.SYMBOLS) == syms


def test_struct_layouts_match_header():
    import ctypes

    from classifier_pipeline_b200 import native

    assert ctypes.sizeof(native.CptRegion) == 40
    assert ctypes.sizeof(native.CptFrameInfo) == 64
    assert ctypes.sizeof(native.CptClip) == 48
    assert native.CptRegion.pixel_variance.offset == 32
    assert native.CptClip.n_frames.offset == 24


def test_no_device_fails_loudly(lib):
    import torch

    from classifier_pipeline_b200 import native

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(native.NativeError):
        native.Context()
    from classifier_pipeline_b200.batch import BatchExtractor

    with pytest.raises(native.NativeError):
        BatchExtractor()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "classifier-pipeline_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), os.path.join(dirpath, f)


def test_no_product_module_calls_the_library_directly():
    """native.py is the only caller of libcptrack.so: every other product module goes through its wrappers."""
    pkg = os.path.join(ROOT, "classifier-pipeline_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py") and path != os.path.join(pkg, "native.py"):
                src = open(path).read()
                assert "lib.cpt_" not in src and not re.search(r"\._h\b", src), path


def test_clip_flags_match_header():
    """The Python constants of the clip, detect, motion and preprocessing flags are the header's #defines."""
    from classifier_pipeline_b200 import native

    text = open(os.path.join(ROOT, "include", "cptrack.h")).read()
    for group, expected in (("CLIP", {"UPDATE_BACKGROUND", "RESUME", "DENOISE", "FRAME_STATS", "SKIP_FIRST_UPDATE", "PREV_IN_OUTPUT"}),
                            ("DETECT", {"CLOSE", "OPEN_GRAY", "DILATE", "OTSU", "MASK_ONLY"}),
                            ("MOTION", {"MEAN", "MEAN_RESTART", "BACKGROUND", "DETECT", "WARMER_ONLY", "ONE_DIFF"}),
                            ("PREPROCESS", {"INC3", "PER_TILE"})):
        flags = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+CPT_%s_([A-Z0-9_]+)\s+(\d+)u?\b" % group, text)}
        assert set(flags) >= expected, group
        for name, value in flags.items():
            assert getattr(native, group + "_" + name) == value, group + "_" + name
        assert len(set(flags.values())) == len(flags) and all(v & (v - 1) == 0 for v in flags.values()), group
