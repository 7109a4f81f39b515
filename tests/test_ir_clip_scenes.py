"""No GPU: the designed IR scenes reach the cases they are named for (on the detector restated on cv2), the records of
cpt_ir_motion_clips have the header's layout (compiled with the host C compiler), and the compiled IR kernels keep the MOG2
update in registers and round every product and sum on its own, as cv2 does."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from tests import ir_clip_scenes as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRAME = "_ZN3cpt15ir_frame_kernel"
ERODE = "_ZN3cpt15ir_erode_kernel"


@pytest.mark.parametrize("name", list(sc.DESIGNS))
def test_designed_scene_reaches_its_case(name):
    pytest.importorskip("cv2")
    sc.check_design(name, sc.cv2_trace(sc.design(name)))


def test_clip_records_match_header(tmp_path):
    from classifier_pipeline_b200 import native

    cc = shutil.which("cc") or shutil.which("gcc")
    if not cc:
        pytest.skip("no host C compiler")
    names = ("cpt_ir_motion_clip", "cpt_ir_motion_clip_step", "cpt_ir_motion_clip_params", "cpt_ir_motion_clip_result")
    types = (native.CptIrMotionClip, native.CptIrMotionClipStep, native.CptIrMotionClipParams, native.CptIrMotionClipResult)
    lines = []
    for name, t in zip(names, types):
        lines.append('printf("{0} %zu\\n", sizeof({0}));'.format(name))
        for field, _ in t._fields_:
            lines.append('printf("{0}.{1} %zu\\n", offsetof({0}, {1}));'.format(name, field))
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "cptrack.h"\nint main(void) {\n' + "\n".join(lines) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, t in zip(names, types):
        assert int(got[name]) == ctypes.sizeof(t), name
        for field, _ in t._fields_:
            assert int(got[name + "." + field]) == getattr(t, field).offset, (name, field)


@pytest.fixture(scope="module")
def lib_path():
    import __graft_entry__ as g

    g.build()
    from classifier_pipeline_b200 import native

    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not installed")
    return tool, native.LIB_PATH


def test_ir_clip_kernels_use_no_local_memory(lib_path):
    tool, lib = lib_path
    out = subprocess.run([tool, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    for name in (FRAME, ERODE):
        m = re.search(r"Function " + name + r"\S*:\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
        assert m, name
        assert int(m.group(2)) == 0 and int(m.group(3)) == 0, m.group(0)


def test_ir_frame_kernel_has_no_contracted_multiply_add(lib_path):
    """The method of tests/test_mog2_sass.py on the kernel of whole clips: every FFMA is a Newton step of a division."""
    tool, lib = lib_path
    sass = subprocess.run([tool, "-sass", lib], capture_output=True, text=True, check=True).stdout
    start = sass.index("Function : " + FRAME)
    end = sass.find("Function : ", start + 1)
    sass = sass[start : end if end > 0 else len(sass)]
    ins = re.findall(r"/\*([0-9a-f]{4,})\*/\s+(.*?);", sass)
    assert len(ins) > 100
    calls = [int(t, 16) for _, i in ins for t in re.findall(r"CALL\.REL\.NOINC 0x([0-9a-f]+)", i)]
    sub = min(calls) if calls else None  # the division's slow path: a subroutine after the kernel body
    since_rcp = 99
    n_ffma = 0
    for addr, i in ins:
        since_rcp = 0 if "MUFU.RCP" in i else since_rcp + 1
        if re.search(r"\bFFMA\b", i):
            n_ffma += 1
            in_division = since_rcp <= 10 or (sub is not None and int(addr, 16) >= sub)
            assert in_division, "FFMA outside a division at 0x{}: {}".format(addr, i)
    assert any("FMUL" in i for _, i in ins) and any("FADD" in i for _, i in ins)
    assert n_ffma > 0
