"""What the compiler made of csrc/mog2_kernels.cu (no GPU needed): the modes stay in registers (no local memory, no stack),
and the only fused multiply-adds are the Newton steps inside the correctly rounded divisions, so every product and sum of
the MOG2 update is rounded on its own as cv2 rounds it."""
import os
import re
import shutil
import subprocess

import pytest

APPLY = "_ZN3cpt17mog2_apply_kernel"
BACKGROUND = "_ZN3cpt22mog2_background_kernel"


@pytest.fixture(scope="module")
def lib_path():
    import __graft_entry__ as g

    g.build()
    from classifier_pipeline_b200 import native

    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not installed")
    return tool, native.LIB_PATH


def test_mog2_kernels_use_no_local_memory(lib_path):
    tool, lib = lib_path
    out = subprocess.run([tool, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    for name in (APPLY, BACKGROUND):
        m = re.search(r"Function " + name + r"\S*:\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
        assert m, name
        assert int(m.group(2)) == 0 and int(m.group(3)) == 0, m.group(0)


def test_mog2_update_has_no_contracted_multiply_add(lib_path):
    tool, lib = lib_path
    sass = subprocess.run([tool, "-sass", lib], capture_output=True, text=True, check=True).stdout
    start = sass.index("Function : " + APPLY)
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
    assert n_ffma > 0  # (the divisions are there: the check above saw them)
