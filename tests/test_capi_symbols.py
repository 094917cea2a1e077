"""The C-ABI library builds, loads and exports every symbol include/dbgsom_b200.h declares (no GPU)."""
import ctypes
import os
import re

import pytest

from dbgsom_b200 import _native as nat
from dbgsom_b200 import build as builder

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    builder.build()
    return nat.load()


def declared_functions():
    text = open(os.path.join(ROOT, "include", "dbgsom_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dbgsom_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree(lib):
    names = declared_functions()
    assert len(names) >= 16
    assert sorted(nat.SIGNATURES) == names
    for n in names:
        assert hasattr(lib, n), n


def test_abi_version_and_status_strings(lib):
    assert lib.dbgsom_abi_version() == nat.ABI_VERSION
    assert lib.dbgsom_status_string(0) == b"ok"
    for code in (-1, -2, -3, -4, -5):
        assert lib.dbgsom_status_string(code).startswith(b"dbgsom:")


def test_argument_errors_do_not_touch_the_gpu(lib):
    # null / invalid arguments are rejected before any CUDA call
    assert lib.dbgsom_colstats(None, 10, 4, 4, None, None, None) == -1
    assert lib.dbgsom_bmu(None, None) == -1
    args = nat.BmuArgs()
    assert lib.dbgsom_bmu(ctypes.byref(args), None) == -1
    assert lib.dbgsom_bmu_candidates(ctypes.byref(args), None) == -1
    assert lib.dbgsom_bmu_resolve(ctypes.byref(args), None) == -1
    assert lib.dbgsom_accumulate(None, None) == -1
    assert lib.dbgsom_smooth(None, None) == -1
    assert lib.dbgsom_apply_row_ops(None, 4, None, 0, None) == -1
    assert lib.dbgsom_gather_rows(None, 4, 4, None, 0, None, None) == -1
    assert lib.dbgsom_bmu_workspace_bytes(1000, 1) >= 1000 * (4 * nat.MAX_CAND + 1)
    assert lib.dbgsom_accumulate_workspace_bytes(1000, 16, 4) >= 4000
    assert lib.dbgsom_smooth_workspace_bytes(16, 8) >= 16 * 8 * 8


def test_struct_sizes_match_the_c_layout():
    # 64-bit layout of the three argument structs (guards against field drift in the binding)
    assert ctypes.sizeof(nat.BmuArgs) == 256
    assert ctypes.sizeof(nat.AccumulateArgs) == 112
    assert ctypes.sizeof(nat.SmoothArgs) == 96


def test_struct_sizes_match_the_header_as_compiled(tmp_path):
    """sizeof() of the argument structs as a C compiler lays out include/dbgsom_b200.h == the ctypes mirror."""
    import shutil
    import subprocess

    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "sizes.c"
    src.write_text(
        '#include <stdio.h>\n#include "dbgsom_b200.h"\n'
        'int main(void) { printf("%zu %zu %zu %d\\n", sizeof(dbgsom_bmu_args), sizeof(dbgsom_accumulate_args), '
        "sizeof(dbgsom_smooth_args), DBGSOM_ABI_VERSION); return 0; }\n"
    )
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out] == [ctypes.sizeof(nat.BmuArgs), ctypes.sizeof(nat.AccumulateArgs),
                                     ctypes.sizeof(nat.SmoothArgs), nat.ABI_VERSION]


def test_engine_refuses_to_run_without_cuda():
    import torch

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from dbgsom_b200.engine import DeviceEngine

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        DeviceEngine()
