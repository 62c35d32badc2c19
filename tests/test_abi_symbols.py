"""The C-ABI shared library loads on a CPU-only box and exports every symbol include/liuzhou_b200.h declares
(no compute calls without a GPU)."""
import ctypes
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    text = (ROOT / "include" / "liuzhou_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lzb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from liuzhou_b200 import build

    lib_path = build.build()
    lib = ctypes.CDLL(str(lib_path))
    names = _declared()
    assert len(names) >= 15
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in include/liuzhou_b200.h but not exported: {missing}"
    lib.lzb_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.lzb_version()


def test_library_is_sm100a_only():
    import subprocess

    from liuzhou_b200 import build

    cuobjdump = str(Path(build.nvcc()).with_name("cuobjdump"))
    out = subprocess.run([cuobjdump, "-lelf", str(build.build())], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_ops_refuse_cpu_tensors():
    import pytest
    import torch

    from liuzhou_b200 import v0_core

    z = torch.zeros((2, 6, 6), dtype=torch.int8)
    b = torch.zeros((2, 6, 6), dtype=torch.bool)
    s = torch.zeros((2,), dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        v0_core.encode_actions_fast(z, b, b, s, s, s, s, s, s, s, 36, 144, 36, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        v0_core.root_puct_allocate_visits(torch.zeros(2, 3), torch.zeros(2, 3), torch.ones(2, 3, dtype=torch.bool), 4, 1.0)
