"""CPU: the C-ABI library builds for sm_100a (nvcc cross-compiles without a GPU), loads, and exports every
symbol include/bde2vid.h declares; the ctypes mirror of bde_gemm_desc matches the C layout."""
import ctypes
import os
import re
import subprocess

import pytest

from conftest import ROOT


def header_symbols():
    text = open(os.path.join(ROOT, "include", "bde2vid.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bde_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib_built):
    lib = ctypes.CDLL(lib_built)
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), "libbde2vid_sm100.so does not export %s" % s
    lib.bde_abi_version.restype = ctypes.c_int
    assert lib.bde_abi_version() == 3
    lib.bde_last_error.restype = ctypes.c_char_p
    assert lib.bde_last_error() is not None


def test_python_binding_covers_header(lib_built):
    from bde2vid_b200 import _lib
    lib = _lib.load()
    missing = [s for s in header_symbols() if s not in _lib.EXPORTS]
    assert not missing, "ctypes prototypes missing for %s" % missing
    assert lib.bde_window_attention_mma_bias_stride(147) == 168
    assert lib.bde_window_attention_mma_bias_stride(98) == 104
    assert lib.bde_window_attention_mma_bias_stride(245) == 0


def test_gemm_desc_layout_matches_c(tmp_path):
    from bde2vid_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\n'
                   'int main(){printf("%%zu %%zu %%zu %%zu %%zu\\n", sizeof(bde_gemm_desc), offsetof(bde_gemm_desc, w),'
                   ' offsetof(bde_gemm_desc, ln_frames), offsetof(bde_gemm_desc, epi), offsetof(bde_gemm_desc, out2));return 0;}\n'
                   % os.path.join(ROOT, "include", "bde2vid.h"))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = _lib.GemmDesc
    assert got == [ctypes.sizeof(D), D.w.offset, D.ln_frames.offset, D.epi.offset, D.out2.offset]


def test_ops_fail_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from bde2vid_b200 import ops
    with pytest.raises(RuntimeError):
        ops.cast(torch.zeros(4), torch.zeros(4))
