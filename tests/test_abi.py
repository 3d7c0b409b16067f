"""The C-ABI library loads on a CPU-only box, exports every symbol include/recoup_b200.h
declares, and refuses to compute without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "recoup_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rcp_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported_and_bound():
    from recoup_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 25
    for name in names:
        assert hasattr(_lib.lib, name), "librecoup_b200.so does not export %s" % name
    assert sorted(_lib.SIGNATURES) == names, "ctypes table and header disagree"
    assert _lib.lib.rcp_abi_version() == 1


def test_no_oracle_import_in_product():
    pkg = os.path.join(ROOT, "recoup_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "oracle/" not in src or f.endswith((".cuh", ".cu")), f


def gpu_visible():
    """Asks the CUDA driver: a machine's GPU need not appear as /dev/nvidia0 (a container may
    expose only, say, /dev/nvidia3)."""
    import torch
    return torch.cuda.is_available()


@pytest.mark.skipif(gpu_visible(), reason="GPU box: compute works there")
def test_compute_fails_loudly_without_gpu():
    import recoup_b200 as rb
    from recoup_b200 import _lib
    assert _lib.lib.rcp_init(0) == _lib.RCP_ERR_NOGPU
    assert b"no CPU fallback" in _lib.lib.rcp_last_error()
    h = C.c_int(0)
    clen = np.array([1000], dtype=np.int64)
    rc = _lib.lib.rcp_reads_load(0, None, None, None, None, 1,
                                 clen.ctypes.data_as(C.POINTER(C.c_int64)), 0, 0, C.byref(h))
    assert rc == _lib.RCP_ERR_NOGPU
    gr = rb.GRanges(np.zeros(3, np.int32), [1, 5, 9], [4, 8, 12], seqlevels=["c0"], seqlengths=[1000])
    mask = rb.GRanges(np.zeros(1, np.int32), [1], [10], seqlevels=["c0"])
    with pytest.raises(rb.RecoupError) as ei:
        rb.calcCoverage(gr, mask)
    assert ei.value.code == _lib.RCP_ERR_NOGPU
