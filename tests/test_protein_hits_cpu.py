"""dctd_l1_protein_hits checks its arguments before it touches CUDA, and dct_sim's distance cut follows the float64
similarity formula.  No device needed."""
import ctypes as C
import os

import numpy as np
import pytest

from dctdomain_b200 import _lib


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def test_protein_hits_rejects_bad_arguments_without_a_device(lib):
    fake = C.c_void_p(0x1000)          # never dereferenced: every call below fails its argument check first
    qoff = np.array([0, 2, 3], dtype=np.int64)
    doff = np.array([0, 1, 1, 4], dtype=np.int64)
    out = [fake] * 4

    def call(qoff=qoff, nq=2, doff=doff, nd=3, d=480, top=5, clamp=17000, cut=12750, cap=32, outs=out):
        return lib.dctd_l1_protein_hits(fake, qoff.ctypes.data if qoff is not None else None, nq, fake,
                                        doff.ctypes.data if doff is not None else None, nd, d, top, clamp, cut, cap,
                                        *outs, fake, 1 << 20, None)
    assert call(nq=-1) == _lib.ERR_ARG
    assert call(nd=-1) == _lib.ERR_ARG
    assert call(d=0) == _lib.ERR_ARG
    assert call(cap=0) == _lib.ERR_ARG
    assert call(clamp=-1) == _lib.ERR_ARG
    assert call(qoff=None) == _lib.ERR_ARG
    assert call(doff=None) == _lib.ERR_ARG
    assert call(qoff=np.array([0, 2, 1], dtype=np.int64)) == _lib.ERR_ARG         # decreasing offsets
    assert call(doff=np.array([0, 3, 1, 4], dtype=np.int64)) == _lib.ERR_ARG
    assert call(qoff=np.array([1, 2, 3], dtype=np.int64)) == _lib.ERR_ARG         # not starting at 0
    for i in range(4):                                                             # a null output
        assert call(outs=out[:i] + [None] + out[i + 1:]) == _lib.ERR_ARG
    assert call(cap=993) == _lib.ERR_UNSUPPORTED                                  # longer rows than the scan's k limit
    assert call(d=4096) == _lib.ERR_UNSUPPORTED                                   # too wide for the tiles
    assert call(nq=0) == _lib.OK                                                  # nothing to do


def test_protein_hits_workspace_sizes_host_logic(lib):
    for nq, nd, cap in [(1, 1, 1), (10, 43, 32), (10_000, 1_000_000, 32), (100_000, 1000, 992), (3, 5, 992)]:
        ws = lib.dctd_l1_protein_hits_workspace_bytes(nq * 5, nq, nd * 5, nd, 480, 5, cap)
        assert ws >= (nd + 31) // 32 * 32 * 480 + min(nq, 1 << 16) * cap * 8
    assert lib.dctd_l1_protein_hits_workspace_bytes(5, 1, 5, 1, 480, 5, 993) == 0
    assert lib.dctd_l1_protein_hits_workspace_bytes(5, 1, 5, 1, 4096, 5, 32) == 0
    assert lib.dctd_l1_protein_hits_workspace_bytes(5, 1, 5, 1, 1024, 5, 32) > 0  # wide vectors: one group per stage


def test_dist_cut_is_the_last_distance_the_float64_similarity_passes():
    from dctdomain_b200.dct_sim import _dist_cut, _sim
    for thr in (0.25, 0.3, 0.5, 0.999, 1.0, 1e-9, 0.7654321):
        cut = _dist_cut(thr)
        assert 0 <= cut < 17000
        assert _sim(cut) >= thr and _sim(cut + 1) < thr
    assert _dist_cut(1.5) == -1 and _dist_cut(1.0 + 1e-12) == -1
    assert _dist_cut(0) == 17000 and _dist_cut(-1) == 17000 and _dist_cut(float('nan')) == 17000
