"""dctd_l1_topk_large (exact L1 top-k for k up to 8192): workspace sizes and argument checks, before any CUDA call.  The
k limit of dctd_l1_topk stays where it was.  No device needed."""
import ctypes as C
import os

import pytest

from dctdomain_b200 import _lib


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def test_workspace_sizes(lib):
    for k in (993, 1024, 4096, 8192):
        for nq, n in ((1, 0), (1, 1), (5, 65_553), (2048, 1_000_000), (2049, 10), (8192, 50_000_000)):
            ws = lib.dctd_l1_topk_large_workspace_bytes(nq, n, 480, k)
            assert ws >= min(nq, 2048) * 16384 * 8, (k, nq, n)       # the candidate lists of one chunk of queries
            assert ws < 300 << 20, (k, nq, n)                        # chunked: a few hundred MB whatever nq is
        for d in (1, 16, 1024, 2048):
            assert lib.dctd_l1_topk_large_workspace_bytes(7, 100_000, d, k) > 0
    assert lib.dctd_l1_topk_large_workspace_bytes(8192, 50_000_000, 480, 1) > 0     # small k too (cross-checks)
    assert lib.dctd_l1_topk_large_workspace_bytes(5, 1000, 480, 8193) == 0
    assert lib.dctd_l1_topk_large_workspace_bytes(5, 1000, 2049, 1024) == 0
    assert lib.dctd_l1_topk_large_workspace_bytes(5, 1000, 480, 0) == 0
    assert lib.dctd_l1_topk_large_workspace_bytes(0, 1000, 480, 1024) == 0
    assert lib.dctd_l1_topk_large_workspace_bytes(5, -1, 480, 1024) == 0
    assert lib.dctd_l1_topk_workspace_bytes(8, 1000, 480, 993) == 0              # the heap path's limit is unchanged


def test_large_rejects_bad_arguments_without_a_device(lib):
    fake = C.c_void_p(0x1000)          # never dereferenced: every call below fails its argument check first
    big = 1 << 40

    def call(q=fake, nq=5, packed=fake, n=100_000, d=480, k=2048, id_base=0, dist=fake, ids=fake, keys=None, ws=fake,
             ws_bytes=big):
        return lib.dctd_l1_topk_large(q, nq, packed, n, d, k, id_base, dist, ids, keys, ws, ws_bytes, None)
    lib.dctd_launch_count(1)
    assert call(nq=-1) == _lib.ERR_ARG
    assert call(n=-1) == _lib.ERR_ARG
    assert call(k=0) == _lib.ERR_ARG
    assert call(d=0) == _lib.ERR_ARG
    assert call(id_base=-1) == _lib.ERR_ARG
    assert call(k=8193) == _lib.ERR_UNSUPPORTED
    assert call(d=2049) == _lib.ERR_UNSUPPORTED
    assert call(nq=0) == _lib.OK                                     # nothing to do
    assert call(q=None) == _lib.ERR_ARG
    assert call(dist=None) == _lib.ERR_ARG                          # ids without distances
    assert call(ids=None, keys=fake) == _lib.ERR_ARG
    assert call(dist=None, ids=None) == _lib.ERR_ARG                # no output at all
    assert call(packed=None) == _lib.ERR_ARG
    assert call(n=1 << 40) == _lib.ERR_UNSUPPORTED                   # positions need 40 bits
    assert call(id_base=(1 << 40) - 100_000) == _lib.ERR_UNSUPPORTED
    assert call(ws=None) == _lib.ERR_WORKSPACE
    need = lib.dctd_l1_topk_large_workspace_bytes(5, 100_000, 480, 2048)
    assert call(ws_bytes=need - 1) == _lib.ERR_WORKSPACE
    assert call(ws=C.c_void_p(0x1080)) == _lib.ERR_ARG               # workspace not 256-byte aligned
    assert call(packed=C.c_void_p(0x1008)) == _lib.ERR_ARG           # packed database not 16-byte aligned
    assert lib.dctd_launch_count(1) == 0


def test_merges_take_k_up_to_8192(lib):
    fake = C.c_void_p(0x1000)
    lib.dctd_launch_count(1)
    assert lib.dctd_l1_keys_merge(fake, 2, 5, 8193, fake, fake, None, None) == _lib.ERR_ARG
    assert lib.dctd_l1_keys_merge(fake, 33, 5, 4096, fake, fake, None, None) == _lib.ERR_ARG
    assert lib.dctd_l1_keys_merge(fake, 2, 5, 4096, None, None, None, None) == _lib.ERR_ARG
    assert lib.dctd_l1_keys_merge(fake, 2, 0, 4096, None, None, fake, None) == _lib.OK
    assert lib.dctd_l1_topk_merge(fake, fake, 2, 5, 8193, fake, fake, None) == _lib.ERR_ARG
    assert lib.dctd_l1_topk_merge(fake, fake, 2, 0, 8192, fake, fake, None) == _lib.OK
    assert lib.dctd_launch_count(1) == 0
