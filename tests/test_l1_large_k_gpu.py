"""Exact L1 search for 992 < k <= 8192 (dctd_l1_topk_large, csrc/l1_large.cuh), bit for bit against the exact oracle.

Every case checks (dist, ids) of IndexFlatL1.search_device against oracle/search_oracle.l1_topk (the C restatement of
faiss) for up to 64 queries, or against the on-device brute force of test_l1_variants_gpu.py (itself checked against the
C oracle on a sample of rows) for more; the packed keys of search_keys_device with id_base = 2^33 + 5; that a second call
gives the same bytes; and the number of histogram passes the call needed (the first word of its workspace): 0 when the
database fits the candidate list, 1 normally, and the position-bit levels when many keys share the k-th distance."""
import argparse
import functools
import logging
import os

import numpy as np
import pytest
import torch

import synth
from minidb import MiniDB
from oracle import search_oracle as so
from test_l1_variants_gpu import brute_force

pytestmark = pytest.mark.gpu
ID_BASE = (1 << 33) + 5
CAND = 16384                # kLargeCand: candidate slots per query
CHUNK = 2048                # kLargeChunk: queries per internal chunk
THREADS = len(os.sched_getaffinity(0))
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@functools.lru_cache(maxsize=2)
def database(d, n, data='std'):
    """(db int8 [n, d], queries int8 [2100, d]).  Queries alternate between database rows and rows perturbed by +-2; the
    first query's row is duplicated on both sides of a group boundary and in the last group.
    data = 'tied': 20 000 rows at distance 5 from query 0 (more than the candidate list at the k-th distance);
    'same': every row equal to query 0."""
    rs = np.random.RandomState(d * 131 + n % 9973)
    db = rs.randint(-128, 128, size=(n, d), dtype=np.int8)
    nq = 2100
    q = db[rs.randint(0, max(n, 1), size=nq)].copy() if n else rs.randint(-128, 128, size=(nq, d), dtype=np.int8)
    q[1::2] = np.clip(q[1::2].astype(np.int16) + rs.randint(-2, 3, size=q[1::2].shape), -128, 127).astype(np.int8)
    if n >= 200:
        db[[62, 63, 64, 65, n - 1]] = q[0]
    if data == 'tied':
        cols = rs.randint(0, d, size=20_000)
        rows = np.repeat(q[0][None, :].astype(np.int16), 20_000, axis=0)
        r = np.arange(20_000)
        rows[r, cols] += np.where(rows[r, cols] + 5 <= 127, 5, -5)
        db[10_000:30_000] = rows.astype(np.int8)
    elif data == 'same':
        db[:] = q[0]
    return db, q


@functools.lru_cache(maxsize=2)
def index(d, n, data='std'):
    from dctdomain_b200 import index as dindex
    idx = dindex.IndexFlatL1(d)
    idx.add(database(d, n, data)[0])
    return idx


def reference(db, q, k):
    if len(q) <= 64:
        return so.l1_topk(q, db, k, threads=THREADS)
    dm, im = brute_force(db, q, k)
    rows = np.unique(np.concatenate([np.random.RandomState(len(q)).choice(len(q), 16, replace=False),
                                     np.arange(len(q) - 4, len(q))]))
    dm2, im2 = so.l1_topk(q[rows], db, k, threads=THREADS)
    assert np.array_equal(im[rows], im2) and np.array_equal(dm[rows], dm2), 'the brute force disagrees with the C oracle'
    return dm, im


def as_keys(dm, im, id_base):
    keys = (np.where(im < 0, 0, dm).astype(np.int64) << 40) | (im + id_base)
    return np.where(im < 0, -1, keys)


def call_large(idx, qd, k, id_base=0):
    """dctd_l1_topk_large with both output forms at once -> (dist, ids, keys, histogram passes)."""
    from dctdomain_b200 import _lib
    L = _lib.lib()
    nq = int(qd.shape[0])
    need = L.dctd_l1_topk_large_workspace_bytes(nq, idx.ntotal, idx.d, k)
    assert need > 0
    ws = torch.full((need,), 0x5a, dtype=torch.uint8, device='cuda')        # garbage: nothing may rely on zeros
    dist = torch.empty((nq, k), dtype=torch.float32, device='cuda')
    ids = torch.empty((nq, k), dtype=torch.int64, device='cuda')
    keys = torch.empty((nq, k), dtype=torch.int64, device='cuda')
    packed = idx._packed.data_ptr() if idx._packed is not None else 0
    rc = L.dctd_l1_topk_large(qd.data_ptr(), nq, packed, idx.ntotal, idx.d, k, id_base, dist.data_ptr(), ids.data_ptr(),
                              keys.data_ptr(), ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, 'dctd_l1_topk_large')
    torch.cuda.synchronize()
    return dist, ids, keys, int(ws[:4].view(torch.int32)[0])


def _equal(what, got, want):
    bad = np.argwhere(got != want)
    assert not len(bad), f'{what}: {len(bad)} entries differ, first (query, rank): {bad[:6].tolist()}, ' \
                         f'got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}'


def check(d, n, nq, k, data='std', passes=None):
    db, q = database(d, n, data)
    idx = index(d, n, data)
    qd = torch.from_numpy(q[:nq]).cuda()
    dist, ids = idx.search_device(qd, k)
    dm, im = reference(db, q[:nq], k)
    _equal('ids', ids.cpu().numpy(), im)
    _equal('distances', dist.cpu().numpy(), dm)
    dist2, ids2 = idx.search_device(qd, k)
    assert torch.equal(dist, dist2) and torch.equal(ids, ids2), 'a second call gave different bytes'
    keys = idx.search_keys_device(qd, k, id_base=ID_BASE)
    _equal('keys', keys.cpu().numpy(), as_keys(dm, im, ID_BASE))
    d3, i3, k3, levels = call_large(idx, qd, k, ID_BASE)
    _equal('ids (both forms)', i3.cpu().numpy() - ID_BASE * (im >= 0), im)
    _equal('keys (both forms)', k3.cpu().numpy(), as_keys(dm, im, ID_BASE))
    if passes is None:
        passes = 0 if n <= CAND else 1
    assert levels == passes, f'{levels} histogram passes, expected {passes}'
    return db, q, dm


CASES = (
    [(480, 65_553, 5, k) for k in (993, 1024, 2048, 4096, 8191, 8192)]           # k range
    + [(dd, 16_385, 5, 2048) for dd in (16, 100, 1024, 2048)]                    # widths
    + [(480, 65_553, nq, 1024) for nq in (1, 64, 300)]                            # query counts
    + [(100, 16_385, CHUNK + 52, 993)]                                            # crosses the internal query chunk
    + [(100, n, 5, 993) for n in (0, 1, 993, 16_384, 16_385)]                     # k > n, k = n, the collect-only limit
    + [(16, 4096, 7, 4096), (16, 8000, 3, 8192)]                                  # k = n; k > n above 4096
    + [(480, 1_000_000, 16, 4096)]
)


@pytest.mark.parametrize('d,n,nq,k', CASES, ids=[f'd{c[0]}-n{c[1]}-nq{c[2]}-k{c[3]}' for c in CASES])
def test_large_k_matches_oracle(d, n, nq, k):
    check(d, n, nq, k)


def test_k_tied_at_the_kth_distance_takes_the_position_levels():
    """20 000 rows at the k-th distance: the distance levels cannot separate them (level 0: bins of 256 distance units,
    level 1: single distances), level 2 splits positions."""
    db, q, dm = check(480, 65_553, 5, 4096, data='tied', passes=3)
    full = np.abs(db.astype(np.int16) - q[0].astype(np.int16)).sum(axis=1)
    assert dm[0, -1] == 5 and (full == 5).sum() > CAND


def test_identical_rows():
    """Every row at the same distance from every query: the window narrows through the position bits only."""
    check(480, 65_553, 5, 8192, data='same', passes=3)
    check(480, 65_553, 3, 993, data='same', passes=3)


@pytest.mark.parametrize('nq', [5, 300])
@pytest.mark.parametrize('k', [50, 992])
def test_small_k_equals_the_heap_and_threshold_paths(nq, k):
    """dctd_l1_topk_large accepts k <= 992 too: the same bytes as dctd_l1_topk (threshold path for these sizes)."""
    idx = index(480, 65_553)
    qd = torch.from_numpy(database(480, 65_553)[1][:nq]).cuda()
    dist, ids = idx.search_device(qd, k)
    d2, i2, k2, _ = call_large(idx, qd, k, 0)
    assert torch.equal(dist, d2) and torch.equal(ids, i2)
    assert torch.equal(idx.search_keys_device(qd, k, id_base=ID_BASE), call_large(idx, qd, k, ID_BASE)[2])


def test_limits():
    from dctdomain_b200 import _lib
    idx = index(100, 993)
    qd = torch.from_numpy(database(100, 993)[1][:3]).cuda()
    with pytest.raises(_lib.DctdError, match='k <= 8192') as e:
        idx.search_device(qd, 8193)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    with pytest.raises(_lib.DctdError, match='k <= 8192'):
        idx.search_keys_device(qd, 8193)
    with pytest.raises(ValueError):
        idx.search_keys_device(qd, 993, bound=torch.zeros(3, dtype=torch.int32, device='cuda'))


@pytest.mark.parametrize('g', [2, 3, 8])
def test_merge_of_shards_equals_whole(g):
    """A database split into g indexes (id_base = first position): keys_merge and dctd_l1_topk_merge of their k = 4096
    results equal the single-index result - the exchange step of ShardedIndex at k > 992."""
    from dctdomain_b200 import index as dindex
    from dctdomain_b200.sharded import merge_parts, shard_bounds
    d, n, nq, k = 100, 40_000, 9, 4096
    db, q = database(d, n)
    qd = torch.from_numpy(q[:nq]).cuda()
    whole_d, whole_i = index(d, n).search_device(qd, k)
    keys, dps, ips = [], [], []
    for r in range(g):
        b, e = shard_bounds(n, g, r)
        sh = dindex.IndexFlatL1(d)
        sh.add(db[b:e])
        keys.append(sh.search_keys_device(qd, k, id_base=b))
        dp, ip = sh.search_device(qd, k, id_base=b)
        dps.append(dp)
        ips.append(ip)
    md, mi = dindex.keys_merge(torch.stack(keys))
    assert torch.equal(mi, whole_i) and torch.equal(md, whole_d)
    mk = dindex.keys_merge(torch.stack(keys), want_keys=True)
    assert torch.equal(mk, torch.from_numpy(as_keys(whole_d.cpu().numpy(), whole_i.cpu().numpy(), 0)).cuda())
    pd, pi = merge_parts(torch.stack(dps), torch.stack(ips))
    assert torch.equal(pi, whole_i) and torch.equal(pd, whole_d)


def _worker(rank, world, port, out_dir):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, 'tests')]
    import torch.distributed as dist
    from dctdomain_b200.sharded import ShardedIndex
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    db, q = database(100, 40_000)
    sh = ShardedIndex(100, len(db))
    sh.add_local(db[sh.begin:sh.end])
    d, i = sh.search(torch.from_numpy(q[:40]).cuda(), 2048)
    ds, is_, qb, qe = sh.search_slice(torch.from_numpy(q[:40]).cuda(), 2048)
    np.savez(os.path.join(out_dir, f'r{rank}.npz'), d=d.cpu().numpy(), i=i.cpu().numpy(), ds=ds.cpu().numpy(),
             is_=is_.cpu().numpy(), qb=qb, qe=qe, path=sh.last_path)
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_two_ranks_k2048(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    db, q = database(100, 40_000)
    dm, im = so.l1_topk(q[:40], db, 2048, threads=THREADS)
    for r in range(2):
        z = np.load(tmp_path / f'r{r}.npz')
        assert np.array_equal(z['i'], im) and np.array_equal(z['d'], dm)
        qb, qe = int(z['qb']), int(z['qe'])
        assert np.array_equal(z['is_'], im[qb:qe]) and np.array_equal(z['ds'], dm[qb:qe])
        assert str(z['path']) == 'all_to_all'


def _search_db_lines(fp, qp, khits, tmp_path, caplog):
    """(lines of search_db, lines of the reference's loop: one index.search per query protein) for the fingerprint
    tables fp (database) and qp (queries), both in the layout of tests/golden/example-dct.npz."""
    from dctdomain_b200 import index as dindex
    from dctdomain_b200 import query_db as dq
    dbp, qbp = str(tmp_path / 'fp.db'), str(tmp_path / 'q.db')
    MiniDB(dbp, fp).close()
    MiniDB(qbp, qp).close()
    idx = dindex.IndexFlatL2(fp['dct'].shape[1])
    idx.add(fp['dct'])
    with caplog.at_level(logging.INFO):
        dq.search_db(argparse.Namespace(khits=khits), MiniDB(qbp), MiniDB(dbp), index=idx)
    got = [r.getMessage() for r in caplog.records if r.getMessage().startswith('Query:')]

    def labels(z):
        out = []
        for p, pid in enumerate(z['sid']):
            out += [(str(pid), str(z['dom'][f])) for f in range(int(z['idx'][p]), int(z['idx'][p + 1]))]
        return out
    db_labels, q_labels = labels(fp), labels(qp)
    qdb = MiniDB(qbp)
    order = [pid for (pid,) in qdb.cur.execute('SELECT pid FROM sequences').fetchall()]
    qdb.close()
    sids = [str(s) for s in qp['sid']]
    want = []
    for pid in order:
        p = sids.index(pid)
        a, b = int(qp['idx'][p]), int(qp['idx'][p + 1])
        if b > a:
            dm, im = so.l1_topk(qp['dct'][a:b], fp['dct'], khits, threads=THREADS)
            want += so.top_hits_lines(dm, im, khits, q_labels[a:b], db_labels)
    return got, want


def test_search_db_khits_1000_on_the_example_database(tmp_path, caplog):
    """query_db --khits 1000 of the 43-row example database against itself: every slot past row 43 is padding."""
    z = np.load(os.path.join(G, 'example-dct.npz'))
    z = {f: z[f] for f in z.files}
    got, want = _search_db_lines(z, z, 1000, tmp_path, caplog)
    assert len(want) == 43 * 43 and got == want


def test_search_db_khits_2000(tmp_path, caplog):
    """query_db --khits 2000 against 2000+ fingerprints: three query proteins, 2000 hits each."""
    rs = np.random.RandomState(3)
    n_prot = 700
    idx = np.concatenate([[0], np.cumsum(rs.randint(2, 5, size=n_prot))])
    dct = synth.fingerprints(7, int(idx[-1]))
    dct[100:130] = dct[5]                                   # ties at one distance across proteins
    fp = {'sid': np.array([f'P{i:05d}' for i in range(n_prot)]), 'idx': idx, 'dct': dct,
          'dom': np.array([f'{1 + j}-{40 + j}' for j in range(len(dct))])}
    rows = np.array([5, 6, 7, 200, 1500, 1501])
    qp = {'sid': np.array(['Q1', 'Q2', 'Q3']), 'idx': np.array([0, 3, 4, 6]), 'dct': dct[rows],
          'dom': np.array([f'{1 + j}-{30 + j}' for j in range(len(rows))])}
    assert len(dct) > 2000
    got, want = _search_db_lines(fp, qp, 2000, tmp_path, caplog)
    assert len(want) == 3 * 2000 and got == want
