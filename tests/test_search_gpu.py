"""Parity of the CUDA search path (through the C ABI) with the CPU oracle and the reference's shipped
fixtures.  Integer work: everything here is bit exact, including hit order with ties by index."""
import argparse
import logging
import os

import numpy as np
import pytest
import torch

import synth
from minidb import MiniDB
from oracle import search_oracle as so

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _index(db, metric_l1=True, pieces=1):
    from dctdomain_b200 import index as dindex
    idx = dindex.IndexFlatL2(db.shape[1])
    for part in np.array_split(db, pieces):
        idx.add(part)
    if metric_l1:
        idx.metric_type = dindex.METRIC_L1
    return idx


def _check(q, db, k, pieces=1):
    dm, im = _index(db, pieces=pieces).search(q, k)
    dm2, im2 = so.l1_topk(q, db, k, threads=4)
    assert dm.dtype == np.float32 and im.dtype == np.int64 and dm.shape == (len(q), k)
    assert np.array_equal(im, im2), np.argwhere(im != im2)[:5]
    assert np.array_equal(dm, dm2)


def test_example_fixture_all_vs_all():
    z = np.load(os.path.join(G, 'example-dct.npz'))
    _check(z['dct'], z['dct'], 50)          # N = 43 < k: (-1, FLT_MAX) padding
    _check(z['dct'], z['dct'], 5)


@pytest.mark.parametrize('n', [1, 31, 32, 33, 129, 5000])
@pytest.mark.parametrize('k', [1, 50, 100])
def test_sizes(n, k):
    db = synth.fingerprints(n, n)
    q = synth.fingerprints(n + 1, 13)
    _check(q, db, k)


@pytest.mark.parametrize('k', [7, 96, 97, 224, 225, 300, 480, 481, 992])
def test_k_range(k):
    db = synth.fingerprints(3, 3000)
    _check(db[:9], db, k)


@pytest.mark.parametrize('nq', [1, 8, 9, 64, 65, 1000])
def test_query_counts(nq):
    db = synth.fingerprints(5, 20000)
    q = np.concatenate([db[:nq // 2], synth.fingerprints(6, nq - nq // 2)])
    _check(q, db, 50)


def test_boundary_ties_and_duplicates():
    rs = np.random.RandomState(0)
    db = rs.randint(0, 3, size=(4000, 480)).astype(np.int8)        # tiny alphabet: massive distance ties
    db[100:140] = db[7]                                            # exact duplicates of one vector
    db[3000:3100] = db[7]
    _check(db[:40], db, 50)
    _check(db[:40], db, 10)
    same = np.tile(synth.fingerprints(1, 1), (2000, 1))            # every distance equal: ids 0..k-1 win
    dm, im = _index(same).search(same[:3], 50)
    assert (im == np.arange(50)[None, :]).all() and (dm == 0).all()


def test_negative_values_and_other_dims():
    rs = np.random.RandomState(1)
    for d in (16, 100, 480, 481, 1024):
        db = rs.randint(-128, 128, size=(1500, d)).astype(np.int8)
        _check(db[:20], db, 20)


def test_add_in_pieces_and_roundtrip(tmp_path):
    from dctdomain_b200 import index as dindex
    db = synth.fingerprints(9, 1000)
    idx = _index(db, pieces=7)
    assert idx.ntotal == 1000 and np.array_equal(idx.reconstruct_n(), db)
    _check(db[:30], db, 50, pieces=7)
    path = str(tmp_path / 'x.index')
    idx = _index(db, metric_l1=False, pieces=7)   # the reference writes the IndexFlatL2 it built (src/database.py:241-243)
    dindex.write_index(idx, path)
    raw = open(path, 'rb').read()
    assert raw[:4] == b'IxF2' and len(raw) == 4 + 4 + 8 * 3 + 1 + 4 + 8 + 1000 * 480 * 4
    back = dindex.read_index(path)
    assert back.ntotal == 1000 and back.d == 480 and back.metric_type == dindex.METRIC_L2
    with pytest.raises(NotImplementedError):
        back.search(db[:2], 5)                 # like the reference, the caller must flip to METRIC_L1
    back.metric_type = dindex.METRIC_L1
    dm, im = back.search(db[:30], 50)
    dm2, im2 = so.l1_topk(db[:30], db, 50)
    assert np.array_equal(im, im2) and np.array_equal(dm, dm2)
    with pytest.raises(ValueError):
        idx.add(np.full((1, 480), 0.5))        # not int8 valued
    # int8 sidecar: used when it matches the .index, ignored (and removed on rewrite) otherwise
    dindex.write_index(idx, path, sidecar=True)
    hdr = 8 + 4 + 8 + 8 + 16                                  # magic, d, ntotal, .index size, payload digest
    assert os.path.getsize(path + '.i8') == hdr + 1000 * 480 and open(path, 'rb').read() == raw
    side = dindex.read_index(path)
    assert np.array_equal(side.reconstruct_n(), db)
    with open(path + '.i8', 'r+b') as f:                      # corrupt the payload: proves the sidecar is what was read
        f.seek(hdr)
        f.write(bytes([db[0, 0] ^ 1]))
    assert dindex.read_index(path).reconstruct_n()[0, 0] == (db[0, 0] ^ 1)
    # the .index rewritten by another tool with the SAME shape but different vectors (what faiss itself would do): the
    # stale sidecar must be ignored - size, d and ntotal all still match, only the payload digest tells
    db2 = db.copy()
    db2[0] = db[1]
    db2[-1] = db[2]
    with open(path, 'r+b') as f:
        f.seek(len(raw) - 1000 * 480 * 4)
        f.write(db2.astype(np.float32).tobytes())
    assert np.array_equal(dindex.read_index(path).reconstruct_n(), db2)
    # an index that carries METRIC_L1 keeps it through a round trip (faiss: fourcc IxFl, metric_type 2, metric_arg)
    l1 = dindex.IndexFlatL1(480)
    l1.add(db[:100])
    dindex.write_index(l1, path)
    raw1 = open(path, 'rb').read()
    assert raw1[:4] == b'IxFl' and len(raw1) == 4 + 4 + 8 * 3 + 1 + 4 + 4 + 8 + 100 * 480 * 4
    back1 = dindex.read_index(path)
    assert back1.metric_type == dindex.METRIC_L1 and back1.ntotal == 100
    assert np.array_equal(back1.search(db[:3], 5)[1], so.l1_topk(db[:3], db[:100], 5)[1])
    other = _index(db[:500])
    dindex.write_index(other, path)                           # rewrite without a sidecar: the stale one goes away
    assert not os.path.exists(path + '.i8') and dindex.read_index(path).ntotal == 500


def test_empty_database_and_empty_queries():
    from dctdomain_b200 import index as dindex
    idx = dindex.IndexFlatL1(480)
    dm, im = idx.search(synth.fingerprints(0, 3), 5)
    assert (im == -1).all() and (dm == np.finfo(np.float32).max).all()
    idx.add(synth.fingerprints(0, 10))
    dm, im = idx.search(np.zeros((0, 480), dtype=np.int8), 5)
    assert dm.shape == (0, 5)


def test_merge_of_sharded_results_equals_whole():
    """What the multi-GPU path does: contiguous shards, per-shard top-k with id_base, k-way merge."""
    from dctdomain_b200 import _lib
    db = synth.fingerprints(21, 10000)
    db[5000:5050] = db[3]                      # ties across shard boundaries
    q = torch.from_numpy(db[:100]).cuda()
    k, parts = 50, 4
    dists, ids = [], []
    bounds = np.linspace(0, len(db), parts + 1).astype(int)
    for s in range(parts):
        idx = _index(db[bounds[s]:bounds[s + 1]])
        d_, i_ = idx.search_device(q, k, id_base=int(bounds[s]))
        dists.append(d_)
        ids.append(i_)
    dp, ip = torch.stack(dists).contiguous(), torch.stack(ids).contiguous()
    out_d = torch.empty((100, k), dtype=torch.float32, device='cuda')
    out_i = torch.empty((100, k), dtype=torch.int64, device='cuda')
    rc = _lib.lib().dctd_l1_topk_merge(dp.data_ptr(), ip.data_ptr(), parts, 100, k, out_d.data_ptr(),
                                       out_i.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc)
    dm2, im2 = so.l1_topk(db[:100], db, k, threads=4)
    assert np.array_equal(out_i.cpu().numpy(), im2) and np.array_equal(out_d.cpu().numpy(), dm2)


def test_search_db_reproduces_example_search_txt(tmp_path, caplog):
    """reference test/test/example-search.txt = query_db.py --khits 50 of the example db against itself."""
    from dctdomain_b200 import query_db as dq
    z = np.load(os.path.join(G, 'example-dct.npz'))
    dbp = str(tmp_path / 'example.db')
    MiniDB(dbp, z).close()
    idx = _index(z['dct'], metric_l1=False)
    with caplog.at_level(logging.INFO):
        dq.search_db(argparse.Namespace(khits=50), MiniDB(dbp), MiniDB(dbp), index=idx)
    lines = [r.getMessage() for r in caplog.records if r.getMessage().startswith('Query:')]
    assert lines == open(os.path.join(G, 'example-search.txt')).read().splitlines()


def test_dct_sim_pair_reproduces_g6pd(tmp_path):
    """reference bench/G6PD/G6PD-dctsim.txt = dct-sim.py --dct G6PD-dct.npz --pair G6PD.pair."""
    from dctdomain_b200 import dct_sim
    out = str(tmp_path / 'sim.txt')
    dct_sim.main(['--dct', os.path.join(G, 'G6PD-dct.npz'), '--pair', os.path.join(G, 'G6PD.pair'), '--output', out])
    assert open(out).read() == open(os.path.join(G, 'G6PD-dctsim.txt')).read()
    z = np.load(os.path.join(G, 'G6PD-dct.npz'))
    a, b = z['dct'][z['idx'][0]:z['idx'][1]], z['dct'][z['idx'][1]:z['idx'][2]]
    assert dct_sim.domain_sim(a, b) == so.domain_sim(a, b)
    assert dct_sim.prostSimilarity(a[0], b[0]) == so.prost_similarity(a[0], b[0])


def test_dct_sim_db_and_all(tmp_path, capsys):
    from dctdomain_b200 import dct_sim
    npz = os.path.join(G, 'example-dct.npz')
    z = np.load(npz)
    blocks = [z['dct'][z['idx'][i]:z['idx'][i + 1]] for i in range(len(z['sid']))]
    out = str(tmp_path / 'all.txt')
    dct_sim.main(['--dct', npz, '--output', out])
    want = ['#prot1 prot2 sim-domain sim-global']
    for i in range(len(blocks) - 1):
        for j in range(i + 1, len(blocks)):
            mx, s = so.domain_sim(blocks[i], blocks[j])
            want.append(f"{z['sid'][i]} {z['sid'][j]} {mx:.3f} {s:.3f}")
    assert open(out).read().splitlines() == want
    out = str(tmp_path / 'db.txt')
    dct_sim.main(['--dct', npz, '--db', npz, '--top', '3', '--threshold', '0.3', '--output', out])
    # the whole output against the UNMODIFIED reference's (tests/golden/make_dctsim_golden.py ran src/dct-sim.py)
    assert open(out).read() == open(os.path.join(G, 'example-dbsearch.txt')).read()
    out = str(tmp_path / 'db2.txt')
    dct_sim.main(['--dct', os.path.join(G, 'G6PD-dct.npz'), '--db', npz, '--output', out])      # default --top / --threshold
    assert open(out).read() == open(os.path.join(G, 'example-dbsearch-g6pd.txt')).read()
    assert open(str(tmp_path / 'all.txt')).read() == open(os.path.join(G, 'example-allsim.txt')).read()


@pytest.mark.parametrize('d', [480, 100, 16])
def test_protein_scores_all_pairs_vs_brute_force(d):
    """dctd_l1_protein_scores (tiled SAD kernel + per-pair reduction) against numpy over every fingerprint pair: proteins
    with 0, 1 and more than 8 fingerprints (a warp slice holds 8), query sets that do not fill a tile, a workspace small
    enough to force several chunks of query proteins; and against the one-warp-per-pair scorer."""
    from dctdomain_b200 import dct_sim
    rs = np.random.RandomState(d)

    def make(n_prot, hi):
        counts = rs.randint(0, hi, size=n_prot)
        counts[rs.randint(n_prot)] = 19
        counts[0] = 1
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        fps = rs.randint(-128, 128, size=(int(off[-1]), d)).astype(np.int8)
        return fps, off

    for (nq, nd, ws) in ((1, 1, None), (300, 150, None), (300, 150, 1 << 20), (37, 61, None)):
        qf, qoff = make(nq, 7)
        df, doff = make(nd, 9)
        dist = np.abs(qf[:, None, :].astype(np.int32) - df[None, :, :].astype(np.int32)).sum(axis=2)      # [NQ_f, ND_f]
        big = np.iinfo(np.int32).max
        want_min = np.full((nq, nd), big, dtype=np.int64)
        want_last = np.full((nq, nd), big, dtype=np.int64)
        for a in range(nq):
            for b in range(nd):
                blk = dist[qoff[a]:qoff[a + 1], doff[b]:doff[b + 1]]
                if blk.size:
                    want_min[a, b] = blk.min()
                    want_last[a, b] = blk[-1, -1]
        mn, last = dct_sim.protein_scores(qf, qoff, df, doff, workspace_bytes=ws)
        assert np.array_equal(mn, want_min) and np.array_equal(last, want_last)
    # the listed-pairs scorer agrees, INT32_MAX for the database proteins without fingerprints included
    cat = np.concatenate([qf, df])
    off = np.concatenate([qoff, doff[1:] + qoff[-1]])
    m1, l1 = dct_sim._pair_dists(cat, off, np.zeros(nd, dtype=np.int32), np.arange(nd, dtype=np.int32) + nq)
    assert (want_last[0] == big).any()
    assert np.array_equal(m1, want_min[0]) and np.array_equal(l1, want_last[0])


def test_properties_at_scale():
    """1M-vector database (configs[3] size): the oracle is too slow here, so check properties - every
    query that is a database row finds itself at distance 0 first, distances ascend, ids are unique, and
    a torch brute force over the same int8 data agrees on 64 of the queries."""
    db = synth.fingerprints(33, 1_000_000)
    idx = _index(db)
    rs = np.random.RandomState(2)
    rows = rs.choice(len(db), size=256, replace=False)
    dm, im = idx.search(db[rows], 50)
    assert (dm[:, 0] == 0).all() and (np.diff(dm, axis=1) >= 0).all()
    assert all(len(set(r)) == 50 for r in im)
    first = im[:, 0]
    assert all(np.array_equal(db[f], db[r]) for f, r in zip(first, rows))
    dbt = torch.from_numpy(db).cuda()
    for qi in range(64):          # an independent brute force (torch, int32 distances, one sort) on a quarter of the queries
        dist = (dbt.to(torch.int16) - dbt[rows[qi]].to(torch.int16)).abs().sum(dim=1, dtype=torch.int32)
        key = dist.to(torch.int64) * (1 << 32) + torch.arange(len(db), device='cuda')
        best = torch.sort(key)[0][:50]
        assert np.array_equal((best % (1 << 32)).cpu().numpy(), im[qi])
        assert np.array_equal((best // (1 << 32)).cpu().numpy().astype(np.float32), dm[qi])


# ---- large databases take the threshold path (sample -> thresholds -> one compaction pass -> select) ----
@pytest.mark.parametrize('nq', [1, 4, 5, 13, 16, 17, 64, 300])
def test_threshold_path_vs_oracle(nq):
    db = synth.fingerprints(51, 100_000)
    rs = np.random.RandomState(nq)
    q = db[rs.choice(len(db), nq, replace=False)].copy()
    q[::2] = np.clip(q[::2].astype(int) + rs.randint(-2, 3, size=q[::2].shape), 0, 127).astype(np.int8)
    _check(q, db, 50)


@pytest.mark.parametrize('k', [1, 10, 100, 256, 300])
def test_threshold_path_k_values(k):
    db = synth.fingerprints(52, 80_000)
    _check(db[1000:1024], db, k)


def test_threshold_path_overflow_falls_back_to_heap_scan():
    """Massive distance ties make the candidate list overflow: those queries are redone by the heap scan."""
    rs = np.random.RandomState(5)
    db = rs.randint(0, 2, size=(70_000, 480)).astype(np.int8)
    db[10_000:30_000] = db[3]                       # 20k exact duplicates of one vector
    q = np.concatenate([db[:6], db[10_000:10_004], rs.randint(0, 2, size=(30, 480)).astype(np.int8)])
    _check(q, db, 50)
    _check(q[:7], db, 20)                           # streaming kernel + fallback


@pytest.mark.parametrize('order', ['ascending', 'descending'])
def test_streaming_thresholds_on_sorted_database_with_ragged_tail(order):
    """Few queries take the streaming path whose thresholds come from lane minima over every 32nd group: a database
    sorted by distance to the query (the worst case for a strided sample), a size that is not a multiple of 32 (the
    padding lanes of the last group must not produce minima) and a k above the per-warp sample."""
    rs = np.random.RandomState(11)
    n = 70_000 + 17
    q = rs.randint(0, 128, size=(3, 480)).astype(np.int8)
    db = rs.randint(0, 128, size=(n, 480)).astype(np.int8)
    db[: n // 2] = np.clip(q[0].astype(int) + rs.randint(-20, 21, size=(n // 2, 480)), 0, 127).astype(np.int8)
    dist = np.abs(db.astype(np.int32) - q[0].astype(np.int32)).sum(axis=1)
    perm = np.argsort(dist, kind='stable')
    db = db[perm if order == 'ascending' else perm[::-1]]
    _check(q, db, 50)
    _check(q[:1], db, 256)


def test_threshold_and_heap_paths_agree_at_scale():
    import torch
    from dctdomain_b200 import index as dindex
    db = synth.fingerprints(53, 400_000)
    idx = _index(db)
    q = db[::4001][:100]
    a = idx.search(q, 50)
    # the same search forced onto the heap scan (flag DCTD_L1_HEAP_ONLY of dctd_l1_topk_keys), returned as packed keys
    keys = idx.search_keys_device(torch.from_numpy(q).cuda(), 50, heap_only=True)
    b = [t.cpu().numpy() for t in dindex.keys_merge(keys.view(1, len(q), 50))]
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    a = idx.search(q[:9], 50)
    assert np.array_equal(a[0], b[0][:9]) and np.array_equal(a[1], b[1][:9])


def test_index_file_field_list_of_faiss_write_index(tmp_path):
    """`.index` bytes against the field list of faiss 1.7.4 (impl/index_write.cpp): write_index(IndexFlat) writes the
    fourcc ("IxF2" for METRIC_L2, "IxFI" inner product, "IxFl" otherwise), then write_index_header - d (int32), ntotal
    (int64), two int64 dummies (1 << 20), is_trained (1 byte), metric_type (int32) and, only if metric_type > 1,
    metric_arg (float32) - then WRITE_XBVECTOR(codes): the element count as uint64 in units of 4 bytes
    (= ntotal * d floats) followed by the raw float32 rows.  No faiss-written file exists offline (faiss is not in the
    image, the reference ships no .index), so this pins OUR reading of that list field by field with an independent
    struct parser; read_index must accept exactly this layout for all three metrics."""
    import struct
    from dctdomain_b200 import index as dindex
    db = synth.fingerprints(4, 77)
    for cls, metric, fourcc, has_arg in ((dindex.IndexFlatL2, dindex.METRIC_L2, b'IxF2', False),
                                         (dindex.IndexFlatL1, dindex.METRIC_L1, b'IxFl', True)):
        idx = cls(480)
        idx.add(db)
        path = str(tmp_path / f'm{metric}.index')
        dindex.write_index(idx, path)
        raw = open(path, 'rb').read()
        pos = 0
        assert raw[:4] == fourcc
        pos += 4
        d, ntotal, dummy1, dummy2 = struct.unpack_from('<iqqq', raw, pos)
        pos += 4 + 8 + 8 + 8
        assert (d, ntotal, dummy1, dummy2) == (480, 77, 1 << 20, 1 << 20)
        (is_trained,) = struct.unpack_from('<B', raw, pos)
        pos += 1
        (metric_type,) = struct.unpack_from('<i', raw, pos)
        pos += 4
        assert is_trained == 1 and metric_type == metric
        if has_arg:
            (metric_arg,) = struct.unpack_from('<f', raw, pos)
            pos += 4
            assert metric_arg == 0.0
        (count,) = struct.unpack_from('<Q', raw, pos)
        pos += 8
        assert count == 77 * 480 and len(raw) == pos + count * 4
        rows = np.frombuffer(raw, dtype='<f4', offset=pos).reshape(77, 480)
        assert np.array_equal(rows, db.astype(np.float32))
        back = dindex.read_index(path)
        assert back.metric_type == metric and back.d == 480 and back.ntotal == 77 and np.array_equal(back.reconstruct_n(), db)
