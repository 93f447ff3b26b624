"""dct_sim.protein_hits / dctd_l1_protein_hits against a numpy restatement of dct-sim's database search
(src/dct-sim.py:126-156): full last / min rows, the stable descending sort on the float64 similarity and the loop's
stopping rule.  Integer work: the hit lists must be bit-identical."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
BIG = np.iinfo(np.int32).max
TOPS = (0, 1, 5, 50, 992)
THRESHOLDS = (0.25, 0.3, 1.0, 1.5, 0.0, -1.0, float('nan'))


def _dists(qf, df):
    """int64 [n_qf, n_df] L1 distances with int32 differences, in row chunks"""
    out = np.empty((len(qf), len(df)), dtype=np.int64)
    dfi = df.astype(np.int32)
    for i in range(0, len(qf), 32):
        out[i:i + 32] = np.abs(qf[i:i + 32, None, :].astype(np.int32) - dfi[None]).sum(axis=2)
    return out


def _rows(qf, qoff, df, doff):
    """int64 [n_q, n_db] last-vs-last and min distances, INT32_MAX where a protein has no fingerprints"""
    dist = _dists(qf, df)
    nq, nd = len(qoff) - 1, len(doff) - 1
    last = np.full((nq, nd), BIG, dtype=np.int64)
    mn = np.full((nq, nd), BIG, dtype=np.int64)
    for a in range(nq):
        for b in range(nd):
            blk = dist[qoff[a]:qoff[a + 1], doff[b]:doff[b + 1]]
            if blk.size:
                last[a, b], mn[a, b] = blk[-1, -1], blk.min()
    return last, mn


def _reference(rows, top, threshold):
    """Expected CSR: for each query, dct-sim's loop over the stable descending sort of s(last)."""
    last, mn = rows
    off, hdb, hmin, hlast = [0], [], [], []
    for a in range(len(last)):
        s = 1.0 - np.minimum(last[a] / 17000, 1.0)
        order = np.argsort(-s, kind='stable')
        n = 0
        for rank in range(len(order)):
            if rank >= top and s[order[rank]] < threshold:
                break
            n += 1
        sel = order[:n]
        hdb += sel.tolist(); hmin += mn[a, sel].tolist(); hlast += last[a, sel].tolist()
        off.append(off[-1] + n)
    return [np.array(x, dtype=np.int64) for x in (off, hdb, hmin, hlast)]


def _at_distance(row, dist, rs):
    """a copy of int8 `row` at L1 distance exactly `dist` (each byte moved towards the end with more room)"""
    out = row.astype(np.int32).copy()
    for j in rs.permutation(len(out)):
        if dist == 0:
            break
        room_up, room_dn = 127 - out[j], out[j] + 128
        step = min(dist, max(room_up, room_dn))
        out[j] += step if room_up >= room_dn else -step
        dist -= step
    assert dist == 0
    return out.astype(np.int8)


def _dataset(d, nq, nd, seed):
    """Proteins with 0, 1 and more than 8 fingerprints on both sides (an empty query protein among them), values
    0..127 (unrelated global fingerprints ~20 000 apart at d = 480: the 17000 tier), near and exact copies of query
    global fingerprints, duplicates straddling 32-vector group boundaries, distances at dist_cut and dist_cut + 1."""
    from dctdomain_b200.dct_sim import _dist_cut
    rs = np.random.RandomState(seed)

    def counts(n, hi):
        c = rs.randint(1, hi, size=n)
        c[rs.choice(n, size=max(1, n // 10), replace=False)] = 0
        c[1] = 1
        c[2] = 11
        return c
    qc, dc = counts(nq, 7), counts(nd, 8)
    qc[0] = 0                                              # an empty query protein
    qoff = np.concatenate([[0], np.cumsum(qc)]).astype(np.int64)
    doff = np.concatenate([[0], np.cumsum(dc)]).astype(np.int64)
    qf = rs.randint(0, 128, size=(int(qoff[-1]), d)).astype(np.int8)
    df = rs.randint(0, 128, size=(int(doff[-1]), d)).astype(np.int8)
    glob = lambda off, b: int(off[b + 1]) - 1             # row of protein b's global fingerprint
    full = [a for a in range(nq) if qc[a] > 0]
    dbs = [b for b in range(nd) if dc[b] > 0]
    cuts = sorted({c for c in (_dist_cut(0.25), _dist_cut(0.3), 0) if c <= d * 127})
    for i, b in enumerate(rs.choice(dbs, size=min(len(dbs), 40), replace=False)):
        a = full[i % len(full)]
        c = cuts[i % len(cuts)] + (i // len(cuts)) % 2    # exactly at a cut, or one past it
        if c <= d * 127:
            df[glob(doff, b)] = _at_distance(qf[glob(qoff, a)], c, rs)
    a = full[-1]
    for b in (31, 32, 63, 64):                             # equal global fingerprints on both sides of group edges
        if b < nd and dc[b] > 0:
            df[glob(doff, b)] = qf[glob(qoff, a)]
    return qf, qoff, df, doff


def _check(got, want):
    for g, w, name in zip(got, want, ('hit_off', 'hit_db', 'hit_min', 'hit_last')):
        assert g.dtype == np.int64 and np.array_equal(g, w), (name, g[:20], w[:20])


@pytest.mark.parametrize('d', [480, 100, 16, 840])       # 840: the heap scan's shared memory at the opt-in limit
def test_hits_match_dct_sim_rule(d):
    from dctdomain_b200 import dct_sim
    qf, qoff, df, doff = _dataset(d, 45, 201, d)           # 201: the database is not a multiple of 32
    rows = _rows(qf, qoff, df, doff)
    for top in TOPS:
        for thr in THRESHOLDS:
            want = _reference(rows, top, thr)
            _check(dct_sim.protein_hits(qf, qoff, df, doff, top, thr), want)


def test_small_database_and_full_rows():
    """n_db < top, every query's row is the whole database in order (threshold 0), cap = 1 (every query rerun)"""
    from dctdomain_b200 import dct_sim
    qf, qoff, df, doff = _dataset(480, 20, 7, 5)
    rows = _rows(qf, qoff, df, doff)
    for top, thr in ((50, 0.25), (5, 0.0), (992, float('nan')), (1, 0.3)):
        want = _reference(rows, top, thr)
        _check(dct_sim.protein_hits(qf, qoff, df, doff, top, thr), want)
        _check(dct_sim.protein_hits(qf, qoff, df, doff, top, thr, cap=1), want)


def test_top_at_the_limit_on_a_large_database():
    """top = 992 over 1500 database proteins: the heap scan at its largest k, rows of 992 hits"""
    from dctdomain_b200 import dct_sim
    qf, qoff, df, doff = _dataset(480, 12, 1500, 7)
    rows = _rows(qf, qoff, df, doff)
    for top, thr in ((992, 0.25), (991, 1.5), (3, 0.3)):
        _check(dct_sim.protein_hits(qf, qoff, df, doff, top, thr), _reference(rows, top, thr))
    with pytest.raises(Exception) as e:                    # more hits than one row holds: the all-pairs route
        dct_sim.protein_hits(qf, qoff, df, doff, 5, 0.0)
    assert getattr(e.value, 'code', None) == -4


def _raw(qf, qoff, df, doff, top, cut, cap, ws_bytes=None):
    """one dctd_l1_protein_hits call: (count, hit_db, hit_min, hit_last rows, launches)"""
    from dctdomain_b200 import _lib
    L = _lib.lib()
    dq, dd = torch.from_numpy(qf).cuda(), torch.from_numpy(df).cuda()
    nq, nd, d = len(qoff) - 1, len(doff) - 1, qf.shape[1]
    need = ws_bytes or L.dctd_l1_protein_hits_workspace_bytes(len(qf), nq, len(df), nd, d, top, cap)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    count = torch.empty(nq, dtype=torch.int32, device='cuda')
    rows = torch.empty((3, nq, cap), dtype=torch.int32, device='cuda')
    L.dctd_launch_count(1)
    rc = L.dctd_l1_protein_hits(dq.data_ptr(), qoff.ctypes.data, nq, dd.data_ptr(), doff.ctypes.data, nd, d, top, 17000,
                                cut, cap, count.data_ptr(), rows[0].data_ptr(), rows[1].data_ptr(), rows[2].data_ptr(),
                                ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    launches = L.dctd_launch_count(1)
    _lib.check(rc, 'dctd_l1_protein_hits')
    torch.cuda.synchronize()
    return count.cpu().numpy(), rows.cpu().numpy(), launches


def test_counts_exact_rows_truncated_chunks_and_repeatable():
    from dctdomain_b200 import dct_sim
    from dctdomain_b200 import _lib
    qf, qoff, df, doff = _dataset(480, 300, 150, 11)
    rows = _rows(qf, qoff, df, doff)
    want = _reference(rows, 5, 0.0)         # every database protein is a hit
    cnt, got, _ = _raw(qf, qoff, df, doff, 5, dct_sim._dist_cut(0.0), 4)
    assert (cnt == 150).all()
    for a in range(300):                                   # rows hold the first cap hits
        w = slice(want[0][a], want[0][a] + 4)
        assert np.array_equal(got[0, a], want[1][w]) and np.array_equal(got[1, a], want[2][w])
        assert np.array_equal(got[2, a], want[3][w])
    want = _reference(rows, 5, 0.25)
    full = _raw(qf, qoff, df, doff, 5, dct_sim._dist_cut(0.25), 32)
    again = _raw(qf, qoff, df, doff, 5, dct_sim._dist_cut(0.25), 32)
    assert np.array_equal(full[0], again[0]) and full[1].tobytes() == again[1].tobytes()     # same bytes twice
    assert np.array_equal(full[0], np.diff(want[0]))
    L = _lib.lib()
    one = L.dctd_l1_protein_hits_workspace_bytes(len(qf), 300, len(df), 150, 480, 5, 32)
    small = (one + L.dctd_l1_protein_hits_workspace_bytes(len(qf), 1, len(df), 150, 480, 5, 32)) // 2
    chunked = _raw(qf, qoff, df, doff, 5, dct_sim._dist_cut(0.25), 32, ws_bytes=small)
    assert chunked[2] > full[2] + 3                        # several query chunks: more launches
    assert np.array_equal(chunked[0], full[0]) and chunked[1].tobytes() == full[1].tobytes()
    _check(dct_sim.protein_hits(qf, qoff, df, doff, 5, 0.25, workspace_bytes=small), want)


def test_goldens_come_from_the_hits_path(tmp_path, monkeypatch):
    from dctdomain_b200 import dct_sim

    def banned(*a, **k):
        raise AssertionError('db_search scored all pairs')
    monkeypatch.setattr(dct_sim, 'protein_scores', banned)
    npz = os.path.join(G, 'example-dct.npz')
    out = str(tmp_path / 'db.txt')
    dct_sim.main(['--dct', npz, '--db', npz, '--top', '3', '--threshold', '0.3', '--output', out])
    assert open(out).read() == open(os.path.join(G, 'example-dbsearch.txt')).read()
    out = str(tmp_path / 'db2.txt')
    dct_sim.main(['--dct', os.path.join(G, 'G6PD-dct.npz'), '--db', npz, '--output', out])
    assert open(out).read() == open(os.path.join(G, 'example-dbsearch-g6pd.txt')).read()


def test_db_search_falls_back_where_rows_would_be_too_long(tmp_path, monkeypatch):
    """threshold 0 on more than 992 database proteins: every protein is a hit, so db_search scores all pairs"""
    from dctdomain_b200 import dct_sim
    qf, qoff, df, doff = _dataset(480, 3, 1100, 3)
    want = _reference(_rows(qf, qoff, df, doff), 5, 0.0)
    q = str(tmp_path / 'q.npz')
    db = str(tmp_path / 'db.npz')
    np.savez(q, sid=np.array([f'q{i}' for i in range(3)]), idx=qoff, dct=qf)
    np.savez(db, sid=np.array([f'd{i}' for i in range(1100)]), idx=doff, dct=df)
    out = str(tmp_path / 'out.txt')
    dct_sim.main(['--dct', q, '--db', db, '--top', '5', '--threshold', '0', '--output', out])
    lines = open(out).read().splitlines()[1:]
    assert len(lines) == 3 * 1100
    exp = []
    for a in range(3):
        for j in range(want[0][a], want[0][a + 1]):
            mx, s = dct_sim._maxs_s(want[2][j], want[3][j])
            exp.append(f'q{a} d{want[1][j]} {mx} {s}')
    assert lines == exp


def test_scale_beyond_the_all_pairs_matrices():
    """4096 query proteins x 1M database proteins (~4.5 fingerprints each): the two int32 matrices of the all-pairs
    route alone would take 33 GB.  The search completes within the inputs, workspace and outputs, and 64 sampled
    queries equal a torch brute force over their rows."""
    from dctdomain_b200 import dct_sim, _lib
    nq, nd, d = 4096, 1_000_000, 480
    g = torch.Generator(device='cuda').manual_seed(5)
    rs = np.random.RandomState(5)
    qc, dc = rs.randint(1, 9, size=nq), rs.randint(1, 9, size=nd)
    dc[::997] = 0                                          # some database proteins without fingerprints
    qoff = np.concatenate([[0], np.cumsum(qc)]).astype(np.int64)
    doff = np.concatenate([[0], np.cumsum(dc)]).astype(np.int64)
    qf = torch.randint(0, 128, (int(qoff[-1]), d), generator=g, device='cuda', dtype=torch.int8)
    df = torch.randint(0, 128, (int(doff[-1]), d), generator=g, device='cuda', dtype=torch.int8)
    sample = np.sort(rs.choice(nq, size=64, replace=False))
    # related database proteins for the sampled queries: their global fingerprint with a few bytes changed
    for i, a in enumerate(sample):
        for b in rs.choice(np.nonzero(dc)[0], size=3 + i % 4, replace=False):
            row = qf[int(qoff[a + 1]) - 1].clone()
            cols = torch.from_numpy(rs.choice(d, size=int(rs.randint(0, 200)), replace=False)).cuda()
            row[cols] = torch.randint(0, 128, (len(cols),), generator=g, device='cuda', dtype=torch.int8)
            df[int(doff[b + 1]) - 1] = row
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    off, hdb, hmin, hlast = dct_sim.protein_hits(qf, qoff, df, doff, 5, 0.25)
    grew = torch.cuda.max_memory_allocated() - base
    ws = _lib.lib().dctd_l1_protein_hits_workspace_bytes(len(qf), nq, len(df), nd, d, 5, 32)
    outputs = 4 * nq * 32 * 4
    assert grew <= ws + outputs + (64 << 20), (grew, ws)
    assert grew < (2 << 30)
    # brute force over the sampled queries' rows
    qlast = qf[torch.from_numpy(qoff[sample + 1] - 1).cuda()].float()
    has = torch.from_numpy(dc > 0).cuda()
    dlast = df[torch.from_numpy(np.maximum(doff[1:] - 1, 0)).cuda()]
    last = torch.empty((64, nd), dtype=torch.int64, device='cuda')
    for c0 in range(0, nd, 1 << 17):
        last[:, c0:c0 + (1 << 17)] = torch.cdist(qlast, dlast[c0:c0 + (1 << 17)].float(), p=1).round().long()
    last[:, ~has] = BIG
    last = last.cpu().numpy()
    qf_h, df_h = None, None
    for i, a in enumerate(sample):
        s = 1.0 - np.minimum(last[i] / 17000, 1.0)
        order = np.argsort(-s, kind='stable')
        n = max(5, int((s >= 0.25).sum()))
        sel = order[:n]
        assert np.array_equal(hdb[off[a]:off[a + 1]], sel), (a, hdb[off[a]:off[a + 1]][:10], sel[:10])
        assert np.array_equal(hlast[off[a]:off[a + 1]], last[i, sel])
        qa = qf[int(qoff[a]):int(qoff[a + 1])].cpu().numpy()
        for j, b in enumerate(sel):
            blk = df[int(doff[b]):int(doff[b + 1])].cpu().numpy()
            want_min = _dists(qa, blk).min() if len(blk) else BIG
            assert hmin[off[a] + j] == want_min
    assert (np.diff(off) >= 5).all()
