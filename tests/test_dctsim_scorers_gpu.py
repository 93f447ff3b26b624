"""The dct-sim scorers against an exact brute force, at every shape they dispatch.

  * dctd_l1_protein_scores (csrc/l1_protein.cuh, driven from csrc/l1topk.cu): the tiled SAD kernel
    l1_protein_kernel<16, 8, 2, 4, CT> (CT = 30 at d = 480, else 0) reduces each run of a protein's query fingerprints
    within an 8-slot warp slice to a segment minimum and writes last-row distances through the host-built segend / lastm
    masks; l1_protein_reduce_kernel then takes the per-pair minima.  The host loop cuts chunks of query proteins at the
    workspace's row budget, at 65 535 proteins (the reduce kernel's gridDim.y) and at 65 535 query tiles.
  * dctd_l1_pair_scores: pair_scores_kernel<true> (16-byte loads: d % 16 == 0 and an aligned base) and <false>.
  * dct_sim.protein_scores' fallback for fingerprints too wide for the tiles (every pair through _pair_dists), and
    dct_sim.main's all-vs-all and --db output at such widths, down to the listed-pairs scorer when the hits search refuses
    the width as well.

The oracle is exact: |a - b| summed in int64 over d for every fingerprint pair (numpy in row chunks; on the device beyond
1e8 byte-ops, checked against numpy on a slice), then per protein pair the min over the block and its [-1, -1] entry,
INT32_MAX for both when either protein has no fingerprints.  The data are int8 over -128..127 with a block of all -128
rows against a block of all 127 rows (distance 255 d) and query rows copied to two database rows each (min 0, tied).
Every direct call gets a workspace of exactly the size it is given followed by sentinel bytes, and outputs followed by
sentinels; both must be unchanged.  Each case checks the number of kernels it launches (the library's launch counter);
test_zz_kernel_forms reads the kernel names of one call per form from torch.profiler, in a process of its own, and
pytest -s prints kernel form -> cases."""
import re

import numpy as np
import pytest
import torch

from oracle import search_oracle as so

pytestmark = pytest.mark.gpu

BIG = np.iinfo(np.int32).max
GUARD = 4096                       # sentinel bytes after every workspace and output buffer
SENTINEL = 0xA5
NUMPY_OPS = 10 ** 8                # larger brute forces run on the device
NW, TQ, QT = 16, 8, 128            # l1_protein_kernel: compute warps, query slots per warp slice, per CTA tile
TD, STAGES = 2, 4                  # database groups of 32 per stage, stages
D_WIDEST, D_REFUSED = 592, 593     # see test_width_limit_is_the_shared_memory_limit


def protein_kernel(d):
    return f'l1_protein_kernel<{NW},{TQ},{TD},{STAGES},{30 if d == 480 else 0}>'


REDUCE = 'l1_protein_reduce_kernel'


def pair_kernel(vec16):
    return f'pair_scores_kernel<{int(vec16)}>'


REQUIRED = sorted([protein_kernel(480), protein_kernel(100), REDUCE, pair_kernel(True), pair_kernel(False)])


def tile_smem(d):
    """dynamic shared memory of l1_protein_kernel: mbarriers, 128 query rows, 4 stages x 2 groups x 32 vectors, 64"""
    dpad = -(-d // 16) * 16
    return 128 + QT * dpad + STAGES * TD * 32 * dpad + 64


# ---------------------------------------------------------------------------------------------------------------------
# oracle
# ---------------------------------------------------------------------------------------------------------------------
def _np_dists(qf, df):
    out = np.empty((len(qf), len(df)), dtype=np.int64)
    dfi = df.astype(np.int16)
    step = max(1, (1 << 24) // max(1, df.size))
    for i in range(0, len(qf), step):
        out[i:i + step] = np.abs(qf[i:i + step, None, :].astype(np.int16) - dfi[None]).sum(axis=2, dtype=np.int64)
    return out


def fp_dists(qf, df):
    """int64 [len(qf), len(df)]: exact L1 distance of every fingerprint pair"""
    nq, nd = len(qf), len(df)
    if nq == 0 or nd == 0:
        return np.zeros((nq, nd), dtype=np.int64)
    if nq * nd * qf.shape[1] <= NUMPY_OPS:
        return _np_dists(qf, df)
    dt = torch.from_numpy(df).cuda().to(torch.int16)
    step = max(1, (1 << 27) // df.size)
    out = []
    for i in range(0, nq, step):
        qq = torch.from_numpy(qf[i:i + step]).cuda().to(torch.int16)
        out.append((qq[:, None, :] - dt[None]).abs().sum(dim=2, dtype=torch.int64).cpu())
    out = torch.cat(out).numpy()
    rows = np.unique(np.r_[0:min(4, nq), max(0, nq - 4):nq])
    assert np.array_equal(out[rows], _np_dists(qf[rows], df)), 'the device brute force disagrees with numpy'
    return out


def protein_oracle(qf, qoff, df, doff):
    """int64 [n_q, n_db] (min over the pair's block, last-vs-last), INT32_MAX for both where a protein is empty"""
    dist = fp_dists(qf, df)
    nq, nd = len(qoff) - 1, len(doff) - 1
    mn = np.full((nq, nd), BIG, dtype=np.int64)
    last = np.full((nq, nd), BIG, dtype=np.int64)
    qa, db = np.flatnonzero(np.diff(qoff) > 0), np.flatnonzero(np.diff(doff) > 0)
    if len(qa) and len(db):
        # the non-empty proteins' first rows, in order: each reduceat segment is exactly one protein's rows
        blk = np.minimum.reduceat(np.minimum.reduceat(dist, qoff[qa], axis=0), doff[db], axis=1)
        mn[np.ix_(qa, db)] = blk
        last[np.ix_(qa, db)] = dist[np.ix_(qoff[qa + 1] - 1, doff[db + 1] - 1)]
    return mn, last


# ---------------------------------------------------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------------------------------------------------
def offsets_of(counts):
    return np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))]).astype(np.int64)


def layout(rs, total, straddle=(), hi=7, empties=0.08):
    """protein sizes covering `total` fingerprints, 1..hi-1 each plus some empty proteins, with no protein edge within
    two fingerprints of any position in `straddle` (a protein straddles each)"""
    cuts, pos = set(), 0
    while True:
        pos += rs.randint(1, hi)
        if pos >= total:
            break
        cuts.add(pos)
    for p in straddle:
        cuts -= set(range(p - 2, p + 3))
    counts = list(np.diff([0] + sorted(cuts) + [total])) if total else []
    for _ in range(int(len(counts) * empties) + 1):
        counts.insert(rs.randint(len(counts) + 1), 0)
    return counts


def slot_offsets_layout():
    """proteins of 1, 7, 8, 9, 16 and 17 fingerprints starting at every slot offset 0..7 of an 8-slot warp slice"""
    counts, cur = [], 0
    for n in (1, 7, 8, 9, 16, 17):
        for o in range(TQ):
            pad = (o - cur) % TQ
            if pad:
                counts.append(pad)
                cur += pad
            counts.append(n)
            cur += n
    return counts


# slots 5..134 and 438..566 span two query tiles, 136..435 and 640..896 (tile-aligned start) three; partial last tile
SPANS = [5, 130, 1, 300, 2, 0, 129, 73, 257, 7]
# empty proteins at the start, in the middle (alone and in runs) and at the end
EMPTIES = [0, 0, 3, 0, 9, 0, 0, 0, 1, 8, 0, 16, 7, 0, 0]


def query_counts(rs, kind):
    if kind == 'slots':
        return slot_offsets_layout()
    if kind == 'spans':
        return list(SPANS)
    if kind == 'empties':
        return list(EMPTIES)
    if kind == 'mixed':
        c = list(rs.randint(0, 10, size=60))
        c[rs.randint(60)] = 19
        return c
    raise ValueError(kind)


def db_counts(rs, kind):
    """database proteins straddling the 32-vector group edges and the 64-vector (2-group) stage edges; the last group
    holds 1 (161 = 5 x 32 + 1) or 31 (191) fingerprints"""
    if kind == 'ragged1':
        return layout(rs, 161, straddle=(32, 64, 128, 160))
    if kind == 'ragged31':
        return layout(rs, 191, straddle=(32, 64, 96, 128))
    raise ValueError(kind)


def make_sets(seed, d, qcounts, dcounts):
    rs = np.random.RandomState(seed)
    qoff, doff = offsets_of(qcounts), offsets_of(dcounts)
    qf = rs.randint(-128, 128, size=(int(qoff[-1]), d)).astype(np.int8)
    df = rs.randint(-128, 128, size=(int(doff[-1]), d)).astype(np.int8)
    plant(rs, qf, qoff, df, doff)
    return qf, qoff, df, doff


def plant(rs, qf, qoff, df, doff):
    """one query protein of all -128 rows against one database protein of all 127 rows (every distance 255 d), and
    query rows - last rows among them - copied to two database rows each, at group edges where possible (min 0, tied)"""
    qa, db = np.flatnonzero(np.diff(qoff) > 0), np.flatnonzero(np.diff(doff) > 0)
    if not len(qa) or not len(db):
        return
    a, b = qa[0], db[len(db) // 2]
    qf[qoff[a]:qoff[a + 1]] = -128
    df[doff[b]:doff[b + 1]] = 127
    free = np.setdiff1d(np.arange(len(df)), np.arange(doff[b], doff[b + 1]))
    edges = [r for r in (31, 32, 63, 64, len(df) - 1) if r in set(free.tolist())]
    for i, a in enumerate(qa[1:13]):
        src = qoff[a + 1] - 1 if i % 2 else rs.randint(qoff[a], qoff[a + 1])
        dst = list(rs.choice(free, size=min(2, len(free)), replace=False))
        if edges:
            dst[0] = edges.pop(0)
        df[dst] = qf[src]


# ---------------------------------------------------------------------------------------------------------------------
# kernel names from torch.profiler
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL_RE = re.compile(r'\b(l1_protein_kernel|l1_protein_reduce_kernel|pair_scores_kernel|l1_hits_scan_kernel|'
                        r'hits_output_kernel)\b(?:\s*<([^<>]*)>)?')


def canonical(name):
    mt = _KERNEL_RE.search(name)
    if not mt:
        return None
    if mt.group(2) is None:
        return mt.group(1)
    args = [{'true': '1', 'false': '0'}.get(a.strip(), a.strip()) for a in mt.group(2).split(',')]
    return f'{mt.group(1)}<{",".join(args)}>'


def launched(fn):
    """(fn(), the scorer kernels it launched, in order)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return res, [c for c in (canonical(nm) for nm in names) if c]


_observed = {}          # kernel -> case ids


def _record(cid, kernels):
    for kn in kernels:
        _observed.setdefault(kn, []).append(cid)


def _equal(cid, what, got, want):
    bad = np.argwhere(got != want)
    assert not len(bad), f'{cid}: {what}: {len(bad)} of {got.size} entries differ, first {bad[:6].tolist()}, ' \
                         f'got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}'


# ---------------------------------------------------------------------------------------------------------------------
# direct calls with guarded buffers
# ---------------------------------------------------------------------------------------------------------------------
def _lib():
    from dctdomain_b200 import _lib as lib
    return lib


def guarded(n_bytes):
    """uint8 device buffer of n_bytes + GUARD, the tail filled with SENTINEL"""
    buf = torch.full((n_bytes + GUARD,), SENTINEL, dtype=torch.uint8, device='cuda')
    return buf


def guard_intact(buf, n_bytes):
    return bool((buf[n_bytes:] == SENTINEL).all())


def device_rows(rows, misalign=0):
    """int8 [n, d] on the device; misalign > 0: a view whose data pointer is that many bytes past a 16-byte boundary"""
    if not misalign:
        return torch.from_numpy(np.ascontiguousarray(rows)).cuda()
    buf = torch.empty(rows.size + 16, dtype=torch.int8, device='cuda')
    view = buf[misalign:misalign + rows.size].view(rows.shape)
    view.copy_(torch.from_numpy(np.ascontiguousarray(rows)))
    assert view.data_ptr() % 16 == misalign and view.is_contiguous()
    return view


def packed_db(df, d):
    L = _lib().lib()
    packed = torch.empty(max(int(L.dctd_l1_packed_bytes(len(df), d)), 16), dtype=torch.uint8, device='cuda')
    if len(df):
        _lib().check(L.dctd_l1_pack(device_rows(df).data_ptr(), len(df), d, 0, packed.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream), 'dctd_l1_pack')
    torch.cuda.synchronize()
    return packed


def scores_tables(n_qf, nq, nd):
    """bytes of dctd_l1_protein_scores' tables in front of its matrix region"""
    al = lambda b: -(-b // 256) * 256
    return al(((n_qf + 7) // 8 + 64) * 16) + 2 * al((nq + 1) * 4) + al((nd + 1) * 8)


def call_scores(q_dev, qoff, packed, doff, d, ws_bytes=None, profile=False):
    """one dctd_l1_protein_scores call: (rc, min, last, kernels launched, or the launch count without profile),
    workspace and output guards checked"""
    L = _lib().lib()
    nq, nd = len(qoff) - 1, len(doff) - 1
    if ws_bytes is None:
        ws_bytes = int(L.dctd_l1_protein_scores_workspace_bytes(int(qoff[-1]), nq, int(doff[-1]), nd, d))
    ws = guarded(ws_bytes)
    out = [guarded(nq * nd * 4) for _ in range(2)]
    stream = torch.cuda.current_stream().cuda_stream
    def call():
        return L.dctd_l1_protein_scores(q_dev.data_ptr(), qoff.ctypes.data, nq, packed.data_ptr(), doff.ctypes.data,
                                        nd, d, out[0].data_ptr(), out[1].data_ptr(), ws.data_ptr(), ws_bytes, stream)
    if profile:
        rc, kernels = launched(call)
    else:
        torch.cuda.synchronize()
        L.dctd_launch_count(1)
        rc = call()
        kernels = int(L.dctd_launch_count(1))
        torch.cuda.synchronize()
    assert guard_intact(ws, ws_bytes), 'bytes past the workspace were written'
    assert all(guard_intact(o, nq * nd * 4) for o in out), 'bytes past an output matrix were written'
    mn, last = (o[:nq * nd * 4].view(torch.int32).view(nq, nd).cpu().numpy().astype(np.int64) for o in out)
    return rc, mn, last, kernels


# ---------------------------------------------------------------------------------------------------------------------
# dctd_l1_protein_scores
# ---------------------------------------------------------------------------------------------------------------------
def _pcase(cid, d, q, db, ws='exact', misalign=0, seed=0):
    return dict(id=cid, d=d, q=q, db=db, ws=ws, misalign=misalign, seed=seed)


SCORE_CASES = (
    # widths: CT = 30 at d = 480; below one 16-byte chunk (2); 464 / 496 around 480; the widest the tiles accept
    [_pcase(f'width-d{d}', d, 'mixed', 'ragged31', seed=d) for d in (2, 16, 100, 464, 480, 496, 576, D_WIDEST)]
    # query proteins against the 8-slot warp slice and the 128-slot tile, database proteins against group / stage edges
    + [_pcase(f'{q}-{db}-d{d}', d, q, db, seed=d + i)
       for i, (q, db) in enumerate((('slots', 'ragged1'), ('spans', 'ragged31'), ('empties', 'ragged1'),
                                    ('slots', 'ragged31')))
       for d in (480, 100)]
    # database split edges (pick_splits) straddled by proteins, one protein covering a whole split
    + [_pcase(f'splits-d{d}', d, 'mixed', 'splits', seed=7) for d in (480, 16)]
    # degenerate sets
    + [_pcase('all-query-empty', 480, [0, 0, 0], 'ragged1'),
       _pcase('all-db-empty', 480, 'mixed', [0, 0, 0, 0]),
       _pcase('both-empty', 100, [0, 0], [0, 0, 0]),
       _pcase('one-fingerprint-each', 480, [1], [1]),
       _pcase('one-fingerprint-each-d16', 16, [0, 1, 0], [0, 0, 1])]
    # the scalar query load (data pointer not 16-byte aligned, d % 16 == 0)
    + [_pcase(f'misaligned-{m}-d{d}', d, 'slots', 'ragged1', misalign=m, seed=3) for d in (480, 16) for m in (1, 8)]
    # workspace: two rows (each chunk one query protein of 1..8 fingerprints)
    + [_pcase(f'ws-one-protein-d{d}', d, 'small', 'ragged31', ws='one', seed=11) for d in (480, 100)])


def _sets(case):
    rs = np.random.RandomState(case['seed'] + 1000)
    d = case['d']
    q = case['q']
    if isinstance(q, list):
        qc = q
    elif q == 'small':
        qc = list(rs.randint(1, 9, size=40))
        qc[3:3] = [0, 0]
        qc.append(0)
    else:
        qc = query_counts(rs, q)
    db = case['db']
    if isinstance(db, list):
        dc = db
    elif db == 'splits':
        dc = split_db_counts(rs, qc)
    else:
        dc = db_counts(rs, db)
    return make_sets(case['seed'], d, qc, dc)


def pick_splits(sms, n_groups, td, n_qtiles, overhead):
    """restatement of l1topk.cu pick_splits: (splits, groups_per_split)"""
    tiles = max(1, -(-n_groups // td))
    s_max = max(1, min(1024, tiles // 4))
    best_s, best_cost = 1, 1e300
    for sp in range(1, s_max + 1):
        tps = -(-tiles // sp)
        real = -(-tiles // tps)
        waves = -(-(real * n_qtiles) // sms)
        cost = float(waves) * float(tps + overhead)
        if cost < best_cost * 0.995:
            best_cost, best_s = cost, sp
        if sp > 4 * sms and sp * n_qtiles > 16 * sms:
            break
    gps = -(-tiles // best_s) * td
    return max(1, -(-n_groups // gps)), gps


SPLIT_DB = 6417                        # 201 groups, the last with 17 vectors


def split_db_counts(rs, qcounts):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_qtiles = -(-int(sum(qcounts)) // QT)
    splits, gps = pick_splits(sms, -(-SPLIT_DB // 32), TD, n_qtiles, 2)
    edge = gps * 32
    assert splits >= 3, (splits, gps)
    # a protein across every split edge, and one over the whole of split 2
    straddle = [k * edge for k in range(1, splits)] + list(range(2 * edge - 8, 3 * edge + 9, 4))
    c = layout(rs, SPLIT_DB, straddle=straddle)
    ends = np.cumsum(c)
    assert any(e - n < 2 * edge and e > 3 * edge for e, n in zip(ends, c)), 'no protein covers split 2'
    return c


@pytest.mark.parametrize('case', SCORE_CASES, ids=[c['id'] for c in SCORE_CASES])
def test_protein_scores_match_oracle(case):
    cid, d = case['id'], case['d']
    qf, qoff, df, doff = _sets(case)
    ws_bytes = None
    if case['ws'] == 'one':        # the matrix region holds exactly two rows of ld columns
        ws_bytes = scores_tables(len(qf), len(qoff) - 1, len(doff) - 1) + 2 * (-(-len(df) // 32) * 32) * 4
    q_dev, packed = device_rows(qf, case['misalign']), packed_db(df, d)
    rc, mn, last, kernels = call_scores(q_dev, qoff, packed, doff, d, ws_bytes)
    assert rc == 0, (cid, rc)
    want_min, want_last = protein_oracle(qf, qoff, df, doff)
    _equal(cid, 'min', mn, want_min)
    _equal(cid, 'last', last, want_last)
    rc2, mn2, last2, _ = call_scores(q_dev, qoff, packed, doff, d, ws_bytes, profile=False)
    assert rc2 == 0 and mn2.tobytes() == mn.tobytes() and last2.tobytes() == last.tobytes(), \
        f'{cid}: a second call differs'
    has_q, has_db = int(qoff[-1]) > 0, int(doff[-1]) > 0
    # one chunk, or one per non-empty query protein (empty ones join the chunk before them); per chunk the tile kernel
    # (unless a side has no fingerprints) and the reduce kernel
    n_chunks = max(1, int((np.diff(qoff) > 0).sum())) if case['ws'] == 'one' else 1
    assert kernels == n_chunks * (2 if has_q and has_db else 1), (cid, kernels, n_chunks)
    _record(cid, {REDUCE} | ({protein_kernel(d)} if has_q and has_db else set()))
    if has_q and has_db:           # the data reach both extremes
        assert (want_min == 255 * d).any(), cid
        if (np.diff(qoff) > 0).sum() > 1:
            assert want_min.min() == 0, cid


@pytest.mark.parametrize('nq', [65_535, 65_536, 70_000])
def test_query_protein_chunks_at_the_grid_limit(nq):
    """single-fingerprint query proteins at d = 16: the reduce kernel's gridDim.y cuts chunks at 65 535 proteins"""
    cid = f'grid-y-{nq}'
    rs = np.random.RandomState(nq)
    qc = [1] * nq
    dc = layout(rs, 70, straddle=(32, 64))
    qf, qoff, df, doff = make_sets(nq, 16, qc, dc)
    packed = packed_db(df, 16)
    rc, mn, last, kernels = call_scores(device_rows(qf), qoff, packed, doff, 16)
    assert rc == 0, rc
    want_min, want_last = protein_oracle(qf, qoff, df, doff)
    _equal(cid, 'min', mn, want_min)
    _equal(cid, 'last', last, want_last)
    chunks = -(-nq // 65_535)
    assert kernels == 2 * chunks, (kernels, chunks)
    _record(cid, {protein_kernel(16), REDUCE})


def test_workspace_too_small_for_a_protein():
    """a workspace whose matrix region holds two rows, and a query protein that needs three (9 fingerprints: two
    segments and a last row) after two that fit: DCTD_ERR_WORKSPACE, nothing written past the workspace"""
    d = 100
    qf, qoff, df, doff = make_sets(4, d, [3, 5, 9, 2], layout(np.random.RandomState(4), 64))
    ld = -(-len(df) // 32) * 32
    ws_bytes = scores_tables(len(qf), 4, len(doff) - 1) + 2 * ld * 4
    rc, _, _, kernels = call_scores(device_rows(qf), qoff, packed_db(df, d), doff, d, ws_bytes)
    assert rc == _lib().ERR_WORKSPACE, rc
    assert kernels == 4, kernels                          # the two proteins before it were scored
    # two bytes short of the tables: refused before any launch
    q, packed = device_rows(qf), packed_db(df, d)
    rc, _, _, n_launch = call_scores(q, qoff, packed, doff, d, scores_tables(len(qf), 4, len(doff) - 1) + 254,
                                     profile=False)
    assert rc == _lib().ERR_WORKSPACE and n_launch == 0, (rc, n_launch)


@pytest.mark.parametrize('which', ['nq0', 'nd0', 'both0'])
def test_no_proteins_returns_at_once(which):
    """n_qprot = 0 or n_dbprot = 0: DCTD_OK, no launch, the outputs untouched"""
    L = _lib().lib()
    d = 480
    qf, qoff, df, doff = make_sets(1, d, [2, 3], [4, 1])
    if which in ('nq0', 'both0'):
        qoff = qoff[:1]
    if which in ('nd0', 'both0'):
        doff = doff[:1]
    out = [guarded(0) for _ in range(2)]
    ws = guarded(1 << 16)
    q, packed = device_rows(qf), packed_db(df, d)
    torch.cuda.synchronize()
    L.dctd_launch_count(1)
    rc = L.dctd_l1_protein_scores(q.data_ptr(), qoff.ctypes.data, len(qoff) - 1, packed.data_ptr(), doff.ctypes.data,
                                  len(doff) - 1, d, out[0].data_ptr(), out[1].data_ptr(), ws.data_ptr(), 1 << 16,
                                  torch.cuda.current_stream().cuda_stream)
    assert rc == 0 and L.dctd_launch_count(1) == 0, rc
    torch.cuda.synchronize()
    assert all(guard_intact(o, 0) for o in out)


def test_width_limit_is_the_shared_memory_limit():
    """The tile needs 192 + 384 * dpad bytes of shared memory (dpad: d rounded up to 16).  Under a B200's 232 448 B
    opt-in limit that is d <= 592: d = 592 runs (the width cases above), d = 593 returns DCTD_ERR_UNSUPPORTED
    without a launch and without touching the outputs."""
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    assert tile_smem(D_WIDEST) <= optin < tile_smem(D_REFUSED), (optin, tile_smem(D_WIDEST), tile_smem(D_REFUSED))
    L = _lib().lib()
    for d in (D_REFUSED, 608, 800, 1024):
        qf, qoff, df, doff = make_sets(d, d, [2, 0, 3], [1, 4])
        q, packed = device_rows(qf), packed_db(df, d)
        rc, mn, last, n_launch = call_scores(q, qoff, packed, doff, d, profile=False)
        assert rc == _lib().ERR_UNSUPPORTED and n_launch == 0, (d, rc, n_launch)
        assert (mn == 0xA5A5A5A5 - (1 << 32)).all() and (last == 0xA5A5A5A5 - (1 << 32)).all()


# ---------------------------------------------------------------------------------------------------------------------
# dctd_l1_pair_scores
# ---------------------------------------------------------------------------------------------------------------------
PAIR_CASES = [(d, m) for d in (16, 480, 2048) for m in (0, 1)] + [(d, 0) for d in (2, 100, 481, 2047)]


@pytest.mark.parametrize('d,misalign', PAIR_CASES, ids=[f'd{d}' + ('-misaligned' if m else '') for d, m in PAIR_CASES])
def test_pair_scores_match_oracle(d, misalign):
    """every ordered pair of 30 proteins (empty ones included, each with itself), in shuffled order, then 45 repeats:
    945 pairs, a partial last block of 4 warps"""
    cid = f'pairs-d{d}' + ('-misaligned' if misalign else '')
    rs = np.random.RandomState(d + misalign)
    counts = list(rs.randint(1, 6, size=30))
    counts[0] = counts[13] = counts[29] = 0
    counts[7] = 19
    fps, off, _, _ = make_sets(d, d, counts, [])
    # extremes and duplicates within the one set
    fps[off[1]:off[2]] = -128
    fps[off[2]:off[3]] = 127
    fps[off[5 + 1] - 1] = fps[off[7 + 1] - 1]
    fps[off[9]] = fps[off[10]]
    n = len(counts)
    pa, pb = (x.ravel() for x in np.meshgrid(np.arange(n), np.arange(n), indexing='ij'))
    order = rs.permutation(len(pa))
    rep = rs.choice(len(pa), size=45)
    pa = np.concatenate([pa[order], pa[rep]]).astype(np.int32)
    pb = np.concatenate([pb[order], pb[rep]]).astype(np.int32)
    assert len(pa) % 4
    L = _lib().lib()
    f_dev = device_rows(fps, 8 if misalign else 0)
    d_off = torch.from_numpy(off).cuda()
    d_a, d_b = torch.from_numpy(pa).cuda(), torch.from_numpy(pb).cuda()
    out = [guarded(len(pa) * 4) for _ in range(2)]
    L.dctd_launch_count(1)
    rc = L.dctd_l1_pair_scores(f_dev.data_ptr(), d, d_off.data_ptr(), d_a.data_ptr(), d_b.data_ptr(), len(pa),
                               out[0].data_ptr(), out[1].data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert L.dctd_launch_count(1) == 1
    torch.cuda.synchronize()
    assert rc == 0, rc
    assert all(guard_intact(o, len(pa) * 4) for o in out), 'bytes past an output were written'
    mn, last = (o[:len(pa) * 4].view(torch.int32).cpu().numpy().astype(np.int64) for o in out)
    want_min, want_last = protein_oracle(fps, off, fps, off)
    _equal(cid, 'min', mn, want_min[pa, pb])
    _equal(cid, 'last', last, want_last[pa, pb])
    assert (want_min[pa, pb] == 0).any() and (want_min[pa, pb] == 255 * d).any() and (want_last[pa, pb] == BIG).any()
    _record(cid, {pair_kernel(d % 16 == 0 and not misalign)})


# ---------------------------------------------------------------------------------------------------------------------
# dct_sim: the all-pairs fallback and the printed output at refused widths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('d', [D_REFUSED, 800, 1024])
def test_protein_scores_fallback_matches_oracle(d):
    """dct_sim.protein_scores where the tiles refuse the width: every pair through dctd_l1_pair_scores, empty proteins
    (INT32_MAX) included"""
    from dctdomain_b200 import dct_sim
    cid = f'fallback-d{d}'
    rs = np.random.RandomState(d)
    qf, qoff, df, doff = make_sets(d, d, query_counts(rs, 'empties'), db_counts(rs, 'ragged1'))
    L = _lib().lib()
    L.dctd_launch_count(1)
    mn, last = dct_sim.protein_scores(qf, qoff, df, doff)
    assert L.dctd_launch_count(1) == 2                     # dctd_l1_pack, then the refusal and one pair-scores launch
    want_min, want_last = protein_oracle(qf, qoff, df, doff)
    _equal(cid, 'min', mn, want_min)
    _equal(cid, 'last', last, want_last)
    _record(cid, {pair_kernel(d % 16 == 0)})


def _at_distance(row, dist, rs):
    """a copy of int8 `row` at L1 distance exactly `dist`"""
    out = row.astype(np.int32).copy()
    for j in rs.permutation(len(out)):
        if dist == 0:
            break
        up, dn = 127 - out[j], out[j] + 128
        step = min(dist, max(up, dn))
        out[j] += step if up >= dn else -step
        dist -= step
    assert dist == 0
    return out.astype(np.int8)


# (query protein, distance) of database global fingerprints planted against query global fingerprints: similarity 1,
# at the 0.3 cut (11900) and one past it, exactly 0.0 (17000: min(d, 1) keeps the float) and 0 (17001), and ties (two
# database proteins at one distance from one query)
PLANTED = ((0, 0), (0, 0), (0, 11900), (0, 11901), (0, 17000), (0, 17001),
           (1, 500), (1, 8500), (1, 8500), (1, 16999), (2, 4250), (2, 4250))


def _npz_pair(tmp_path, d, seed):
    """query and database npz files in dct-sim's layout (sid / idx / dct); every protein has fingerprints"""
    rs = np.random.RandomState(seed)
    qc, dc = rs.randint(1, 5, size=6), rs.randint(1, 5, size=24)
    qf, qoff, df, doff = make_sets(seed, d, qc, dc)
    slots = rs.permutation(len(dc))
    for (a, dist), b in zip(PLANTED, slots):
        df[doff[b + 1] - 1] = _at_distance(qf[qoff[a + 1] - 1], dist, rs)
    df[doff[slots[-1]]] = qf[qoff[1]]                             # an exact copy of a query fingerprint
    q, db = str(tmp_path / f'q{d}.npz'), str(tmp_path / f'db{d}.npz')
    np.savez(q, sid=np.array([f'q{i}' for i in range(len(qc))]), idx=qoff, dct=qf)
    np.savez(db, sid=np.array([f'd{i}' for i in range(len(dc))]), idx=doff, dct=df)
    return q, db


def _blocks(npz):
    z = np.load(npz)
    # widened: the oracle's int8 subtraction would wrap over -128..127
    return list(z['sid']), [z['dct'][z['idx'][i]:z['idx'][i + 1]].astype(np.int64) for i in range(len(z['sid']))]


def _want_all(npz):
    sid, blk = _blocks(npz)
    out = ['#prot1 prot2 sim-domain sim-global']
    for i in range(len(blk) - 1):
        for j in range(i + 1, len(blk)):
            mx, s = so.domain_sim(blk[i], blk[j])
            out.append(f'{sid[i]} {sid[j]} {mx:.3f} {s:.3f}')
    return out


def _want_db(q, db, top, threshold):
    """dct-sim's database search: per query, every database protein's (max, global) similarity, sorted by the global
    one descending (stable), printed until rank >= top and the similarity is below the threshold"""
    qs, qb = _blocks(q)
    ds, dbk = _blocks(db)
    out = ['#prot1 prot2 sim-domain sim-global']
    for i in range(len(qb)):
        res = sorted([(ds[j],) + so.domain_sim(qb[i], dbk[j]) for j in range(len(dbk))], key=lambda r: r[2],
                     reverse=True)
        for rank, (name, mx, s) in enumerate(res):
            if rank >= top and s < threshold:
                break
            out.append(f'{qs[i]} {name} {mx} {s}')
    return out


@pytest.mark.parametrize('d', [D_REFUSED, 2064])
def test_dct_sim_output_at_refused_widths(tmp_path, d):
    """dct_sim.main at widths the tiles refuse: all-vs-all through the fallback; --db through the hits search at 593
    and, where that refuses too (d > 2048), all the way down to dctd_l1_pair_scores"""
    from dctdomain_b200 import dct_sim
    q, db = _npz_pair(tmp_path, d, d)
    out = str(tmp_path / 'all.txt')
    dct_sim.main(['--dct', db, '--output', out])
    assert open(out).read().splitlines() == _want_all(db)
    _record(f'main-all-d{d}', {pair_kernel(d % 16 == 0)})
    for top, thr in ((5, 0.25), (2, 0.3), (0, 0.3)):
        out = str(tmp_path / f'db{top}.txt')
        args = ['--dct', q, '--db', db, '--output', out, '--top', str(top), '--threshold', str(thr)]
        L = _lib().lib()
        L.dctd_launch_count(1)
        dct_sim.main(args)
        assert open(out).read().splitlines() == _want_db(q, db, top, thr), (d, top, thr)
        if d > 2048:                   # pack, the refusal of the tiles, one pair-scores launch
            assert L.dctd_launch_count(1) == 2
            _record(f'main-db-d{d}-top{top}', {pair_kernel(d % 16 == 0)})


def test_hits_width_limit():
    """dctd_l1_protein_hits takes d <= 2048 (its heap scan keeps one group per stage there, also at 992 hits per
    query) and refuses 2049"""
    from dctdomain_b200 import dct_sim
    rs = np.random.RandomState(3)
    d = 2048
    qf, qoff, df, doff = make_sets(3, d, rs.randint(1, 4, size=8), rs.randint(1, 3, size=1000))
    for a in range(len(qoff) - 1):                         # related database proteins, 0..20000 from the query
        for b in rs.choice(1000, size=6, replace=False):
            df[doff[b + 1] - 1] = _at_distance(qf[qoff[a + 1] - 1], int(rs.randint(0, 20000)), rs)
    mn, last = protein_oracle(qf, qoff, df, doff)
    for top in (5, 992):
        off, hdb, hmin, hlast = dct_sim.protein_hits(qf, qoff, df, doff, top, 1.5)     # no threshold hits: top rows
        for a in range(len(qoff) - 1):
            order = np.argsort(np.minimum(last[a], 17000), kind='stable')[:top]
            assert np.array_equal(hdb[off[a]:off[a + 1]], order)
            assert np.array_equal(hmin[off[a]:off[a + 1]], mn[a, order])
            assert np.array_equal(hlast[off[a]:off[a + 1]], last[a, order])
    qf, qoff, df, doff = make_sets(3, 2049, [1, 2], [2, 1])
    with pytest.raises(_lib().DctdError) as e:
        dct_sim.protein_hits(qf, qoff, df, doff, 5, 0.25)
    assert e.value.code == _lib().ERR_UNSUPPORTED


# ---------------------------------------------------------------------------------------------------------------------
def kernel_forms():
    """One call per kernel form in one torch.profiler session: [(kernels the call must launch, kernels it launched)]"""
    L = _lib().lib()
    stream = torch.cuda.current_stream().cuda_stream
    calls = []
    for d in (480, 100):
        qf, qoff, df, doff = make_sets(d, d, [3, 9, 1], [2, 5, 1])
        q, packed = device_rows(qf), packed_db(df, d)
        calls.append(({protein_kernel(d), REDUCE}, lambda q=q, qoff=qoff, packed=packed, doff=doff, d=d:
                      call_scores(q, qoff, packed, doff, d)[0]))
    for m in (0, 8):
        fps, off, _, _ = make_sets(m, 480, [3, 0, 2], [])
        f_dev, d_off = device_rows(fps, m), torch.from_numpy(off).cuda()
        pa = torch.tensor([0, 1, 2], dtype=torch.int32, device='cuda')
        pb = torch.tensor([2, 0, 2], dtype=torch.int32, device='cuda')
        outs = [torch.empty(3, dtype=torch.int32, device='cuda') for _ in range(2)]
        calls.append(({pair_kernel(not m)}, lambda f=f_dev, o=d_off, pa=pa, pb=pb, outs=outs:
                      L.dctd_l1_pair_scores(f.data_ptr(), 480, o.data_ptr(), pa.data_ptr(), pb.data_ptr(), 3,
                                            outs[0].data_ptr(), outs[1].data_ptr(), stream)))
    out = []
    for want, fn in calls:
        rc, kernels = launched(fn)
        assert rc == 0, rc
        out.append((sorted(want), kernels))
    return out


def test_zz_kernel_forms():
    """The kernel names behind the launch counts above, read with torch.profiler in a process of its own: a profiler
    session opened in the test process before other GPU test files run has made later sessions miss kernel records."""
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.dirname(here), here]))
    code = 'import json, test_dctsim_scorers_gpu as t; print("FORMS" + json.dumps(t.kernel_forms()))'
    res = subprocess.run([sys.executable, '-s', '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    forms = json.loads(next(ln for ln in res.stdout.splitlines() if ln.startswith('FORMS'))[5:])
    seen = set()
    for want, kernels in forms:
        assert set(want) <= set(kernels), (want, kernels)
        seen |= set(want)
    assert seen == set(REQUIRED), sorted(seen)
    # kernel form -> cases (shown with pytest -s)
    for kn in sorted(_observed):
        cids = sorted(set(_observed[kn]))
        print(f'{kn:40s} cases {len(cids):3d}: {", ".join(cids)}')
    assert not _observed or not set(REQUIRED) - set(_observed), sorted(set(REQUIRED) - set(_observed))
