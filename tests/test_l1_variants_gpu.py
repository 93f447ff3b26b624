"""Every kernel that run_topk can launch in a release build, each against the exact L1 top-k oracle.

run_topk (csrc/l1topk.cu, csrc/l1_stream.cuh) picks its kernels from the query count nq, the database size n, the width
d and k: the heap scan l1_scan_kernel<TQ, TD, STAGES> alone (small databases, large k, or no room for the threshold
scan), or the threshold path - the fused streaming kernel (nq <= 16), the non-fused streaming chain (nq <= 16 and d <= 32,
where the ring cannot hold the selection buffer) or the sampled threshold scan (nq > 16) - followed by the heap redo of
queries whose candidate list overflowed.  Each case below names the kernels it must launch and checks:

  * that exactly these kernels ran (torch.profiler kernel names);
  * (dist, ids) of IndexFlatL1.search_device, bit for bit, against oracle/search_oracle.l1_topk (the C restatement of
    faiss), or for more than 64 queries against an exact brute force on the device that is itself checked against the
    C oracle on a seeded subset including the partial last query tile;
  * the packed keys of search_keys_device with id_base > 0 (dist << 40 | id_base + position, -1 = empty slot);
  * that a second call gives the same bytes.

The data: int8 values over -128..127, queries that are database rows and rows perturbed by +-2, exact duplicates of a
query's nearest row on both sides of a 32-vector group boundary and in the ragged last group, and clusters of 40 rows at
one distance each (3, 6, 9, ..), so that the k-th distance is tied and position order decides.  n = 65 553 = 2^16 + 17:
large enough for the threshold path, with a last group of 17 vectors.

Forced paths, one case per path family: a candidate list that overflows (more than kCmax = 8192 vectors within the k-th
distance), the fused kernel's fallback from select_query_fast to select_query (more than 1024 keys tie at the k-th
distance), and an external distance bound through dctd_l1_topk_keys.  The last test requires the kernels observed to
equal the release table, so that a dispatcher change which orphans a kernel fails there."""
import functools
import os
import re

import numpy as np
import pytest
import torch

from oracle import search_oracle as so

pytestmark = pytest.mark.gpu

N = 65_553                  # 2^16 + 17: threshold-eligible (n >= 65 536), ragged last group
CMAX = 8192                 # kCmax: candidate slots per query on the threshold path
FAST_SORT_CAP = 1024        # kFastSortCap: ties select_query_fast sorts itself
ID_BASE = (1 << 33) + 5
CLUSTER, CLUSTER_STEP, N_CLUSTERS = 40, 3, 26      # tie clusters: 40 rows each at distance 3, 6, .., 78
BF_CHECK = 24               # seeded queries (plus the last 9) on which the brute force is checked against the C oracle
THREADS = len(os.sched_getaffinity(0))


def scan(tq, td, st):
    return f'l1_scan_kernel<{tq},{td},{st}>'


def thresh(nw, tq, ct=0):
    return f'l1_thresh_scan_kernel<{nw},{tq},2,4,{ct}>'


def fused(tq, nw, ct=0):
    return f'l1_stream_fused_kernel<{tq},{nw},1,{ct},0>'


def tstream(tq):
    return f'l1_thresh_stream_kernel<{tq},{int(tq <= 4)}>'


def smin(tq):
    return f'l1_sample_min_kernel<{tq}>'


KTH, SEED, SELECT, MERGE = 'l1_kth_kernel', 'l1_seed_kernel', 'l1_select_kernel', 'l1_merge_kernel<0>'


# The kernels run_topk launches in a release build, as (dist, ids) or keys.  Left out:
#   * the DCTD_TUNING build's forms (dctd_l1_set_mode 2, 3, 5 and 6..27: heap-scan thresholds in the streaming regime,
#     rescanned samples, rolled chunk loops, the fused kernel with TD = 2 and 5 / 6 consumer warps, VAR 1 / 2);
#   * fused kernels compiled into the release library that no shape reaches: the fused kernel runs only when the heap scan
#     keeps two groups per stage (d <= 848), and up to that width stream_cfg always finds room for 4 consumer warps, so NW
#     = 2 / 1 never run; d = 480 always has 7, so NW = 4 with CT = 30 never runs; and with 4 or 8 queries per pass the
#     ring holds 7 warps' slots up to d = 848;
#   * l1_merge_kernel<1> (dctd_l1_topk_merge, the sharded search) and the dct-sim kernels (l1_protein*, l1_hits*).
REQUIRED = sorted(
    [scan(tq, 2, 4) for tq in (1, 2, 4, 8)] + [scan(tq, 1, 2) for tq in (1, 2, 4, 8)]
    + [thresh(8, 4), thresh(8, 8), thresh(16, 8), thresh(16, 8, 30)]
    + [fused(tq, 7, ct) for tq in (4, 8, 12, 16) for ct in (0, 30)] + [fused(12, 4), fused(16, 4)]
    + [smin(tq) for tq in (4, 8, 16)] + [tstream(tq) for tq in (4, 8, 16)]
    + [KTH, SEED, SELECT, MERGE])


def heap_only(tq, td=2, st=4):
    return {scan(tq, td, st), MERGE}


def fused_path(tq, nw, ct, redo_tq):
    return {fused(tq, nw, ct), scan(redo_tq, 2, 4), MERGE}


def stream_path(tq, redo_tq):
    return {smin(tq), KTH, tstream(tq), SELECT, scan(redo_tq, 2, 4), MERGE}


def thresh_path(nw, tq, ct, heap_tq):
    """sample heap scan + merge + seeds, threshold scan, selection, heap redo of overflowed queries + merge"""
    return {scan(heap_tq, 2, 4), MERGE, SEED, thresh(nw, tq, ct), SELECT}


def _case(d, nq, k, kernels, n=N, data='std', note=''):
    return dict(d=d, nq=nq, k=k, n=n, data=data, kernels=frozenset(kernels), note=note)


CASES = [
    # d = 480, the reference's fingerprints (CT = 30): fused kernel for 1..16 queries, TQ = 4 / 8 / 12 / 16
    _case(480, 1, 50, fused_path(4, 7, 30, 1)),
    _case(480, 4, 50, fused_path(4, 7, 30, 1)),
    _case(480, 5, 50, fused_path(8, 7, 30, 1)),
    _case(480, 8, 50, fused_path(8, 7, 30, 1)),
    _case(480, 9, 50, fused_path(12, 7, 30, 2)),
    _case(480, 12, 50, fused_path(12, 7, 30, 2)),
    _case(480, 13, 50, fused_path(16, 7, 30, 2)),
    _case(480, 16, 50, fused_path(16, 7, 30, 2)),
    # sampled threshold scan: 8 x 4, 8 x 8 and (nq >= 1024) 16 x 8 queries per CTA
    _case(480, 17, 50, thresh_path(8, 4, 0, 4)),
    _case(480, 32, 50, thresh_path(8, 4, 0, 4)),
    _case(480, 33, 50, thresh_path(8, 8, 0, 8)),
    _case(480, 1023, 50, thresh_path(8, 8, 0, 8)),
    _case(480, 1024, 50, thresh_path(16, 8, 30, 8), note='bench.py search'),
    _case(480, 1061, 50, thresh_path(16, 8, 30, 8)),
    # k: gstride = 8192 / 4 / k >= 8 keeps the threshold path up to k = 256
    _case(480, 17, 225, thresh_path(8, 4, 0, 2)),
    _case(480, 33, 225, thresh_path(8, 8, 0, 2)),
    _case(480, 17, 256, thresh_path(8, 4, 0, 2)),
    _case(480, 33, 256, thresh_path(8, 8, 0, 2)),
    _case(480, 17, 257, heap_only(2)),
    _case(480, 33, 257, heap_only(2)),
    # n: the threshold path starts at 65 536 vectors
    _case(480, 5, 50, heap_only(1), n=65_535),
    _case(480, 40, 50, heap_only(8), n=65_535),
    _case(480, 5, 50, fused_path(8, 7, 30, 1), n=65_536),
    _case(480, 3, 50, heap_only(1), n=33, note='fewer vectors than k: (FLT_MAX, -1) padding'),
    # d <= 32: the ring cannot hold the selection buffer; the non-fused streaming chain
    _case(16, 3, 50, stream_path(4, 1)),
    _case(16, 8, 50, stream_path(8, 1)),
    _case(16, 16, 50, stream_path(16, 2)),
    _case(32, 4, 50, stream_path(4, 1)),
    _case(32, 5, 50, stream_path(8, 1)),
    _case(32, 9, 50, stream_path(16, 2)),
    # fused kernel with a runtime chunk count (CT = 0); 33 is the first width above the non-fused chain
    _case(33, 9, 50, fused_path(12, 7, 0, 2)),
    _case(100, 12, 50, fused_path(12, 7, 0, 2)),
    _case(100, 16, 50, fused_path(16, 7, 0, 2)),
    _case(100, 40, 50, thresh_path(8, 8, 0, 8)),
    _case(100, 1061, 50, thresh_path(16, 8, 0, 8)),
    # ring slot counts that are not a multiple of the consumer warps (wait_issued): 13 / 13 / 10 / 8 slots
    _case(481, 12, 50, fused_path(12, 7, 0, 2)),
    _case(497, 2, 50, fused_path(4, 7, 0, 1)),
    _case(640, 8, 50, fused_path(8, 7, 0, 1)),
    _case(840, 6, 50, fused_path(8, 7, 0, 1)),
    _case(496, 2, 50, fused_path(4, 7, 0, 1), note='14 slots: the widest d without wait_issued for TQ = 4'),
    # 4 consumer warps: 8 slots (d = 832) and 7 slots (wait_issued)
    _case(832, 16, 50, fused_path(16, 4, 0, 1)),
    _case(840, 13, 50, fused_path(16, 4, 0, 1)),
    _case(844, 12, 50, fused_path(12, 4, 0, 1)),
    _case(848, 16, 50, fused_path(16, 4, 0, 1)),
    # heap scan alone: the threshold scan's shared memory does not fit (d = 640, 1061 queries), one group per stage
    # (TD = 1, d >= 849).  d = 833..848 (848 padded bytes) leaves the heap scan 96 B of the 232 448 B opt-in shared
    # memory: it runs only if the kernel has no static shared memory
    _case(640, 1061, 50, heap_only(4)),
    _case(848, 40, 50, heap_only(1)),
    _case(849, 40, 50, heap_only(8, 1, 2)),
    _case(1024, 300, 97, heap_only(4, 1, 2)),
    _case(1297, 40, 50, heap_only(4, 1, 2)),
    _case(2048, 40, 225, heap_only(2, 1, 2)),
    _case(2048, 5, 992, heap_only(1, 1, 2)),
]

# forced paths: one configuration per path family
FAMILIES = {
    'fused': (480, 5, 50, fused_path(8, 7, 30, 1)),
    'stream': (16, 3, 50, stream_path(4, 1)),
    'thresh': (480, 40, 50, thresh_path(8, 8, 0, 8)),
    'heap_td1': (1024, 20, 50, heap_only(4, 1, 2)),
}
for _fam, (_d, _nq, _k, _kern) in FAMILIES.items():
    CASES.append(_case(_d, _nq, _k, _kern, data='overflow', note=_fam))
    if _fam != 'heap_td1':
        CASES.append(_case(_d, _nq, _k, _kern, data='ties', note=_fam))


def _case_id(c):
    s = f'd{c["d"]}-nq{c["nq"]}-k{c["k"]}'
    if c['n'] != N:
        s += f'-n{c["n"]}'
    if c['data'] != 'std':
        s += f'-{c["data"]}-{c["note"]}'
    return s


# ---------------------------------------------------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------------------------------------------------
def _near(v, cols, t):
    """v with column cols[i] moved by t (up if that stays <= 127, else down): L1 distance t from v."""
    out = np.repeat(v[None, :].astype(np.int16), len(cols), axis=0)
    r = np.arange(len(cols))
    up = out[r, cols] + t <= 127
    out[r, cols] += np.where(up, t, -t)
    return out.astype(np.int8)


@functools.lru_cache(maxsize=2)
def database(d, n, data='std'):
    """(db int8 [n, d], queries int8 [max_nq, d]); queries[:nq] are the queries of any case on this database.

    Query 0 is a database row, duplicated at 62..65 (around the boundary of groups 1 and 2) and in the last group;
    query 1 a row perturbed by +-2 whose source row, its nearest, is duplicated the same way; queries 0 and 2 have the
    tie clusters.  Further queries alternate between rows and perturbed rows.  data = 'overflow': 20 000 rows at distance 5 from query 0;
    'ties': about 3000 rows at distance 6 from query 0, at least one in every group."""
    rs = np.random.RandomState(d * 7919 + n % 7907 + {'std': 0, 'overflow': 1, 'ties': 2}[data])
    db = rs.randint(-128, 128, size=(n, d), dtype=np.int8)
    max_nq = max(c['nq'] for c in CASES + BOUND_CASES if c['d'] == d and c['n'] == n and c['data'] == data)
    if n < 4096:
        src = rs.permutation(n)[:max_nq]
        q = db[src].copy()
        q[1::2] = np.clip(q[1::2].astype(np.int16) + rs.randint(-2, 3, size=q[1::2].shape), -128, 127).astype(np.int8)
        return db, q
    used = np.zeros(n, dtype=bool)
    last = (n - 1) // 32 * 32                           # first vector of the last group
    dup_at = [[62, 63, 64, 65, last - 1, last, n - 1], [126, 127, 128, last - 2, last + 1, n - 2]]
    for p in dup_at:
        used[p] = True
    if data == 'overflow':
        used[10_000:30_000] = True
    free = np.flatnonzero(~used)
    picks = rs.permutation(free)
    src, picks = picks[:max_nq], picks[max_nq:]
    used[src] = True
    q = db[src].copy()
    q[1::2] = np.clip(q[1::2].astype(np.int16) + rs.randint(-2, 3, size=q[1::2].shape), -128, 127).astype(np.int8)
    for i in range(min(2, max_nq)):
        db[dup_at[i]] = db[src[i]]
    for i in range(0, min(3, max_nq), 2):
        for c in range(N_CLUSTERS):
            rows, picks = picks[:CLUSTER], picks[CLUSTER:]
            used[rows] = True
            db[rows] = _near(q[i], rs.randint(0, d, size=CLUSTER), CLUSTER_STEP * (c + 1))
    if data == 'overflow':
        db[10_000:30_000] = _near(q[0], rs.randint(0, d, size=20_000), 5)
    elif data == 'ties':
        lanes = []
        for g in range(0, n, 32):                       # one free vector of every group, then more up to 3000
            cand = np.flatnonzero(~used[g:g + 32])
            lanes.append(g + cand[rs.randint(len(cand))])
        extra = np.setdiff1d(np.flatnonzero(~used), lanes)
        rows = np.concatenate([lanes, rs.choice(extra, 3000 - len(lanes), replace=False)])
        db[rows] = _near(q[0], rs.randint(0, d, size=len(rows)), 6)
    return db, q


@functools.lru_cache(maxsize=2)
def index(d, n, data):
    from dctdomain_b200 import index as dindex
    idx = dindex.IndexFlatL1(d)
    idx.add(database(d, n, data)[0])
    return idx


def _pool(d, n, data):
    """Queries and k of the C-oracle run shared by every case of one database with at most 64 queries."""
    cs = [c for c in CASES + BOUND_CASES if (c['d'], c['n'], c['data']) == (d, n, data) and c['nq'] <= 64]
    return max(c['nq'] for c in cs), max(c['k'] for c in cs)


@functools.lru_cache(maxsize=2)
def _oracle_pool(d, n, data):
    db, q = database(d, n, data)
    nq, k = _pool(d, n, data)
    return so.l1_topk(q[:nq], db, k, threads=THREADS)


def brute_force(db, q, k):
    """Exact top-k on the device: int16 |a - b| summed in int32, k smallest of dist << 32 | position."""
    dbt = torch.from_numpy(db).cuda().to(torch.int16)
    n, d = db.shape
    pos = torch.arange(n, device='cuda', dtype=torch.int64)
    chunk = max(1, (1 << 27) // (n * d))
    out = []
    for b in range(0, len(q), chunk):
        qq = torch.from_numpy(q[b:b + chunk]).cuda().to(torch.int16)
        dist = (dbt[None, :, :] - qq[:, None, :]).abs().sum(dim=2, dtype=torch.int32)
        key = (dist.to(torch.int64) << 32) | pos[None, :]
        out.append(torch.topk(key, min(k, n), dim=1, largest=False, sorted=True).values)
    key = torch.cat(out).cpu().numpy()
    dm = np.full((len(q), k), so.FLT_MAX, dtype=np.float32)
    im = np.full((len(q), k), -1, dtype=np.int64)
    dm[:, :key.shape[1]] = (key >> 32).astype(np.float32)
    im[:, :key.shape[1]] = key & 0xffffffff
    return dm, im


def reference(d, n, data, nq, k):
    """(dist float32 [nq, k], ids int64 [nq, k]) of faiss' flat L1 search."""
    db, q = database(d, n, data)
    if nq <= 64:
        dm, im = _oracle_pool(d, n, data)
        return dm[:nq, :k], im[:nq, :k]
    dm, im = brute_force(db, q[:nq], k)
    rs = np.random.RandomState(nq)
    rows = np.unique(np.concatenate([rs.choice(nq, BF_CHECK, replace=False), np.arange(nq - 9, nq)]))
    dm2, im2 = so.l1_topk(q[rows], db, k, threads=THREADS)
    assert np.array_equal(im[rows], im2) and np.array_equal(dm[rows], dm2), 'the brute force disagrees with the C oracle'
    return dm, im


def as_keys(dm, im, id_base):
    """faiss' (dist, ids) -> packed keys dist << 40 | id_base + position, -1 for an empty slot."""
    keys = (np.where(im < 0, 0, dm).astype(np.int64) << 40) | (im + id_base)
    return np.where(im < 0, -1, keys)


# ---------------------------------------------------------------------------------------------------------------------
# kernel names from torch.profiler
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL_RE = re.compile(r'\b(l1_scan_kernel|l1_thresh_scan_kernel|l1_stream_fused_kernel|l1_thresh_stream_kernel|'
                        r'l1_sample_min_kernel|l1_kth_kernel|l1_select_kernel|l1_seed_kernel|l1_merge_kernel)\b'
                        r'(?:\s*<([^<>]*)>)?')


def canonical(name):
    """'void (anonymous namespace)::l1_thresh_stream_kernel<4, true>(...)' -> 'l1_thresh_stream_kernel<4,1>'."""
    mt = _KERNEL_RE.search(name)
    if not mt:
        return None
    if mt.group(2) is None:
        return mt.group(1)
    args = [a.strip() for a in mt.group(2).split(',')]
    args = [{'true': '1', 'false': '0'}.get(a, a) for a in args]
    return f'{mt.group(1)}<{",".join(args)}>'


def launched(fn):
    """Runs fn() in a profiler session of its own; returns (its result, the search kernels launched, in order)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return res, [c for c in (canonical(nm) for nm in names) if c]


_observed = {}          # kernel -> case ids
_forced = {}            # (forced path, family) -> case ids


def _record(cid, kernels, want):
    for kn in kernels:
        _observed.setdefault(kn, []).append(cid)
    assert kernels, f'{cid}: the profiler recorded no search kernel at all'
    assert set(kernels) == set(want), \
        f'{cid}: launched {sorted(set(kernels))}, expected {sorted(want)}'


def _equal(cid, what, got, want):
    bad = np.argwhere(got != want)
    assert not len(bad), f'{cid}: {what}: {len(bad)} entries differ, first (query, rank): {bad[:6].tolist()}, ' \
                         f'got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}'


@pytest.mark.parametrize('case', CASES, ids=[_case_id(c) for c in CASES])
def test_variant_matches_oracle(case):
    cid = _case_id(case)
    d, n, nq, k, data = case['d'], case['n'], case['nq'], case['k'], case['data']
    db, q = database(d, n, data)
    idx = index(d, n, data)
    qd = torch.from_numpy(q[:nq]).cuda()
    (dist, ids), kernels = launched(lambda: idx.search_device(qd, k))
    _record(cid, kernels, case['kernels'])
    dm, im = reference(d, n, data, nq, k)
    _equal(cid, 'ids', ids.cpu().numpy(), im)
    _equal(cid, 'distances', dist.cpu().numpy(), dm)
    dist2, ids2 = idx.search_device(qd, k)
    assert torch.equal(dist, dist2) and torch.equal(ids, ids2), f'{cid}: a second call gave different bytes'
    keys = idx.search_keys_device(qd, k, id_base=ID_BASE)
    _equal(cid, 'keys', keys.cpu().numpy(), as_keys(dm, im, ID_BASE))
    if data != 'std':
        # the forced path was taken: read it off the reference distances of query 0
        full = np.abs(db.astype(np.int16) - q[0].astype(np.int16)).sum(axis=1)
        within = int((full <= dm[0, k - 1]).sum())
        if data == 'overflow':
            assert within > CMAX, f'{cid}: only {within} vectors within the k-th distance: no overflow'
        else:
            ties = int((full == dm[0, k - 1]).sum())
            assert FAST_SORT_CAP < ties and within <= 4096, f'{cid}: {ties} ties at the k-th distance, {within} within'
        _forced.setdefault((data, case['note']), []).append(cid)


# ---------------------------------------------------------------------------------------------------------------------
# external bound (dctd_l1_topk_keys with d_bound): the per-rank step of a sharded search
# ---------------------------------------------------------------------------------------------------------------------
BOUND_CASES = [
    _case(480, 5, 50, fused_path(8, 7, 30, 1), note='fused'),          # own_bound == false: no phase A
    _case(100, 9, 50, fused_path(12, 7, 0, 2), note='fused'),
    _case(16, 3, 50, {tstream(4), SELECT, scan(1, 2, 4), MERGE}, note='stream'),
    _case(480, 40, 50, {thresh(8, 8), SELECT, scan(8, 2, 4), MERGE}, note='thresh'),   # no sample, no seeds
    _case(100, 17, 50, {thresh(8, 4), SELECT, scan(4, 2, 4), MERGE}, note='thresh'),
]


@pytest.mark.parametrize('mode', ['kth', 'zero'])
@pytest.mark.parametrize('case', BOUND_CASES, ids=[_case_id(c) + '-' + c['note'] for c in BOUND_CASES])
def test_external_bound(case, mode):
    """With the true k-th distance as the bound the keys are the full top-k; with a bound of 0 only the exact matches
    are returned (duplicates by position), nothing is invented or reordered, the rest is -1."""
    cid = f'{_case_id(case)}-bound-{mode}'
    d, n, nq, k, data = case['d'], case['n'], case['nq'], case['k'], case['data']
    _, q = database(d, n, data)
    idx = index(d, n, data)
    qd = torch.from_numpy(q[:nq]).cuda()
    dm, im = reference(d, n, data, nq, k)
    if mode == 'kth':
        bound = torch.from_numpy(dm[:, k - 1].astype(np.int32)).cuda()
        want = as_keys(dm, im, ID_BASE)
    else:
        bound = torch.zeros(nq, dtype=torch.int32, device='cuda')
        want = np.where(dm == 0, as_keys(dm, im, ID_BASE), -1)
        assert (want[0] != -1).sum() > 1 and (want == -1).any()
    keys, kernels = launched(lambda: idx.search_keys_device(qd, k, id_base=ID_BASE, bound=bound))
    _record(cid, kernels, case['kernels'])
    _equal(cid, 'keys', keys.cpu().numpy(), want)
    _forced.setdefault(('bound', case['note']), []).append(cid)


def test_width_2049_is_unsupported_before_any_launch():
    """d = 2049 is beyond every kernel: dctd_l1_topk and dctd_l1_topk_keys return DCTD_ERR_UNSUPPORTED without a launch,
    and the workspace query returns 0."""
    from dctdomain_b200 import _lib
    L = _lib.lib()
    d, n, nq, k = 2049, 1000, 5, 50
    idx = __import__('dctdomain_b200.index', fromlist=['IndexFlatL1']).IndexFlatL1(d)
    idx.add(np.random.RandomState(0).randint(-128, 128, size=(n, d)).astype(np.int8))
    qd = torch.zeros((nq, d), dtype=torch.int8, device='cuda')
    assert L.dctd_l1_topk_workspace_bytes(nq, n, d, k) == 0
    ws = torch.empty(1 << 24, dtype=torch.uint8, device='cuda')
    dist = torch.empty((nq, k), dtype=torch.float32, device='cuda')
    ids = torch.empty((nq, k), dtype=torch.int64, device='cuda')
    stream = torch.cuda.current_stream().cuda_stream
    L.dctd_launch_count(1)

    def calls():
        return (L.dctd_l1_topk(qd.data_ptr(), nq, idx._packed.data_ptr(), n, d, k, 0, dist.data_ptr(), ids.data_ptr(),
                               ws.data_ptr(), ws.numel(), stream),
                L.dctd_l1_topk_keys(qd.data_ptr(), nq, idx._packed.data_ptr(), n, d, k, 0, 0, ids.data_ptr(),
                                    ws.data_ptr(), ws.numel(), 0, stream))
    rcs, kernels = launched(calls)
    assert rcs == (_lib.ERR_UNSUPPORTED, _lib.ERR_UNSUPPORTED), rcs
    assert kernels == [] and L.dctd_launch_count(1) == 0, kernels


# ---------------------------------------------------------------------------------------------------------------------
# coverage of the dispatch table
# ---------------------------------------------------------------------------------------------------------------------
def test_zz_every_release_kernel_was_launched():
    # kernel -> cases, forced path -> cases (shown with pytest -s)
    for kn in sorted(_observed):
        cids = sorted(set(_observed[kn]))
        print(f'{kn:42s} cases {len(cids):3d}')
    for (path, fam), cids in sorted(_forced.items()):
        print(f'forced {path:8s} {fam:8s} cases {len(cids):3d}: {", ".join(cids)}')
    assert _observed, 'no search kernel was observed: run the whole file'
    missing, extra = sorted(set(REQUIRED) - set(_observed)), sorted(set(_observed) - set(REQUIRED))
    assert not missing and not extra, f'never launched: {missing}; launched but not in the release table: {extra}'
    want = {('overflow', f) for f in FAMILIES} | {('ties', f) for f in FAMILIES if f != 'heap_td1'} \
        | {('bound', 'fused'), ('bound', 'stream'), ('bound', 'thresh')}
    assert set(_forced) == want, sorted(want ^ set(_forced))
