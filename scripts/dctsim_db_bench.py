"""dct-sim --db at scale: the hits path (dct_sim.protein_hits, dctd_l1_protein_hits) against the all-pairs path it
replaces (dct_sim.protein_scores + the host-side sort and cut of db_search), on synthetic proteins of 1-8 fingerprints
(4.5 on average, d = 480, values 0..127).

    python scripts/dctsim_db_bench.py [--out DIR] [--big-db N]

1. 10 000 x 10 000 proteins through both paths: CUDA-event times (end to end: H2D offsets, kernels, D2H, CSR /
   selection on the host), identical hit lists asserted.
2. 10 000 x 1 000 000 proteins through the hits path only (the all-pairs matrices would take 80 GB of HBM).
Each row reports global pairs per second (query x database proteins over the time) beside the measured SAD issue
peak of one B200 (profiles/sad_peak.json: 1.53e11 480-byte pairs/s), and the peak device memory of the call.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dctdomain_b200 import dct_sim  # noqa: E402

SAD_PEAK_PAIRS = 1.53e11          # 480-byte pairs/s on one B200 (profiles/sad_peak.json)
TOP, THRESHOLD = 5, 0.25          # dct-sim's defaults


def proteins(n, seed):
    rs = np.random.RandomState(seed)
    off = np.concatenate([[0], np.cumsum(rs.randint(1, 9, size=n))]).astype(np.int64)
    g = torch.Generator(device='cuda').manual_seed(seed)
    fps = torch.randint(0, 128, (int(off[-1]), 480), generator=g, device='cuda', dtype=torch.int8)
    return fps, off


def plant(q, db, n_related, seed):
    """global fingerprints of some database proteins = a query's with a few bytes changed (hits above the threshold)"""
    rs = np.random.RandomState(seed)
    (qf, qoff), (df, doff) = q, db
    a = rs.randint(0, len(qoff) - 1, size=n_related)
    b = rs.choice(len(doff) - 1, size=n_related, replace=False)
    rows = qf[torch.from_numpy(qoff[a + 1] - 1).cuda()].clone()
    noise = torch.from_numpy(rs.rand(n_related, 480) < 0.1).cuda()
    rows[noise] = torch.randint(0, 128, (int(noise.sum()),), device='cuda', dtype=torch.int8)
    df[torch.from_numpy(doff[b + 1] - 1).cuda()] = rows


def old_path(q, db):
    """db_search before protein_hits: all pairs, then the reference's sort and loop on the host"""
    (qf, qoff), (df, doff) = q, db
    mn, last = dct_sim.protein_scores(qf, qoff, df, doff)
    s_all = 1.0 - np.minimum(last / 17000, 1.0)
    order = np.argsort(-s_all, axis=1, kind='stable')
    off, hdb, hmin, hlast = [0], [], [], []
    for i in range(len(order)):
        n = 0
        for rank in range(order.shape[1]):
            j = int(order[i, rank])
            if rank >= TOP and s_all[i, j] < THRESHOLD:
                break
            hdb.append(j); hmin.append(mn[i, j]); hlast.append(last[i, j])
            n += 1
        off.append(off[-1] + n)
    return [np.array(x, dtype=np.int64) for x in (off, hdb, hmin, hlast)]


def new_path(q, db):
    (qf, qoff), (df, doff) = q, db
    return dct_sim.protein_hits(qf, qoff, df, doff, TOP, THRESHOLD)


def timed(fn, reps):
    """(result, [ms per call]) with CUDA events around each call (the call ends in device-to-host copies)"""
    fn()                                                   # warm-up: module load, allocator
    out, ms = None, []
    for _ in range(reps):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
        peak = torch.cuda.max_memory_allocated() - base
    return out, ms, peak


def row(name, nq, nd, ms, peak):
    best = min(ms)
    rate = nq * nd / (best * 1e-3)
    r = {'path': name, 'n_query': nq, 'n_db': nd, 'ms': [round(x, 2) for x in ms], 'best_ms': round(best, 2),
         'global_pairs_per_s': float(f'{rate:.4g}'), 'share_of_sad_peak': round(rate / SAD_PEAK_PAIRS, 4),
         'peak_device_bytes_over_inputs': int(peak)}
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='directory for the JSON summary')
    ap.add_argument('--big-db', type=int, default=1_000_000)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                          capture_output=True, text=True).stdout.strip()
    print('card:', card, flush=True)
    rows = []
    q = proteins(10_000, 1)
    db = proteins(10_000, 2)
    plant(q, db, 2_000, 3)
    got, ms, peak = timed(lambda: new_path(q, db), args.reps)
    rows.append(row('protein_hits', 10_000, 10_000, ms, peak))
    want, ms, peak = timed(lambda: old_path(q, db), args.reps)
    rows.append(row('protein_scores + host selection', 10_000, 10_000, ms, peak))
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    print('identical hit lists:', len(got[1]), 'hits', flush=True)
    del db
    torch.cuda.empty_cache()
    big = proteins(args.big_db, 4)
    plant(q, big, 20_000, 5)
    got, ms, peak = timed(lambda: new_path(q, big), args.reps)
    rows.append(row('protein_hits', 10_000, args.big_db, ms, peak))
    print('hits:', len(got[1]), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'dctsim_db_bench.json'), 'w') as f:
            json.dump({'card': card, 'top': TOP, 'threshold': THRESHOLD, 'rows': rows}, f, indent=1)


if __name__ == '__main__':
    main()
