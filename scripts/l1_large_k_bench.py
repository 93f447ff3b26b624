"""Rate of the exact L1 search at large k (dctd_l1_topk_large, csrc/l1_large.cuh) next to the heap / threshold path at
k = 992, on one GPU.

For every (nq, k): ms per call (CUDA events around `reps` calls of IndexFlatL1.search_device after one warm-up call),
pairs/s = nq * n / time, the share of the measured SAD issue peak (profiles/sad_peak.json: the fastest sad4/s over
ceil(d / 4) sad4 per pair; 1.53e11 pairs/s at d = 480) and, for k > 992, the histogram passes the call needed (the first
word of the workspace of one more call).  The database (n random int8 rows, 480 MB at the default size) is larger than
the 126 MB L2, so every pass reads HBM.  Prints the card and its power limit with the results; --out writes them as JSON.

    python scripts/l1_large_k_bench.py [--n 1000000] [--d 480] [--nqs 16,1024,8192] [--ks 992,993,2048,4096,8192]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from dctdomain_b200 import _lib  # noqa: E402
from dctdomain_b200 import index as dindex  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader',
                                '-i', str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def sad_peak_pairs(d):
    with open(os.path.join(ROOT, 'profiles', 'sad_peak.json')) as f:
        peak = max(r['sad4_per_s'] for r in json.load(f)['results'])
    return peak / ((d + 3) // 4)


def passes(idx, q, k):
    L = _lib.lib()
    nq = int(q.shape[0])
    need = L.dctd_l1_topk_large_workspace_bytes(nq, idx.ntotal, idx.d, k)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    keys = torch.empty((nq, k), dtype=torch.int64, device='cuda')
    _lib.check(L.dctd_l1_topk_large(q.data_ptr(), nq, idx._packed.data_ptr(), idx.ntotal, idx.d, k, 0, 0, 0,
                                    keys.data_ptr(), ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return int(ws[:4].view(torch.int32)[0])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--n', type=int, default=1_000_000)
    ap.add_argument('--d', type=int, default=480)
    ap.add_argument('--nqs', default='16,1024,8192')
    ap.add_argument('--ks', default='992,993,2048,4096,8192')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('needs a CUDA device')
    name, power = card()
    peak = sad_peak_pairs(args.d)
    print(f'# {name}, power limit / max SM clock: {power}; SAD peak at d = {args.d}: {peak:.3g} pairs/s', flush=True)
    g = torch.Generator(device='cuda').manual_seed(1)
    db = torch.randint(-128, 128, (args.n, args.d), dtype=torch.int8, device='cuda', generator=g)
    idx = dindex.IndexFlatL1(args.d)
    idx.add(db)
    rows = []
    for nq in (int(x) for x in args.nqs.split(',')):
        pick = torch.randint(0, args.n, (nq,), device='cuda', generator=g)
        q = (db[pick].to(torch.int16) + torch.randint(-2, 3, (nq, args.d), device='cuda', generator=g,
                                                     dtype=torch.int16)).clamp(-128, 127).to(torch.int8)
        for k in (int(x) for x in args.ks.split(',')):
            idx.search_device(q, k)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.reps):
                idx.search_device(q, k)
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / args.reps
            rate = nq * args.n / (ms * 1e-3)
            row = {'nq': nq, 'n': args.n, 'd': args.d, 'k': k, 'path': 'large' if k > dindex.K_HEAP_MAX else 'heap/threshold',
                   'ms': round(ms, 3), 'pairs_per_s': float(f'{rate:.4g}'), 'share_of_sad_peak': round(rate / peak, 4),
                   'hist_passes': passes(idx, q, k) if k > dindex.K_HEAP_MAX else None}
            rows.append(row)
            print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            json.dump({'card': name, 'power_limit_max_sm_clock': power, 'sad_peak_pairs_per_s': peak, 'reps': args.reps,
                       'results': rows}, f, indent=1)


if __name__ == '__main__':
    main()
