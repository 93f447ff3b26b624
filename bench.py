#!/usr/bin/env python
"""Benchmark of the two DCTdomain hot paths on B200 (contract: see the task statement / DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # ours (N > 1: launched by torchrun)
    python bench.py --impl reference [...]                       # the reference's CPU path (oracle port)
    python bench.py [...] --dump-outputs DIR                     # + the last timed step's fingerprints as DIR/*.npy

Primary line = BASELINE.json metric part (i), domain fingerprints/s, on configs[1]:
  100k synthetic domains, L ~ U{40..500}, two ESM-2 layers x 1280 fp32.  A step is one batch of
  --batch domains (default 4096, ~11 GB of embeddings: far larger than the 126 MB L2); the
  default 200 steps stream 819,200 domains (8x the 100k of configs[1], ~0.4 s timed).  `value` times the kernel path with inputs resident in
  HBM; `e2e` times the public Python API (`quantize_stream`: `quantize_batch` on lists of Fingerprint objects, three
  batches in flight) with pinned host embeddings, H2D + kernel + D2H of every batch inside the timed region
  (`e2e.single_call`: the same batches through back-to-back `quantize_batch` calls).
The same JSON line carries part (ii) of the metric, L1 top-50 query.DB pairs/s, with the database sharded over the
N ranks (contiguous ranges, NCCL exchange of packed keys, merge by (distance, position)):
  `search`          configs[4]: 10k-query batch x 50M fingerprints (24 GB)
  `search_1m`       8192-query batch x 1M fingerprints (configs[3] size) + the CPU restatement timed beside it
  `search_allvsall` configs[3] in full: 1M x 1M, one pass, results distributed by query slice (all_to_all)
  `search_stream`   the HBM-bound regime: 8 queries per call x the configs[4] shards (roofline: HBM)
each with `parity`: the result of the timed call compared bit for bit with the oracle over the whole database on a
subsample of the queries.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

D = 1280
LAYERS = 2
QDIM = [3, 80, 3, 80]
LMIN, LMAX = 40, 500
SAD4_PEAK_PER_GPU = 1.83e13   # measured on the B200: scripts/microbench/sad_peak.cu (63 lanes/clk/SM)


def batch_lengths(seed: int, n: int) -> np.ndarray:
    return np.random.RandomState(seed).randint(LMIN, LMAX + 1, size=n)


# ------------------------------------------------------------------------------------------------
# CPU reference arm: the reference's own Fingerprint.quantize under multiprocessing.Pool, like make_db --cpu N
# ------------------------------------------------------------------------------------------------
_CPU_EMB = None
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')      # verbatim copy of the reference's src/*.py (scripts/install_reference.py)


def reference_fingerprint_class():
    """(Fingerprint class, kind): the UNMODIFIED reference class from baseline/_ref (kind 'reference'), or None when it
    is not installed (then the oracle port stands in, kind 'port')."""
    if os.path.exists(os.path.join(REF_DIR, 'fingerprint.py')):
        import importlib.util
        spec = importlib.util.spec_from_file_location('dctd_reference_fingerprint', os.path.join(REF_DIR, 'fingerprint.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod.Fingerprint, 'reference'
    return None, 'port'


_REF_CLS = None


def _cpu_task(i):
    emb = _CPU_EMB[i % len(_CPU_EMB)]
    L = emb[15].shape[0]
    if _REF_CLS is not None:          # reference src/make_db.py:29: fp.quantize([3, 80, 3, 80]) in a Pool worker
        fp = _REF_CLS(pid=f'p{i}', seq='', embed=emb, domains=[f'1-{L}'], quants={})
        fp.quantize(QDIM)
        return int(fp.quants[f'1-{L}'].sum())
    from oracle import fingerprint_oracle as fo
    q, _ = fo.quantize_faithful(emb, [f'1-{L}'], QDIM)
    return int(q[f'1-{L}'].sum())


class CpuArm:
    """The reference's CPU path: ``Fingerprint.quantize`` of the unmodified reference module (baseline/_ref) under
    multiprocessing.Pool(cores), the `make_db.py --cpu N` pattern (src/make_db.py:48-49).  The pool and the input
    embeddings are created once (workers are forked after the inputs exist: no pickling of embeddings, which the
    reference does pay); `rate(n)` times one pool.map over n domains."""

    def __init__(self, cores: int, distinct: int = 64):
        import multiprocessing as mp
        import synth
        global _CPU_EMB, _REF_CLS
        _REF_CLS, self.kind = reference_fingerprint_class()
        lens = batch_lengths(12345, distinct)
        _CPU_EMB = [synth.layers(900 + i, int(L), D, 'white') for i, L in enumerate(lens)]
        self.cores = cores
        self.pool = mp.get_context('fork').Pool(cores)
        self.pool.map(_cpu_task, range(cores))                  # warm the workers

    def what(self):
        return ('unmodified reference src/fingerprint.py Fingerprint.quantize (baseline/_ref)' if self.kind == 'reference'
                else 'oracle port of reference fingerprint.py quantize (baseline/_ref not installed)')

    def rate(self, n_domains: int):
        t0 = time.perf_counter()
        self.pool.map(_cpu_task, range(n_domains), chunksize=1)
        dt = time.perf_counter() - t0
        return n_domains / dt, dt

    def close(self):
        self.pool.close()
        self.pool.join()


def primary_config(batch, pool, world):
    """`config` of the primary line - the same dict for our arm and for the reference arm (same workload)."""
    return {'workload': workload_name(batch), 'domains_per_step': batch, 'resident_batches': pool,
            'l2': 'inputs larger than L2 (a step streams the embeddings of domains_per_step domains, ~2.8 MB each on average)',
            'parallelism': f'domains sharded over {world} rank(s), no collective'}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    arm = CpuArm(cores)
    r0, _ = arm.rate(max(cores * 2, 16))                              # calibration, untimed
    budget_s = 90.0 / max(1, args.steps + args.warmup)                # whole run ~1.5 minutes
    per_step = int(min(max(r0 * min(budget_s, 3.0), cores * 2), 5000))
    rates = []
    for s in range(args.warmup + args.steps):
        r, dt = arm.rate(per_step)
        if s >= args.warmup:
            rates.append((r, dt))
    arm.close()
    total_t = sum(dt for _, dt in rates)
    value = per_step * len(rates) / total_t
    sample = (f'each step = {per_step} domains of the workload (L~U{{{LMIN}..{LMAX}}}, {LAYERS}x{D} fp32), {arm.what()} '
              f'under multiprocessing.Pool({cores})')
    line = {
        'impl': 'reference', 'metric': 'domain fingerprints/s', 'value': value, 'unit': 'fingerprints/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_t / len(rates) * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': primary_config(args.batch, args.pool, max(1, args.gpus)),
        'cpu_baseline': {'value': value, 'unit': 'fingerprints/s', 'cores': cores, 'kind': arm.kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'fingerprints/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


def workload_name(batch):
    return (f'configs[1]: batched fingerprinting of synthetic domains, L~U{{{LMIN}..{LMAX}}}, {LAYERS} ESM-2 layers '
            f'x {D} fp32, qdim {QDIM}; {batch} domains per step')


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.proc, self.index = None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '20', '-i', str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for row in out.strip().splitlines():
            f = [x.strip() for x in row.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        # under load = the upper half of the samples (the sampler also sees the idle edges)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {'sm_mhz': statistics.median(load) if load else None, 'sm_max_mhz': max(smax) if smax else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md, MEASURED_PEAKS.json absent)'


def traffic_for(kernel):
    path = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
    if os.path.exists(path):
        return json.load(open(path)).get(kernel)
    return None


DUMP_BYTES = 64 << 20


def dump_outputs(path, out):
    """--dump-outputs: the int8 fingerprints [domains, 480] that the last timed step wrote, as DIR/fingerprints.npy in
    float32.  The inputs come from fixed seeds, so two builds run with the same arguments can be compared row for row.
    Above DUMP_BYTES a fixed, seeded sample of rows is kept and their positions go to DIR/fingerprint_rows.npy."""
    a = out.cpu().numpy().astype(np.float32)
    os.makedirs(path, exist_ok=True)
    if a.nbytes > DUMP_BYTES:
        keep = (DUMP_BYTES - (1 << 16)) // (a.shape[1] * 4 + 8)
        rows = np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))
        a = a[rows]
        np.save(os.path.join(path, 'fingerprint_rows.npy'), rows.astype(np.float64))
    np.save(os.path.join(path, 'fingerprints.npy'), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dctdomain_b200 import _lib
    from dctdomain_b200 import index as dindex
    from dctdomain_b200.fingerprint import Fingerprint, execute_plan, make_plan, quantize_batch, quantize_stream
    from dctdomain_b200.sharded import ShardedIndex, shard_bounds, shared_pool
    import synth

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL_DEBUG is left as the caller set it (the driver reads the rank count from NCCL's own log)
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    L = _lib.lib()
    B = args.batch
    # ---- fingerprint workload: `pool` distinct resident batches (each >> L2), cycled ----
    pool = []
    torch.manual_seed(1234 + rank)
    for b in range(args.pool):
        lens = batch_lengths(1000 * rank + b, B)
        off = np.concatenate([[0], np.cumsum(lens)])
        total = int(off[-1])
        layers = [torch.randn(total, D, device=dev) for _ in range(LAYERS)]
        plan = make_plan(LAYERS, D, QDIM[0], QDIM[1], [total], [0], [1], [0] * B, list(range(B + 1)), off[:-1], off[1:])
        out = torch.empty((B, LAYERS * QDIM[0] * QDIM[1]), dtype=torch.int8, device=dev)
        ws = torch.empty(max(plan.workspace_bytes, 256), dtype=torch.uint8, device=dev)
        execute_plan(plan, [[layers[0]], [layers[1]]], out, workspace=ws)        # uploads the plan tables
        pool.append((plan, layers, out, ws))
    torch.cuda.synchronize()

    def step(i):
        plan, layers, out, ws = pool[i % len(pool)]
        execute_plan(plan, [[layers[0]], [layers[1]]], out, tables_resident=True, workspace=ws)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # warm-up: at least W steps and at least ~0.3 s, so that clocks are at their loaded level
    t_w = time.perf_counter()
    i = 0
    while i < args.warmup or time.perf_counter() - t_w < 0.3:
        step(i)
        i += 1
        if i % 8 == 0:
            torch.cuda.synchronize()
    barrier()
    L.dctd_launch_count(1)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    evs[0].record()
    for i in range(args.steps):
        step(args.warmup + i)
        evs[i + 1].record()
    barrier()
    launches = int(L.dctd_launch_count(0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pool[(args.warmup + args.steps - 1) % len(pool)][2])
    total_ms = evs[0].elapsed_time(evs[-1])
    per_step = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    algo = [pool[(args.warmup + i) % len(pool)][0].algorithmic_bytes for i in range(args.steps)]
    total_ms = max_over_ranks(total_ms)
    clocks = sampler.stop() if rank == 0 else None
    value = B * args.steps * world / (total_ms * 1e-3)
    peak, peak_src = peaks()
    achieved = sum(algo) / (sum(per_step) * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': traffic_for('fp_ws_kernel'),
                'kernel': 'fp_ws_kernel<K=2,D=1280> (csrc/fp_ws_kernel.cuh: TMA producer / FFMA2 consumers / finisher warps)',
                'algorithmic_bytes_per_launch': sum(algo) / len(algo), 'avg_launch_ms': sum(per_step) / len(per_step),
                'peak_source': peak_src,
                'frac_of_nominal_7700': achieved / 7700.0,
                'note': 'peak = measured STREAM-style copy (read + write); this kernel only reads, so frac can exceed 1'}

    # ---- e2e: public API, pinned host embeddings -> int8 fingerprints on the host ----
    Be = args.e2e_batch
    elens = batch_lengths(777 + rank, Be)
    host_fps = []
    gen = torch.Generator().manual_seed(99 + rank)
    for i, Ln in enumerate(elens):
        emb = {15: torch.randn(int(Ln), D, generator=gen).pin_memory(), 21: torch.randn(int(Ln), D, generator=gen).pin_memory()}
        host_fps.append((f'p{i}', int(Ln), emb))
    h2d = int(sum(2 * int(Ln) * D * 4 for Ln in elens))
    d2h = Be * LAYERS * QDIM[0] * QDIM[1]

    # context for e2e: what one big pinned H2D copy achieves on this box - alone, and with every rank copying at once
    big = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    dbig = torch.empty_like(big, device=dev)
    dbig.copy_(big, non_blocking=True)
    torch.cuda.synchronize()

    def link_rate():
        t0 = time.perf_counter()
        for _ in range(4):
            dbig.copy_(big, non_blocking=True)
        torch.cuda.synchronize()
        return 4 * big.numel() / (time.perf_counter() - t0) / 1e9

    link_gbps = link_rate()
    link_all = None
    if world > 1:
        barrier()
        mine = link_rate()                     # all ranks copy at the same time
        t = torch.tensor([mine, -mine], dtype=torch.float64, device=dev)
        tsum = torch.tensor([mine], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum)
        link_all = {'per_rank_max': float(t[0].item()), 'per_rank_min': float(-t[1].item()), 'aggregate': float(tsum.item())}
    del big, dbig

    def make_batch():
        return [Fingerprint(pid=pid, seq='', embed=emb, domains=[f'1-{Ln}'], quants={}) for pid, Ln, emb in host_fps]

    e2e_runs = [0]

    def e2e_run(staging, steps, pipelined, make_batch=make_batch):
        """steps * world batches of Be proteins through the public API; every batch: Fingerprint objects, H2D of all
        embeddings, kernel, D2H, quants dicts.  pipelined: quantize_stream (three batches in flight), else one
        quantize_batch call after the other.  With several ranks the batches are one shared pool: a rank draws the next
        batch index from a counter in the rendezvous store when its pipeline has room (a work queue, what a make_db over
        several GPUs would do) - the ranks of a box do not get the same share of the host's PCIe / memory bandwidth
        (gpurun_out/r2g_numa_n8.log: 20.5 vs 35.7 GB/s per rank with all eight copying), and with equal shares the slow
        ranks would set the time.  Returns (seconds: max over ranks, batches this rank processed)."""
        e2e_runs[0] += 1
        key = f'dctd_e2e_pool_{e2e_runs[0]}'
        mine = [0]

        def pool(total):
            for _ in shared_pool(total, key):
                mine[0] += 1
                yield make_batch()

        def run(batches):
            if pipelined:
                for _ in quantize_stream(batches, QDIM, device=dev, depth=e2e_depth, staging=staging):
                    pass
            else:
                for fps in batches:
                    quantize_batch(fps, QDIM, device=dev, staging=staging)
        run(make_batch() for _ in range(3))
        barrier()
        t0 = time.perf_counter()
        run(pool(steps * world))
        barrier()
        return max_over_ranks(time.perf_counter() - t0), mine[0]

    def sum_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return float(t.item())

    e2e_steps = max(3, min(args.steps, 16)) * (2 if world > 1 else 1)     # a longer pool keeps the queue's tail (<= depth batches) small
    e2e_depth = 3 if world == 1 else 2
    half_steps = max(3, e2e_steps // 2)
    e2e_s, n_mine = e2e_run('auto', e2e_steps, True)
    bytes_all = sum_over_ranks(n_mine * h2d)                       # bytes that crossed PCIe on all ranks together
    counts = None
    if world > 1:
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = n_mine
        dist.all_reduce(t)
        counts = [int(v) for v in t.tolist()]
    single_s, _ = e2e_run('auto', half_steps, False)

    def measure_pageable():
        """The same batches as plain numpy arrays in pageable memory (what the reference's .cpu().numpy() leaves in
        Fingerprint.embed, src/embedding.py:191): host threads stage them through a pinned ring (dctd_h2d_rows_staged).
        Runs after the device-resident legs: allocating and freeing 1.4 GB of separate numpy arrays leaves the host
        allocator in a state that slows the interpreter-bound `e2e_device.objects` leg for a while
        (scripts/objects_regress.py: 3.9 -> 12.4 ms per step right after the allocation)."""
        from dctdomain_b200.fingerprint import _stage_threads
        pageable_fps = [(pid, Ln, {k: np.array(v.numpy()) for k, v in emb.items()}) for pid, Ln, emb in host_fps]

        def make_batch_pageable():
            return [Fingerprint(pid=pid, seq='', embed=emb, domains=[f'1-{Ln}'], quants={}) for pid, Ln, emb in pageable_fps]

        page_steps = max(3, e2e_steps // 4)
        page_s, _ = e2e_run('auto', page_steps, True, make_batch_pageable)
        return {'value': Be * page_steps * world / page_s, 'unit': 'fingerprints/s', 'host_threads': _stage_threads(),
                'api': 'the same call on numpy arrays in pageable memory: staged through a pinned ring by host threads '
                       '(one cudaMemcpyAsync per array from pageable memory: 3.5 k fingerprints/s, gpurun_out/r2h_pageable.log)'}

    e2e = {'value': Be * e2e_steps * world / e2e_s, 'unit': 'fingerprints/s', 'h2d_bytes_per_step': int(bytes_all / (e2e_steps * world)),
           'd2h_bytes_per_step': d2h, 'steps': e2e_steps, 'domains_per_step': Be,
           'h2d_GBps_achieved': bytes_all / world / e2e_s / 1e9, 'h2d_GBps_link_pinned_copy': link_gbps,
           'h2d_GBps_link_all_ranks_copying': link_all,
           'h2d_GBps_ceiling_sm_reads': 51.5,
           'batches_per_rank': counts,
           'distribution': 'one rank' if world == 1 else 'work queue: ranks draw batches of 512 proteins from a shared counter '
                           '(steps x ranks batches in all); h2d_GBps_achieved is the mean over ranks',
           'single_call': {'value': Be * half_steps * world / single_s, 'unit': 'fingerprints/s',
                           'api': 'one quantize_batch(list[Fingerprint]) call after the other (no overlap between calls)'},
           'api': 'dctdomain_b200.fingerprint.quantize_stream(batches of list[Fingerprint]) with pinned host embeddings: '
                  f'quantize_batch per batch, {e2e_depth} batches in flight (H2D of one overlaps the host work of its neighbours); '
                  'every byte of every batch crosses PCIe inside the timed region',
           'note': 'h2d ceiling: SM-initiated reads of pinned memory (16-byte loads or TMA bulk copies alike) stop at 51.5 GB/s on '
                   'this link, one copy-engine transfer at 55.6, one transfer per array at 47.6 (scripts/microbench/h2d_pull.cu, '
                   'scripts/e2e_ab.py)'}
    if world > 1:
        # the same through one copy-engine transfer per array instead of the gather kernel: which staging route shares
        # the host's memory and PCIe root complexes better when every rank is copying
        dma_s, _ = e2e_run('dma', half_steps, True)
        e2e['staging_gather_vs_dma'] = {'gather_fingerprints_per_s': e2e['value'],
                                        'dma_fingerprints_per_s': Be * half_steps * world / dma_s}

    # ---- e2e with device-resident embeddings (the ESM-2 output never leaves the GPU) ----
    e2e_device = None
    if not args.no_fused:
        e2e_device = run_e2e_device(torch, dev, rank, world, barrier, max_over_ranks)
    e2e['pageable'] = measure_pageable()

    # ---- protein-shaped batch: 4 contiguous domains + the global '1-L' domain per protein (what make_db feeds
    #      quantize()); the global fingerprint rides on the domain items, so every row is read once ----
    fused = None
    if not args.no_fused:
        fused = run_fused(torch, dev, rank, make_plan, execute_plan, barrier, max_over_ranks, world, peak)

    longseq = None
    if not args.no_fused:
        longseq = run_windows(torch, dev, rank, make_plan, execute_plan, barrier, max_over_ranks, world, peak)

    # ---- search: part (ii) of the metric ----
    cores = os.cpu_count() or 1
    search = search_1m = allvsall = stream = None
    if not args.no_search:
        common = (dev, rank, world, dist, torch, barrier, max_over_ranks, L, cores)
        # configs[3]-sized database: a batch of 8192 queries, then the full all-vs-all pass
        sh1, rows1 = build_sharded(torch, dev, ShardedIndex, args.search_db, rank, world, 4242, keep_rows=True)
        q1 = perturbed_queries(torch, dev, dist, sh1, args.search_queries, rank, world, 7)
        search_1m = run_search(args, 'configs[3]-sized', sh1, q1, max(2, min(args.steps, 5)), 64, *common)
        if not args.no_allvsall:
            allvsall = run_allvsall(args, sh1, rows1, *common)
        del sh1, rows1, q1
        torch.cuda.empty_cache()
        if not args.no_cfg4:
            # configs[4]: 50M fingerprints (24 GB), 10k-query batch; then the streaming regime on the same shards
            sh4, _ = build_sharded(torch, dev, ShardedIndex, args.cfg4_db, rank, world, 99)
            q4 = perturbed_queries(torch, dev, dist, sh4, args.cfg4_queries, rank, world, 8)
            search = run_search(args, 'configs[4]', sh4, q4, 2, 8, *common)
            stream = run_search_stream(args, sh4, dev, rank, world, dist, torch, barrier, max_over_ranks, L, peak, cores)
            del sh4, q4
            torch.cuda.empty_cache()
        else:
            search = search_1m

    # ---- dct-sim --db / all-vs-all: protein-level scores for all pairs of two sets (SURVEY.md 8f rank 4) ----
    dctsim = None
    if not args.no_search and not args.no_dctsim and rank == 0:
        dctsim = run_dctsim(torch, dev, L, cores)

    # ---- CPU baseline (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        arm = CpuArm(cores)
        r0, _ = arm.rate(max(cores * 2, 16))                          # calibration
        n = int(min(max(r0 * 12.0, cores * 4), 20000))                # ~12 s of CPU work
        r, dt = arm.rate(n)
        arm.close()
        if search_1m is not None:
            search_1m['cpu_baseline'] = cpu_search_rate(cores)
        cpu = {'value': r, 'unit': 'fingerprints/s', 'cores': cores, 'kind': arm.kind, 'seconds': dt,
               'sample': f'{n} domains, L~U{{{LMIN}..{LMAX}}}, {LAYERS}x{D} fp32: {arm.what()} under '
                         f'multiprocessing.Pool({cores}) (embeddings pre-forked, not pickled)'}

    if rank == 0:
        line = {
            'metric': 'domain fingerprints/s', 'value': value, 'unit': 'fingerprints/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': primary_config(B, len(pool), world),
            'clocks': clocks, 'e2e': e2e, 'e2e_device': e2e_device, 'gpu_launches': launches, 'roofline': roofline, 'cpu_baseline': cpu,
            'protein_batch': fused, 'long_sequences': longseq, 'search': search, 'search_1m': search_1m,
            'search_allvsall': allvsall, 'search_stream': stream, 'dct_sim_all_pairs': dctsim,
            # part (ii) of the metric, for the strong-scaling curve (the primary line above is collective-free by nature)
            'search_scaling_input': None if search is None else {
                'metric': search['metric'], 'value': search['value'], 'unit': 'pairs/s', 'scaling': 'strong',
                'n_gpus': world, 'workload': search['config']['workload'], 'parity_mismatches': search['parity']['mismatches']},
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        # the JSON line is the LAST thing on stdout: NCCL_DEBUG output (left as the caller set it) goes to the same
        # stream from every rank, so the other ranks have finished and the group is torn down before it is printed
        if world > 1:
            time.sleep(1.0)
        sys.stdout.flush()
        print(json.dumps(line), flush=True)


def run_e2e_device(torch, dev, rank, world, barrier, max_over_ranks, n_prot=512, steps=20):
    """Public API with the embeddings already on the device (what an ESM-2 forward pass leaves there), protein-shaped
    batches (4 contiguous domains + the global one), RecCut strings in, int8 fingerprints on the host out.
    `arrays`: quantize_device over whole-batch layer tensors, results copied into pinned host memory; the host prepares
    batch i+1 (string parsing, plan) while batch i runs, as a pipeline would.  `objects`: quantize_batch on
    reference-style Fingerprint objects holding CUDA tensors, quants dicts filled (per-protein Python work dominates)."""
    from dctdomain_b200.fingerprint import Fingerprint, quantize_batch, quantize_device
    rs = np.random.RandomState(90 + rank)
    plens = rs.randint(200, 1001, size=n_prot)
    off = np.concatenate([[0], np.cumsum(plens)])
    layers = [torch.randn(int(off[-1]), D, device=dev) for _ in range(LAYERS)]
    doms = []
    for Lp in plens:
        cuts = np.sort(rs.choice(np.arange(30, Lp - 30, 25), size=3, replace=False))
        edges = [0] + [int(c) for c in cuts] + [int(Lp)]
        doms.append([f'{a + 1}-{b}' for a, b in zip(edges[:-1], edges[1:])] + [f'1-{Lp}'])
    nd = sum(len(d) for d in doms)
    width = LAYERS * QDIM[0] * QDIM[1]
    host = [torch.empty((nd, width), dtype=torch.int8).pin_memory() for _ in range(2)]
    outs = [torch.empty((nd, width), dtype=torch.int8, device=dev) for _ in range(2)]
    evs = [torch.cuda.Event() for _ in range(2)]

    def run(n):
        check = 0
        for i in range(n):
            b = i & 1
            if i >= 2:
                evs[b].synchronize()                       # batch i-2 is on the host: consume it
                check += int(host[b][0, 0])
            res = quantize_device(layers, off[:-1], plens, doms, out=outs[b])
            host[b].copy_(res.fingerprints, non_blocking=True)
            evs[b].record()
        torch.cuda.synchronize()
        return check

    run(4)
    barrier()
    t0 = time.perf_counter()
    run(steps)
    barrier()
    dt = max_over_ranks(time.perf_counter() - t0)
    embeds = [{15: layers[0][off[i]:off[i + 1]], 21: layers[1][off[i]:off[i + 1]]} for i in range(n_prot)]

    def objects_step():
        fps = [Fingerprint(pid=f'p{i}', seq='', embed=embeds[i], domains=list(doms[i]), quants={}) for i in range(n_prot)]
        quantize_batch(fps, QDIM, device=dev)
        return fps

    for _ in range(2):
        objects_step()
    barrier()
    osteps = max(3, steps // 4)
    t0 = time.perf_counter()
    for _ in range(osteps):
        objects_step()
    barrier()
    dto = max_over_ranks(time.perf_counter() - t0)
    return {'value': nd * steps * world / dt, 'unit': 'fingerprints/s', 'steps': steps, 'proteins_per_step': n_prot,
            'fingerprints_per_step': nd, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': nd * width,
            'ms_per_step': dt / steps * 1e3,
            'api': 'dctdomain_b200.fingerprint.quantize_device(layer tensors on the device, row ranges, RecCut strings) -> int8 '
                   'fingerprints copied to pinned host memory; two batches in flight',
            'objects': {'value': nd * osteps * world / dto, 'unit': 'fingerprints/s', 'steps': osteps, 'ms_per_step': dto / osteps * 1e3,
                        'api': 'quantize_batch(list[Fingerprint] holding CUDA tensors): quants dicts filled with int64 arrays '
                               'like the reference; per-protein Python work (object walk, dict updates) dominates'},
            'config': {'workload': f'{n_prot} proteins per step, L~U{{200..1000}}, 4 contiguous domains + global 1-L each, '
                                   f'{LAYERS} x {D} fp32 resident in HBM'}}


def run_fused(torch, dev, rank, make_plan, execute_plan, barrier, max_over_ranks, world, peak):
    n_prot = 2048
    rs = np.random.RandomState(50 + rank)
    plens = rs.randint(200, 1001, size=n_prot)
    poff = np.concatenate([[0], np.cumsum(plens)])
    total = int(poff[-1])
    layers = [torch.randn(total, D, device=dev) for _ in range(LAYERS)]
    dom_prot, sb, se = [], [], []
    for p, Lp in enumerate(plens):
        cuts = np.sort(rs.choice(np.arange(30, Lp - 30, 25), size=3, replace=False))
        edges = [0] + [int(c) for c in cuts] + [int(Lp)]
        for a, b in zip(edges[:-1], edges[1:]):
            dom_prot.append(p); sb.append(a); se.append(b)
        dom_prot.append(p); sb.append(0); se.append(int(Lp))
    nd = len(dom_prot)
    srcs = [[layers[l][poff[p]:poff[p + 1]] for p in range(n_prot)] for l in range(LAYERS)]
    plan = make_plan(LAYERS, D, QDIM[0], QDIM[1], plens, list(range(n_prot)), [1] * n_prot, dom_prot,
                     list(range(nd + 1)), sb, se)
    out = torch.empty((nd, LAYERS * QDIM[0] * QDIM[1]), dtype=torch.int8, device=dev)
    ws = torch.empty(max(plan.workspace_bytes, 256), dtype=torch.uint8, device=dev)
    for _ in range(3):
        execute_plan(plan, srcs, out, workspace=ws)
    barrier()
    steps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        execute_plan(plan, srcs, out, tables_resident=True, workspace=ws)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    unique = LAYERS * total * D * 4
    return {'metric': 'domain fingerprints/s (protein-shaped batch, global fingerprint fused)', 'value': nd * world / ms * 1e3,
            'unit': 'fingerprints/s', 'ms_per_step': ms, 'proteins_per_step': n_prot, 'fingerprints_per_step': nd,
            'config': {'workload': '2048 proteins, L~U{200..1000}, 4 contiguous domains + global 1-L each, 2 x 1280 fp32'},
            'roofline': {'bound': 'hbm', 'achieved': unique / ms / 1e6, 'peak': peak, 'unit': 'GB/s',
                         'frac': unique / ms / 1e6 / peak,
                         'algorithmic_bytes_per_launch': unique,
                         'note': 'algorithmic bytes = every embedding row once (SURVEY.md 8d: the global and the domain '
                                 'fingerprints share one read); unfused, the same work reads 2x the bytes'}}


def run_windows(torch, dev, rank, make_plan, execute_plan, barrier, max_over_ranks, world, peak, n_prot=384,
                maxlen=500, overlap=200):
    """configs[2]: long proteins (L ~ U{501..4000}) delivered as the maxlen windows `extract_esm2` returns (stride
    maxlen - overlap; rows covered by two windows are averaged in-kernel, src/embedding.py:153-192), 3-12 contiguous
    domains + the global fingerprint per protein."""
    rs = np.random.RandomState(70 + rank)
    stride = maxlen - overlap
    src_rows, prot_src0, prot_nsrc, plens = [], [], [], []
    for Lp in rs.randint(501, 4001, size=n_prot):
        prot_src0.append(len(src_rows))
        start = 0
        while True:
            rows = int(min(maxlen, Lp - start))
            if start > 0 and rows <= overlap:        # split_seq keeps a window only if it is longer than the overlap
                break
            src_rows.append(rows)
            if start + rows >= Lp:
                break
            start += stride
        prot_nsrc.append(len(src_rows) - prot_src0[-1])
        plens.append((prot_nsrc[-1] - 1) * stride + src_rows[-1])
    total = int(sum(src_rows))
    layers = [torch.randn(total, D, device=dev) for _ in range(LAYERS)]
    off = np.concatenate([[0], np.cumsum(src_rows)])
    srcs = [[layers[l][off[i]:off[i + 1]] for i in range(len(src_rows))] for l in range(LAYERS)]
    dom_prot, sb, se = [], [], []
    for p, Lp in enumerate(plens):
        cuts = np.sort(rs.choice(np.arange(30, Lp - 30, 10), size=rs.randint(3, 13) - 1, replace=False))
        edges = [0] + [int(c) for c in cuts] + [int(Lp)]
        for a, b in zip(edges[:-1], edges[1:]):
            dom_prot.append(p); sb.append(a); se.append(b)
        dom_prot.append(p); sb.append(0); se.append(int(Lp))
    nd = len(dom_prot)
    plan = make_plan(LAYERS, D, QDIM[0], QDIM[1], src_rows, prot_src0, prot_nsrc, dom_prot, list(range(nd + 1)), sb, se,
                     maxlen=maxlen, overlap=overlap)
    out = torch.empty((nd, LAYERS * QDIM[0] * QDIM[1]), dtype=torch.int8, device=dev)
    ws = torch.empty(max(plan.workspace_bytes, 256), dtype=torch.uint8, device=dev)
    for _ in range(3):
        execute_plan(plan, srcs, out, workspace=ws)
    barrier()
    steps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        execute_plan(plan, srcs, out, tables_resident=True, workspace=ws)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    nbytes = LAYERS * total * D * 4
    return {'metric': 'domain fingerprints/s (long sequences delivered as maxlen windows)', 'value': nd * world / ms * 1e3,
            'unit': 'fingerprints/s', 'ms_per_step': ms, 'proteins_per_step': n_prot, 'fingerprints_per_step': nd,
            'config': {'workload': f'configs[2]: {n_prot} proteins, L~U{{501..4000}} as windows of {maxlen} rows / stride '
                                   f'{stride} ({len(src_rows)} windows), 3-12 contiguous domains + global 1-L each, 2 x 1280 fp32'},
            'roofline': {'bound': 'hbm', 'achieved': nbytes / ms / 1e6, 'peak': peak, 'unit': 'GB/s',
                         'frac': nbytes / ms / 1e6 / peak, 'algorithmic_bytes_per_launch': nbytes,
                         'note': 'algorithmic bytes = every window row once (SURVEY.md 8d); the overlap average and the '
                                 'riding global fingerprint add no reads'}}


SLICE = 1 << 20     # rows generated / copied per piece


def synth_rows(torch, dev, n, seed):
    """n synthetic int8[480] fingerprints on the device (values 0..127, clip(N(63.6, 27.7)) like real ones)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.clamp(torch.randn((n, 480), generator=g, device=dev) * 27.7 + 63.6, 0, 127).round().to(torch.int8)


def build_sharded(torch, dev, ShardedIndex, n_db, rank, world, seed, keep_rows=False):
    """This rank's contiguous shard of an n_db-row database, generated on the device piece by piece."""
    sh = ShardedIndex(480, n_db, rank=rank, world=world, device=dev)
    n_local = sh.end - sh.begin
    sh.index.reserve(n_local)
    kept = []
    for a in range(0, n_local, SLICE):
        rows = synth_rows(torch, dev, min(SLICE, n_local - a), seed * 1000003 + rank * 7919 + a // SLICE)
        sh.index.add(rows)
        if keep_rows:
            kept.append(rows)
    return sh, (torch.cat(kept) if keep_rows and kept else None)


def perturbed_queries(torch, dev, dist, sh, nq, rank, world, seed):
    """Queries = perturbed rows of rank 0's shard (so that true neighbours and ties exist), replicated."""
    if rank == 0:
        g = torch.Generator(device=dev).manual_seed(seed)
        pool_n = min(sh.end - sh.begin, SLICE)
        pool = torch.from_numpy(sh.index.reconstruct_n(0, pool_n)).to(dev)
        rows = torch.randint(0, pool_n, (nq,), generator=g, device=dev)
        q = torch.clamp(pool[rows].to(torch.int16) + torch.randint(-3, 4, (nq, 480), generator=g, device=dev).to(torch.int16),
                        0, 127).to(torch.int8)
    else:
        q = torch.empty((nq, 480), dtype=torch.int8, device=dev)
    if world > 1:
        dist.broadcast(q, 0)
    return q


def oracle_topk_sharded(torch, dist, dev, sh, q_host, k, world, threads):
    """The oracle (oracle/l1_flat.c, faiss flat-L1 restated) over the WHOLE database: every rank scans its own shard
    piece by piece on the host, the per-rank lists are exchanged and merged by (distance, id) with numpy.  Collective:
    all ranks call it with the same queries.  This is the checker, never the thing measured."""
    from oracle import search_oracle as so
    m = len(q_host)
    big = np.iinfo(np.int64).max

    def merge(d, i):
        order = np.lexsort((np.where(i < 0, big, i), d), axis=1)[:, :k]
        return np.take_along_axis(d, order, 1), np.take_along_axis(i, order, 1)

    bd = np.full((m, k), so.FLT_MAX, dtype=np.float32)
    bi = np.full((m, k), -1, dtype=np.int64)
    n_local = sh.end - sh.begin
    for a in range(0, n_local, SLICE):
        rows = sh.index.reconstruct_n(a, min(SLICE, n_local - a))
        d, i = so.l1_topk(q_host, rows, k, threads=threads)
        i = np.where(i >= 0, i + sh.begin + a, -1)
        bd, bi = merge(np.concatenate([bd, d], 1), np.concatenate([bi, i], 1))
    if world > 1:
        td, ti = torch.from_numpy(bd).to(dev), torch.from_numpy(bi).to(dev)
        ad = torch.empty((world,) + td.shape, dtype=td.dtype, device=dev)
        ai = torch.empty((world,) + ti.shape, dtype=ti.dtype, device=dev)
        dist.all_gather_into_tensor(ad, td)
        dist.all_gather_into_tensor(ai, ti)
        bd, bi = merge(ad.permute(1, 0, 2).reshape(m, world * k).cpu().numpy(),
                       ai.permute(1, 0, 2).reshape(m, world * k).cpu().numpy())
    return bd, bi


def parity_record(got_d, got_i, want_d, want_i, note):
    bad = int((~((got_i == want_i).all(axis=1) & (got_d == want_d).all(axis=1))).sum())
    return {'checked': int(len(want_i)), 'mismatches': bad,
            'oracle': 'oracle/l1_flat.c (faiss 1.7.4 flat-L1 restated) over the full database, shard by shard, merged '
                      'by (distance, id) with numpy; compared bit for bit (ids and float32 distances)', 'queries': note}


def phase_ms(sh, fn):
    """Per-step CUDA-event times of one call of fn() (ShardedIndex marks an event after every step)."""
    sh.events = []
    fn()
    import torch
    torch.cuda.synchronize()
    ev, out = sh.events, {}
    sh.events = None
    for (n0, e0), (n1, e1) in zip(ev[:-1], ev[1:]):
        if n1 != 'start':
            out[n1] = out.get(n1, 0.0) + e0.elapsed_time(e1)
    return out


def search_roofline(pairs, ms_total, db_bytes_rank, world):
    sad_peak = SAD4_PEAK_PER_GPU * world          # scripts/microbench/sad_peak.cu, profiles/sad_peak.json
    sad_rate = pairs * 120 / (ms_total * 1e-3)
    return {'bound': 'integer pipe (VABSDIFF4.U8.ACC, 120 per pair; not HBM: the shard streams at %.1f GB/s per rank)'
                     % (db_bytes_rank / (ms_total * 1e-3) / 1e9),
            'achieved': sad_rate, 'peak': sad_peak, 'unit': 'SAD4 lane-ops/s', 'frac': sad_rate / sad_peak,
            'peak_source': 'measured VABSDIFF4 issue peak, 63 lanes/clk/SM x 148 SMs x 1.965 GHz '
                           '(scripts/microbench/sad_peak.cu)'}


def run_search(args, tag, sh, q, steps, parity_q, dev, rank, world, dist, torch, barrier, max_over_ranks, L, cores):
    """Part (ii) of the metric on one sharded database: timed ShardedIndex.search (queries and shard in HBM), the
    per-step times of one call, the same call through the host-array API (e2e) and the oracle comparison."""
    n_db, nq, k = sh.n_total, int(q.shape[0]), 50
    for _ in range(2):
        dd, ii = sh.search(q, k)
    barrier()
    L.dctd_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        dd, ii = sh.search(q, k)
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = int(L.dctd_launch_count(0))
    path = sh.last_path
    phases = phase_ms(sh, lambda: sh.search(q, k))
    pairs = float(nq) * n_db * steps
    # e2e: host queries in, host results out on every rank (faiss-style index.search)
    qh = q.cpu().numpy()
    sh.search(qh, k)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        hd, hi = sh.search(qh, k)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    # parity on a subsample of the queries against the oracle over the full database
    rs = np.random.RandomState(17)
    sel = np.sort(rs.choice(nq, size=min(parity_q, nq), replace=False))
    want_d, want_i = oracle_topk_sharded(torch, dist, dev, sh, qh[sel], k, world, max(1, cores // world))
    parity = parity_record(hd[sel], hi[sel], want_d, want_i, f'{len(sel)} of the {nq} timed queries (host-array API result)')
    dev_same = bool(np.array_equal(dd.cpu().numpy(), hd) and np.array_equal(ii.cpu().numpy(), hi))
    parity['device_api_equals_host_api'] = dev_same
    return {'metric': 'L1 top-50 query.DB pairs/s', 'value': pairs / (ms * 1e-3), 'unit': 'pairs/s', 'ms_per_step': ms / steps,
            'steps': steps, 'scaling': 'strong', 'dtype': 'u8', 'gpu_launches': launches, 'n_gpus': world,
            'config': {'workload': f'{tag}: {nq} queries x {n_db} int8[480] fingerprints, k=50, database sharded over '
                                   f'{world} rank(s) (contiguous ranges), exchange: {path}',
                       'n_db': n_db, 'nq': nq, 'k': k},
            'phases_ms': phases,
            'e2e': {'value': pairs / e2e_s, 'unit': 'pairs/s', 'h2d_bytes_per_step': nq * 480, 'd2h_bytes_per_step': nq * k * 12,
                    'api': 'ShardedIndex.search(numpy queries, k) -> numpy (dist, ids) on every rank'},
            'e2e_pairs_per_s': pairs / e2e_s,
            'parity': parity,
            'roofline': search_roofline(pairs, ms, (sh.end - sh.begin) * 480 * steps, world)}


def run_allvsall(args, sh, rows_local, dev, rank, world, dist, torch, barrier, max_over_ranks, L, cores):
    """configs[3] in full: every fingerprint of the database against the whole database, top-50.  Queries go through in
    batches of 8192; every rank scans its shard for the whole batch and merges / keeps the results of its slice of the
    batch (all_to_all of the packed keys)."""
    n_db, k, B = sh.n_total, 50, 8192
    if n_db % world:
        return None
    if world > 1:
        allrows = torch.empty((n_db, 480), dtype=torch.int8, device=dev)
        dist.all_gather_into_tensor(allrows, rows_local.contiguous())
    else:
        allrows = rows_local
    sh.search_slice(allrows[:B], k)                     # warm-up of this code path
    barrier()
    L.dctd_launch_count(1)
    keep = None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for b in range(0, n_db, B):
        r = sh.search_slice(allrows[b:b + B], k)
        if b == 0:
            keep = r
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = int(L.dctd_launch_count(0))
    path = sh.last_path
    # parity: 4 queries of every rank's slice of the first batch
    per = -(-min(B, n_db) // world)
    sel = np.concatenate([np.arange(j * per, j * per + 4) for j in range(world)])
    want_d, want_i = oracle_topk_sharded(torch, dist, dev, sh, allrows[sel].cpu().numpy(), k, world, max(1, cores // world))
    dm, im, qb, qe = keep
    mine = slice(rank * 4, rank * 4 + 4)
    rec = parity_record(dm[:4].cpu().numpy(), im[:4].cpu().numpy(), want_d[mine], want_i[mine], '')
    bad = torch.tensor([rec['mismatches']], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(bad)
    rec.update(checked=4 * world, mismatches=int(bad.item()),
               queries='4 queries of every rank\'s slice of the first batch (each rank checks the rows it keeps)')
    pairs = float(n_db) * n_db
    return {'metric': 'L1 top-50 query.DB pairs/s (all-vs-all)', 'value': pairs / (ms * 1e-3), 'unit': 'pairs/s',
            'seconds': ms * 1e-3, 'batches': -(-n_db // B), 'scaling': 'strong', 'dtype': 'u8', 'gpu_launches': launches,
            'n_gpus': world,
            'config': {'workload': f'configs[3]: all-vs-all L1 top-50 over {n_db} int8[480] fingerprints, one full pass, '
                                   f'database sharded over {world} rank(s), results distributed by query slice, exchange: {path}',
                       'n_db': n_db, 'nq': n_db, 'k': k},
            'parity': rec, 'roofline': search_roofline(pairs, ms, (sh.end - sh.begin) * 480 * (-(-n_db // B)), world)}


def run_search_stream(args, sh, dev, rank, world, dist, torch, barrier, max_over_ranks, L, peak, cores):
    """The HBM-bound regime: a reference-style call (8 query fingerprints, src/query_db.py:87) against the sharded
    configs[4] database; per call every rank streams its shard once, then all_gather + merge."""
    n_db, nq, k = sh.n_total, 8, 50
    q = synth_rows(torch, dev, nq, 5)
    if world > 1:
        dist.broadcast(q, 0)
    for _ in range(3):
        sh.search(q, k)
    barrier()
    steps = 20
    L.dctd_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        dd, ii = sh.search(q, k)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    launches = int(L.dctd_launch_count(0))
    path = sh.last_path
    phases = phase_ms(sh, lambda: sh.search(q, k))
    qh = q.cpu().numpy()                     # e2e: faiss-style index.search(host int8 array) -> host arrays
    sh.search(qh, k)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        hd, hi = sh.search(qh, k)
    barrier()
    e2e_ms = max_over_ranks(time.perf_counter() - t0) / steps * 1e3
    want_d, want_i = oracle_topk_sharded(torch, dist, dev, sh, qh, k, world, max(1, cores // world))
    parity = parity_record(hd, hi, want_d, want_i, 'all 8 queries')
    shard_bytes = (sh.end - sh.begin) * 480
    gbs = shard_bytes / ms / 1e6
    return {'metric': 'L1 top-50 query.DB pairs/s (streaming regime)', 'value': nq * n_db / ms * 1e3, 'unit': 'pairs/s',
            'ms_per_step': ms, 'steps': steps, 'dtype': 'u8', 'gpu_launches': launches, 'n_gpus': world,
            'e2e_pairs_per_s': nq * n_db / e2e_ms * 1e3, 'e2e_ms_per_call': e2e_ms, 'phases_ms': phases, 'parity': parity,
            'config': {'workload': f'{nq} queries per call (the reference calls index.search with 1-13, src/query_db.py:87) x '
                                   f'{n_db} int8[480] fingerprints sharded over {world} rank(s) ({shard_bytes / 1e9:.1f} GB per '
                                   f'rank >> L2), k=50, exchange: {path}',
                       'n_db': n_db, 'nq': nq, 'k': k},
            'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s per GPU', 'frac': gbs / peak,
                         'algorithmic_bytes_per_launch': shard_bytes,
                         'note': 'per rank: shard bytes / time of the WHOLE call (threshold sample, stream, select, NCCL '
                                 'all-gather, merge), max over ranks',
                         'kernel': 'l1 streaming kernel (csrc/l1topk.cu), every shard streamed once per call'}}


def run_dctsim(torch, dev, L, cores, n_prot=10_000):
    """`dct-sim.py --db` at scale (src/dct-sim.py:126-156): n_prot query proteins against n_prot database proteins, 2-7
    fingerprints each (RecCut domains + the global one); per protein pair the minimum over all fingerprint pairs and the
    last-vs-last distance.  Device time of dctd_l1_protein_scores (both sets resident), the whole call from host arrays,
    and a numpy check of a sample of protein pairs."""
    from dctdomain_b200 import dct_sim
    rs = np.random.RandomState(11)
    sets = []
    for sd in (1, 2):
        counts = rs.randint(2, 8, size=n_prot)
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        sets.append((synth_rows(torch, dev, int(off[-1]), 500 + sd), off))
    (qf, qoff), (df, doff) = sets
    n_qf, n_df = int(qoff[-1]), int(doff[-1])
    stream = torch.cuda.current_stream(dev).cuda_stream
    packed = torch.empty(int(L.dctd_l1_packed_bytes(n_df, 480)), dtype=torch.uint8, device=dev)
    L.dctd_l1_pack(df.data_ptr(), n_df, 480, 0, packed.data_ptr(), stream)
    ws = torch.empty(int(L.dctd_l1_protein_scores_workspace_bytes(n_qf, n_prot, n_df, n_prot, 480)), dtype=torch.uint8, device=dev)
    mn = torch.empty((n_prot, n_prot), dtype=torch.int32, device=dev)
    last = torch.empty_like(mn)

    def call():
        rc = L.dctd_l1_protein_scores(qf.data_ptr(), qoff.ctypes.data, n_prot, packed.data_ptr(), doff.ctypes.data, n_prot, 480,
                                      mn.data_ptr(), last.data_ptr(), ws.data_ptr(), ws.numel(), stream)
        assert rc == 0, rc

    call()
    torch.cuda.synchronize()
    L.dctd_launch_count(1)
    steps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    launches = int(L.dctd_launch_count(0)) // steps
    qh, dh = qf.cpu().numpy(), df.cpu().numpy()
    t0 = time.perf_counter()
    hm, hl = dct_sim.protein_scores(qh, qoff, dh, doff)
    e2e_s = time.perf_counter() - t0
    bad = 0
    sel = rs.randint(0, n_prot, size=(64, 2))
    for a, b in sel:
        blk = np.abs(qh[qoff[a]:qoff[a + 1], None, :].astype(np.int32) - dh[None, doff[b]:doff[b + 1], :].astype(np.int32)).sum(axis=2)
        bad += int(hm[a, b] != blk.min() or hl[a, b] != blk[-1, -1])
    same = bool(np.array_equal(mn.cpu().numpy(), hm) and np.array_equal(last.cpu().numpy(), hl))
    fp_pairs = float(n_qf) * n_df
    sad = fp_pairs * 120 / (ms * 1e-3)
    return {'metric': 'protein pairs/s (dct-sim --db: min over fingerprint pairs + last-vs-last)', 'value': float(n_prot) * n_prot / ms * 1e3,
            'unit': 'protein pairs/s', 'ms_per_step': ms, 'steps': steps, 'gpu_launches': launches, 'dtype': 'u8',
            'fingerprint_pairs_per_s': fp_pairs / ms * 1e3,
            'e2e': {'value': float(n_prot) * n_prot / e2e_s, 'unit': 'protein pairs/s', 'seconds': e2e_s,
                    'h2d_bytes_per_step': (n_qf + n_df) * 480, 'd2h_bytes_per_step': 2 * n_prot * n_prot * 4,
                    'api': 'dctdomain_b200.dct_sim.protein_scores(host arrays) -> int64 [n_q, n_db] x 2 (pack + kernel + D2H + widening)'},
            'parity': {'checked': 64, 'mismatches': bad, 'oracle': 'numpy |a - b|.sum over every fingerprint pair of 64 random protein pairs',
                       'device_api_equals_host_api': same},
            'config': {'workload': f'{n_prot} x {n_prot} proteins, 2-7 int8[480] fingerprints each ({n_qf} x {n_df} fingerprint pairs)'},
            'roofline': {'bound': 'integer pipe (VABSDIFF4.U8.ACC, 120 per fingerprint pair)', 'achieved': sad, 'peak': SAD4_PEAK_PER_GPU,
                         'unit': 'SAD4 lane-ops/s', 'frac': sad / SAD4_PEAK_PER_GPU,
                         'kernel': 'l1_protein_kernel<16,8,2,4,30> + l1_protein_reduce_kernel (csrc/l1_protein.cuh)'}}


def cpu_search_rate(cores):
    """pairs/s of the faiss-style CPU restatement (oracle/l1_flat.c: float32 database, OpenMP over queries) on a
    bounded sample of the configs[3] workload."""
    from oracle import search_oracle as so
    rs = np.random.RandomState(3)
    n_db = 200_000
    db = np.clip(np.rint(rs.randn(n_db, 480) * 27.7 + 63.6), 0, 127).astype(np.float32)
    nq0 = 4 * max(cores, 8)
    q = db[rs.randint(0, n_db, size=nq0)].copy()
    so.l1_topk(q, db, 50, threads=cores)                        # warm-up + calibration
    t0 = time.perf_counter()
    so.l1_topk(q, db, 50, threads=cores)
    r0 = nq0 * n_db / (time.perf_counter() - t0)
    nq = int(min(max(r0 * 6.0 / n_db, nq0), 4096)) // cores * cores or cores      # ~6 s of CPU work
    q = db[rs.randint(0, n_db, size=nq)].copy()
    t0 = time.perf_counter()
    so.l1_topk(q, db, 50, threads=cores)
    dt = time.perf_counter() - t0
    return {'value': nq * n_db / dt, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'seconds': dt,
            'sample': f'{nq} queries x {n_db} float32[480] vectors, k=50: C restatement of faiss 1.7.4 IndexFlat L1 '
                      f'(knn_extra_metrics, OpenMP over queries, {cores} threads); faiss itself is not in the image'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=4096, help='domains per step')
    ap.add_argument('--pool', type=int, default=3, help='distinct resident batches cycled through')
    ap.add_argument('--e2e-batch', type=int, default=512)
    ap.add_argument('--search-db', type=int, default=1_000_000)
    ap.add_argument('--search-queries', type=int, default=8192)
    ap.add_argument('--cfg4-db', type=int, default=50_000_000, help='configs[4] database size (sharded over the ranks)')
    ap.add_argument('--cfg4-queries', type=int, default=10_000)
    ap.add_argument('--no-cfg4', action='store_true')
    ap.add_argument('--no-allvsall', action='store_true')
    ap.add_argument('--no-search', action='store_true')
    ap.add_argument('--no-dctsim', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-fused', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the fingerprints of the last timed step to DIR/*.npy (float32), for comparing two builds')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
