"""Every kernel instantiation that dctd_fp_execute can pick in a release build, each against the float64 oracle.

dctd_fp_execute (csrc/fingerprint.cu) chooses among the warp-specialised kernel fp_ws_kernel<K, DC, RIDER> and ~40
instantiations of the general kernel fp_kernel<K, VEC, U, MAXT, MINB, LDC, RLC, RIDER>.  The choice depends on D, n
(K = n - 1), m, whether every source row is 16-byte aligned (VEC = 4), whether ld == D, whether the batch holds a fused
protein (RIDER) and the plan flags.  Each case below names the instantiation it is meant to reach and checks:

  * that this instantiation, and no other, was launched (torch.profiler kernel names);
  * the bytes against oracle/fingerprint_oracle.quantize_matrix on the stitched float32 inputs: every byte within 1 LSB,
    at most 1 % of a case's bytes off and at most 0.1 % of an instantiation's bytes over all its cases;
  * that a second launch gives the same bytes;
  * that nothing is read outside a source: every source sits in one NaN-filled arena with NaN rows between sources (and
    NaN pad columns when ld > D), so a stray read turns a (domain, layer) into zeros;
  * that nothing is written outside the fingerprint: the output rows are wider than n_layers * n * m and the pad
    columns keep a sentinel.

The last tests check that the instantiations observed are exactly the release dispatch table (a dispatcher change that
orphans a variant fails there), the user-facing entry points quantize_batch / quantize_device, and the widths that do
not fit in shared memory."""
import functools
import re

import numpy as np
import pytest
import torch

import cases
import synth
from oracle import fingerprint_oracle as fo

pytestmark = pytest.mark.gpu

TOL_CASE = 1e-2         # bytes off by 1 LSB, per case
TOL_INST = 1e-3         # bytes off by 1 LSB, summed over the cases of one instantiation (BASELINE.json north_star)
MAXLEN, OVERLAP = 500, 200
SENTINEL = -99          # the kernel writes 0..127 only
OUT_PAD = 13            # extra bytes per output row
GAP_ROWS = 2            # NaN rows between two sources of the arena
NO_FUSION, GENERAL = 1, 2   # _lib.FP_PLAN_NO_FUSION, _lib.FP_PLAN_GENERAL_KERNEL


def ws(dc, rider):
    return f'fp_ws_kernel<2,{dc},{int(rider)}>'


def fk(*args):
    """fp_kernel<K, VEC, U, MAXT, MINB, LDC = 0, RLC = 0, RIDER = 0> with the defaults spelled out."""
    args = list(args) + [0] * (8 - len(args))
    return 'fp_kernel<' + ','.join(str(int(a)) for a in args) + '>'


def pick_k(vec, maxt, minb, k):
    return fk(k, vec, 8, maxt, minb)


def pick_rider(vec, maxt, minb, k):
    return fk(k, vec, 8, maxt, minb, 0, 0, 1)


# The release dispatch table of dctd_fp_execute.  Left out: fp_kernel<2,4,8,320,2,640,2> (needs two row lanes at
# D = 640, which make_layout only chooses for dctd_fp_set_variant(5)) and the g_variant 1 / 2 / 4 / 6 kernels: they are
# reachable through dctd_fp_set_variant only, which exists in the tuning build alone.
REQUIRED = sorted(
    [ws(dc, r) for dc in (1280, 640, 1024, 480) for r in (False, True)]
    + [fk(2, 4, 8, 320, 2, 1280, 1), fk(2, 4, 8, 160, 4, 640, 1), fk(2, 4, 8, 256, 2, 1024, 1),
       fk(2, 4, 8, 320, 2, 320, 4), fk(2, 4, 8, 640, 1, 2560, 1),
       fk(2, 4, 8, 320, 2, 1280, 1, 1), fk(2, 4, 8, 160, 3, 640, 1, 1)]
    + [pick_k(v, t, b, k) for v, t, b in ((4, 320, 2), (4, 640, 1), (1, 640, 1)) for k in range(1, 8)]
    + [pick_rider(v, t, b, k) for v, t, b in ((4, 320, 2), (4, 640, 1), (1, 640, 1)) for k in range(1, 4)])


def _case(target, D, n, m, layout='contig', fused=False, flags=0, pad=0):
    """layout: 'contig' (16-byte aligned sources, ld == D), 'shift4' (every source 4 bytes past a 16-byte boundary)
    or 'ld' (rows of ld = D + pad floats, columns D.. are NaN).  fused: the batch keeps its fused proteins; otherwise
    the plan is made with FP_PLAN_NO_FUSION (the same batch, every domain streamed on its own)."""
    if not fused:
        flags |= NO_FUSION
    return dict(target=target, D=D, qdim=(n, m, n, m), layout=layout, fused=fused, flags=flags, pad=pad)


CASES = []
# warp-specialised kernel: n = 3, contiguous aligned rows, m <= 84 (3 * ((m + 1) / 2) * 2 <= 256 finisher threads);
# pass-2a pairs (k, k + H), the parity-split cosine table and the pass-2b column pairs c / m-1-c all depend on m
for _dc, (_odd, _even) in ((1280, (47, 58)), (640, (63, 30)), (1024, (33, 66)), (480, (71, 12))):
    for _r in (False, True):
        for _m in (_odd, _even, 2, 84):
            CASES.append(_case(ws(_dc, _r), _dc, 3, _m, fused=_r))
CASES += [
    # m = 85 does not fit the warp-specialised finishers: the general kernel's D = 1280 specialisations
    _case(fk(2, 4, 8, 320, 2, 1280, 1), 1280, 3, 85),
    _case(fk(2, 4, 8, 320, 2, 1280, 1, 1), 1280, 3, 85, fused=True),
    # the other width specialisations
    _case(fk(2, 4, 8, 160, 4, 640, 1), 640, 3, 100),
    _case(fk(2, 4, 8, 160, 3, 640, 1, 1), 640, 3, 96, fused=True),
    _case(fk(2, 4, 8, 256, 2, 1024, 1), 1024, 3, 72, flags=GENERAL),
    _case(fk(2, 4, 8, 320, 2, 320, 4), 320, 3, 80),                      # ESM-2 t6: four row lanes
    _case(fk(2, 4, 8, 640, 1, 2560, 1), 2560, 3, 80),                    # ESM-2 3B without fusion
    # pick_k<4,8,320,2>: float4 rows, T <= 320 (D <= 1280)
    _case(pick_k(4, 320, 2, 1), 768, 2, 64),
    _case(pick_k(4, 320, 2, 2), 768, 3, 80),                             # a width without a specialisation
    _case(pick_k(4, 320, 2, 2), 1280, 3, 80, layout='ld', pad=8),        # ld > D
    _case(pick_k(4, 320, 2, 3), 256, 4, 100),                            # five row lanes
    _case(pick_k(4, 320, 2, 4), 1280, 5, 128, layout='ld', pad=4),
    _case(pick_k(4, 320, 2, 5), 512, 6, 37),
    _case(pick_k(4, 320, 2, 6), 96, 7, 16),                              # thirteen row lanes
    _case(pick_k(4, 320, 2, 7), 1024, 8, 61),
    # pick_k<4,8,640,1>: float4 rows, D > 1280; D > 2560 has more than one column tile per thread (CT > 1)
    _case(pick_k(4, 640, 1, 1), 1536, 2, 80),
    _case(pick_k(4, 640, 1, 2), 4096, 3, 80),                            # CT = 2
    _case(pick_k(4, 640, 1, 2), 2560, 3, 80, layout='ld', pad=4),
    _case(pick_k(4, 640, 1, 3), 2048, 4, 99),
    _case(pick_k(4, 640, 1, 4), 2560, 5, 50),
    _case(pick_k(4, 640, 1, 5), 2576, 6, 128),                           # CT = 2, the second tile nearly empty
    _case(pick_k(4, 640, 1, 6), 1536, 7, 7),
    _case(pick_k(4, 640, 1, 7), 1792, 8, 120),
    # pick_k<1,8,640,1>: scalar loads (odd D, D % 4 != 0, ld % 4 != 0 or sources not 16-byte aligned)
    _case(pick_k(1, 640, 1, 1), 333, 2, 50),                             # odd D: the middle column of pass 2a
    _case(pick_k(1, 640, 1, 2), 1280, 3, 80, layout='shift4'),           # CT = 2
    _case(pick_k(1, 640, 1, 3), 1023, 4, 64),                            # odd D, CT = 2
    _case(pick_k(1, 640, 1, 4), 640, 5, 81, layout='ld', pad=3),
    _case(pick_k(1, 640, 1, 5), 127, 6, 31),                             # odd D, two row lanes
    _case(pick_k(1, 640, 1, 6), 1280, 7, 9, layout='shift4'),
    _case(pick_k(1, 640, 1, 7), 481, 8, 128),
    # fused proteins (n <= 4) on the general kernel
    _case(pick_rider(4, 320, 2, 1), 640, 2, 80, fused=True),
    _case(pick_rider(4, 320, 2, 2), 320, 3, 80, fused=True),             # four row lanes
    _case(pick_rider(4, 320, 2, 2), 1280, 3, 80, layout='ld', pad=4, fused=True),
    _case(pick_rider(4, 320, 2, 3), 1024, 4, 61, fused=True),
    _case(pick_rider(4, 640, 1, 1), 2560, 2, 80, fused=True),
    _case(pick_rider(4, 640, 1, 2), 2560, 3, 80, fused=True),
    _case(pick_rider(4, 640, 1, 3), 3072, 4, 100, fused=True),           # CT = 2
    _case(pick_rider(1, 640, 1, 1), 1280, 2, 80, layout='shift4', fused=True),
    _case(pick_rider(1, 640, 1, 2), 333, 3, 47, fused=True),
    _case(pick_rider(1, 640, 1, 3), 1000, 4, 128, layout='ld', pad=3, fused=True),
]


def _case_id(c):
    n, m = c['qdim'][:2]
    lay = c['layout'] + (f'{c["pad"]}' if c['layout'] == 'ld' else '')
    return f'{c["target"]}-D{c["D"]}-n{n}m{m}-{lay}-{"fused" if c["fused"] else "plain"}-f{c["flags"]}'


# ---------------------------------------------------------------------------------------------------------------------
# the batch: three proteins, all three synth.KINDS
# ---------------------------------------------------------------------------------------------------------------------
def proteins(n):
    """(seed, L, kind, windowed, domain strings) per protein.  Domain strings depend on n: a domain of exactly n rows
    and one of fewer than 8 rows (row lanes left idle) where n allows it."""
    short = max(n, 6)
    return [
        # fusable: the global domain next to disjoint domains (one discontinuous, unsorted); rows 9.., 17.., 25..29
        # are covered by no other domain and stream as filler items of the global domain
        (7001, 40, 'white', False, [f'1-{n}', f'11-{10 + short}', '30-40,21-24', '1-40']),
        # around the 512-row item split: 511, 512 and 513 rows, and 1025 rows = three items meeting in the workspace
        (7002, 1030, 'esm', False, ['1-511', '2-513', '1-513', '4-1028']),
        # longer than maxlen: four windows, rows of two windows averaged, window cuts inside the domains; fusable, with
        # rows no other domain covers
        (7003, 1234, 'offset', True, ['700-900,100-300', '301-690', '1-1234']),
    ]


@functools.lru_cache(maxsize=2)
def inputs(D):
    """Per protein the list of its sources (maxlen windows), each {15: float32[rows, D], 21: ...}."""
    out = []
    for seed, L, kind, windowed, _ in proteins(3):
        if windowed:
            out.append(cases.stitch_chunks_for(dict(seed=seed, L=L, D=D, maxlen=MAXLEN, kind=kind)))
        else:
            out.append([synth.layers(seed, L, D, kind)])
    return out


def stitched(D):
    """Per protein {layer: float32[L, D]}: what the reference quantizes (embedding.py stitches the windows)."""
    return [{lay: fo.stitch_chunks([w[lay] for w in wins], OVERLAP) for lay in (15, 21)} for wins in inputs(D)]


def geometry(D, n):
    """make_plan arguments (after n_layers, D, n, m) and the domain strings in output-row order."""
    src_rows, prot_src0, prot_nsrc, dom_prot, seg_off, sb, se, names = [], [], [], [], [0], [], [], []
    for p, ((_, L, _, _, doms), wins) in enumerate(zip(proteins(n), inputs(D))):
        prot_src0.append(len(src_rows))
        prot_nsrc.append(len(wins))
        src_rows += [w[15].shape[0] for w in wins]
        for d in doms:
            segs, kept = fo.parse_domain(d, L)
            assert kept == d
            dom_prot.append(p)
            for b, e in segs:
                sb.append(b)
                se.append(e)
            seg_off.append(len(sb))
            names.append((p, d))
    return (src_rows, prot_src0, prot_nsrc, dom_prot, seg_off, sb, se), names


def oracle(D, qdim):
    _, names = geometry(D, qdim[0])
    emb = stitched(D)
    per_prot = {}
    rows = []
    for p, d in names:
        if p not in per_prot:
            per_prot[p], _ = fo.quantize_matrix(emb[p], [dd for pp, dd in names if pp == p], list(qdim))
        rows.append(per_prot[p][d])
    return np.array(rows).astype(int)


def arena(D, layout, pad):
    """Every (layer, source) of the batch in one NaN-filled CUDA buffer, NaN rows between sources.  Returns
    src_tensors[layer][source] as [rows, D] views with stride(0) = ld."""
    ld = D + (pad if layout == 'ld' else 0)
    shift = 1 if layout == 'shift4' else 0
    srcs = [[w[lay] for wins in inputs(D) for w in wins] for lay in (15, 21)]
    offs, pos = [], 0
    for layer in srcs:
        offs.append([])
        for a in layer:
            pos = (pos + GAP_ROWS * ld + 63) // 64 * 64 + shift
            offs[-1].append(pos)
            pos += a.shape[0] * ld
    pos += GAP_ROWS * ld
    host = np.full(pos, np.nan, dtype=np.float32)
    for layer, lo in zip(srcs, offs):
        for a, o in zip(layer, lo):
            host[o:o + a.shape[0] * ld].reshape(a.shape[0], ld)[:, :D] = a
    dev = torch.from_numpy(host).cuda()
    views = [[dev[o:o + a.shape[0] * ld].view(a.shape[0], ld)[:, :D] for a, o in zip(layer, lo)]
             for layer, lo in zip(srcs, offs)]
    if layout == 'shift4':
        assert all(v.data_ptr() % 16 == 4 for layer in views for v in layer)
    elif D % 4 == 0 and ld % 4 == 0:
        assert all(v.data_ptr() % 16 == 0 for layer in views for v in layer)
    assert views[0][0].stride(0) == ld
    return dev, views


# ---------------------------------------------------------------------------------------------------------------------
# kernel names from torch.profiler
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL_RE = re.compile(r'\b(fp_ws_kernel|fp_kernel)\s*<([^<>]*)>')


def canonical(name):
    """'void (anonymous namespace)::fp_kernel<2, 4, 8, 320, 2, 1280, 1, false>(...)' -> 'fp_kernel<2,4,8,320,2,1280,1,0>'."""
    mt = _KERNEL_RE.search(name)
    if not mt:
        return None
    args = [a.strip() for a in mt.group(2).split(',')]
    args = [{'true': '1', 'false': '0'}.get(a, a) for a in args]
    args = [re.sub(r'^\((?:int|bool|unsigned int)\)', '', a).rstrip('uU') for a in args]
    return f'{mt.group(1)}<{",".join(args)}>'


def launched(fn):
    """Runs fn() in a profiler session of its own; returns (its result, the fingerprint kernels launched, in order)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any('fp_table_kernel' in nm for nm in names), \
        f'the profiler recorded no fingerprint kernels at all (CUDA events: {sorted(set(names))[:8]})'
    return res, [c for c in (canonical(nm) for nm in names) if c]


_observed = set()
_stats = {}             # case id -> (instantiation, bytes off by 1, bytes compared)


def _compare(cid, inst, got, want):
    got, want = np.asarray(got).astype(int), np.asarray(want).astype(int)
    assert got.shape == want.shape, (got.shape, want.shape)
    diff = np.abs(got - want)
    _stats[cid] = (inst, int((diff != 0).sum()), int(diff.size))
    bad = np.argwhere(diff > 1)
    assert not len(bad), f'{cid}: {len(bad)} bytes off by more than 1 LSB (max {diff.max()}), first (row, col): {bad[:6].tolist()}'
    assert (diff != 0).mean() <= TOL_CASE, f'{cid}: {(diff != 0).sum()} of {diff.size} bytes differ by 1'


def run_case(c):
    """One case through make_plan / execute_plan; returns the output rows [n_dom, n_layers * n * m] as int."""
    from dctdomain_b200.fingerprint import execute_plan, make_plan
    D, (n, m) = c['D'], c['qdim'][:2]
    geo, names = geometry(D, n)
    plan = make_plan(2, D, n, m, *geo, maxlen=MAXLEN, overlap=OVERLAP, flags=c['flags'])
    _, srcs = arena(D, c['layout'], c['pad'])
    width = 2 * n * m
    outs, kernels = [], None
    for rep in range(2):
        out = torch.full((len(names), width + OUT_PAD), SENTINEL, dtype=torch.int8, device='cuda')
        if rep == 0:
            _, kernels = launched(lambda: execute_plan(plan, srcs, out))
        else:
            execute_plan(plan, srcs, out)
        outs.append(out.cpu().numpy())
    _observed.update(kernels)
    cid = _case_id(c)
    assert kernels == [c['target']], f'{cid}: launched {kernels}'
    assert (outs[0][:, width:] == SENTINEL).all(), f'{cid}: bytes written past n_layers * n * m'
    assert np.array_equal(outs[0], outs[1]), f'{cid}: a second launch gave different bytes'
    return outs[0][:, :width].astype(int)


@pytest.mark.parametrize('case', CASES, ids=[_case_id(c) for c in CASES])
def test_variant_matches_oracle(case):
    got = run_case(case)
    _compare(_case_id(case), case['target'], got, oracle(case['D'], case['qdim']))


# ---------------------------------------------------------------------------------------------------------------------
# user-facing entry points
# ---------------------------------------------------------------------------------------------------------------------
QDIM_MIXED = [3, 44, 3, 100]     # layer 15 on fp_ws_kernel (m = 44), layer 21 on the general kernel (m = 100)


def _fingerprints(D, windowed):
    from dctdomain_b200.fingerprint import Fingerprint
    fps = []
    for (seed, L, _, _, doms), wins, emb in zip(proteins(3), inputs(D), stitched(D)):
        if windowed and len(wins) > 1:
            embed = {lay: [w[lay] for w in wins] for lay in (15, 21)}
        else:
            embed = dict(emb)
        fps.append(Fingerprint(pid=f'p{seed}', seq='A' * L, embed=embed, domains=list(doms), quants={}))
    return fps


def test_quantize_batch_mixed_qdim_launches_both_kernels():
    """One quantize_batch call with two (n, m) groups at D = 1280: the warp-specialised kernel for (3, 44) and the general
    kernel for (3, 100), windows averaged in the kernel, fused proteins in both launches."""
    from dctdomain_b200.fingerprint import quantize_batch
    D = 1280
    fps = _fingerprints(D, windowed=True)
    _, kernels = launched(lambda: quantize_batch(fps, QDIM_MIXED, maxlen=MAXLEN, overlap=OVERLAP))
    _observed.update(kernels)
    assert sorted(kernels) == sorted([ws(1280, True), fk(2, 4, 8, 320, 2, 1280, 1, 1)]), kernels
    got, want = [], []
    for fp, emb, (_, _, _, _, doms) in zip(fps, stitched(D), proteins(3)):
        assert fp.domains == doms
        q, _ = fo.quantize_matrix(emb, list(doms), QDIM_MIXED)
        got += [fp.quants[d] for d in doms]
        want += [q[d] for d in doms]
    _compare('quantize_batch/[3,44,3,100]', 'quantize_batch', np.array(got), np.array(want))


def test_quantize_device_matches_quantize_batch():
    """quantize_device on whole-batch layer tensors (padding rows around every protein, as a padded model output has)
    writes the second (n, m) group through a column-offset view of its output; its bytes equal quantize_batch's."""
    from dctdomain_b200.fingerprint import quantize_batch, quantize_device
    D = 1280
    emb = stitched(D)
    lens = [e[15].shape[0] for e in emb]
    row_start = np.cumsum([0] + [L + 2 for L in lens[:-1]]) + 1          # one padding row before and after each
    layers = []
    for lay in (15, 21):
        t = torch.full((int(row_start[-1]) + lens[-1] + 1, D), float('nan'), device='cuda')
        for r0, e in zip(row_start, emb):
            t[int(r0):int(r0) + e[lay].shape[0]] = torch.from_numpy(e[lay]).cuda()
        layers.append(t)
    doms = [p[4] for p in proteins(3)]
    res = quantize_device(layers, row_start, lens, doms, qdim=QDIM_MIXED)
    fps = quantize_batch(_fingerprints(D, windowed=False), QDIM_MIXED)
    want = np.array([fp.quants[d] for fp in fps for d in fp.domains]).astype(int)
    assert res.names == [d for fp in fps for d in fp.domains]
    assert res.dom_prot.tolist() == [p for p, fp in enumerate(fps) for _ in fp.domains]
    got = res.fingerprints.cpu().numpy().astype(int)
    assert np.array_equal(got, want), np.argwhere(got != want)[:6].tolist()


# ---------------------------------------------------------------------------------------------------------------------
# widths that do not fit in shared memory, and the calls after them
# ---------------------------------------------------------------------------------------------------------------------
def _after_rejection():
    """A normal call on the same thread and stream right after a rejected one must run and match."""
    c = _case(ws(1280, True), 1280, 3, 80, fused=True)
    got = run_case(c)
    _compare(_case_id(c) + '/after-rejection', c['target'], got, oracle(1280, c['qdim']))


def test_width_5120_is_unsupported_and_the_next_call_runs():
    """D = 5120 (ESM-2 15B) at (3, 80): the general kernel would need 234 544 B of dynamic shared memory, more than a
    B200 block may have (232 448 B)."""
    from dctdomain_b200 import _lib
    c = _case(pick_k(4, 640, 1, 2), 5120, 3, 80)
    with pytest.raises(_lib.DctdError) as ei:
        run_case(c)
    assert ei.value.code == _lib.ERR_UNSUPPORTED, str(ei.value)
    _after_rejection()


@pytest.mark.parametrize('D', [5068, 5072])
def test_widths_at_the_shared_memory_limit_run_or_are_unsupported(D):
    """D = 5072 at (3, 80) needs 232 432 B of dynamic shared memory, under the 232 448 B limit, but fp_kernel also has
    176 B of static shared memory: it cannot launch and must be refused as unsupported, not fail as a CUDA error.
    D = 5068 (232 256 B + 176 B) fits.  Either way the next call runs."""
    from dctdomain_b200 import _lib
    c = _case(pick_k(4, 640, 1, 2), D, 3, 80)
    rejected = after = None
    try:
        got = run_case(c)
    except _lib.DctdError as e:
        rejected = e
    else:
        _compare(_case_id(c), c['target'], got, oracle(D, c['qdim']))
    try:
        _after_rejection()
    except Exception as e:          # reported together with the outcome of the call before it
        after = e
    assert (rejected is None or rejected.code == _lib.ERR_UNSUPPORTED) and after is None, \
        f'D = {D}: {rejected!r}; the next call: {after!r}'


# ---------------------------------------------------------------------------------------------------------------------
# coverage of the dispatch table
# ---------------------------------------------------------------------------------------------------------------------
def test_zz_every_release_instantiation_was_launched_and_within_budget():
    table = {}
    for cid, (inst, off, n) in sorted(_stats.items()):
        t = table.setdefault(inst, {'cases': [], 'bytes_off_by_1': 0, 'bytes': 0})
        t['cases'].append(cid)
        t['bytes_off_by_1'] += off
        t['bytes'] += n
    # instantiation -> cases -> bytes off by 1 / bytes compared (shown with pytest -s)
    for inst, t in sorted(table.items()):
        print(f'{inst:40s} cases {len(t["cases"]):2d}  bytes off by 1: {t["bytes_off_by_1"]:4d} / {t["bytes"]:7d}')
        for cid in t['cases']:
            print(f'    {cid}')
    assert _observed, 'no fingerprint kernel was observed: run the whole file'
    missing, extra = sorted(set(REQUIRED) - _observed), sorted(_observed - set(REQUIRED))
    assert not missing and not extra, f'never launched: {missing}; launched but not in the release table: {extra}'
    over = {k: (t['bytes_off_by_1'], t['bytes']) for k, t in table.items() if t['bytes_off_by_1'] > TOL_INST * t['bytes']}
    assert not over, over
