"""Drop-in for reference ``src/dct-sim.py``: same functions, flags and output text; the L1
distances come from the GPU - listed pairs through dctd_l1_pair_scores, the hits of ``--db`` through
dctd_l1_protein_hits (a search of each query's global fingerprint against the database's, then the min over fingerprint
pairs of the selected hits only), all-vs-all through dctd_l1_protein_scores (the tiled SAD kernel of the search path) -
the float64 similarity formula ``1 - min(d / 17000, 1)`` (dct-sim.py:23-26) is applied on the host exactly as the
reference does.

    python -m dctdomain_b200.dct_sim --dct x-dct.npz --pair x.pair --output x-dctsim.txt
"""
from __future__ import annotations

import argparse
import time

import numpy as np
import torch

from . import _lib
from .fingerprint import _device


def _pair_dists(fps: np.ndarray, off: np.ndarray, pa: np.ndarray, pb: np.ndarray):
    """(min over fingerprint pairs, last-vs-last) int L1 distances for protein pairs (pa[i], pb[i]); INT32_MAX for both
    where either protein has no fingerprints."""
    dev = _device()
    fps = _as_int8(fps)
    n = len(pa)
    mn = torch.empty(n, dtype=torch.int32, device=dev)
    last = torch.empty(n, dtype=torch.int32, device=dev)
    if n:
        d_f = torch.from_numpy(fps).to(dev)
        d_off = torch.from_numpy(np.ascontiguousarray(off, dtype=np.int64)).to(dev)
        d_a = torch.from_numpy(np.ascontiguousarray(pa, dtype=np.int32)).to(dev)
        d_b = torch.from_numpy(np.ascontiguousarray(pb, dtype=np.int32)).to(dev)
        with torch.cuda.device(dev):
            rc = _lib.lib().dctd_l1_pair_scores(d_f.data_ptr(), fps.shape[1], d_off.data_ptr(), d_a.data_ptr(),
                                                d_b.data_ptr(), n, mn.data_ptr(), last.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, 'dctd_l1_pair_scores')
    return mn.cpu().numpy().astype(np.int64), last.cpu().numpy().astype(np.int64)


def _as_int8(fps: np.ndarray) -> np.ndarray:
    fps = np.ascontiguousarray(fps)
    if fps.dtype != np.int8:
        if fps.size and (fps.min() < -128 or fps.max() > 127 or not np.array_equal(np.rint(fps), fps)):
            raise ValueError('fingerprints must be int8 valued')
        fps = fps.astype(np.int8)
    return fps


def protein_scores(q_fps, q_off, db_fps, db_off, workspace_bytes: int = None):
    """(min over fingerprint pairs, last-vs-last) int L1 distances for ALL pairs of two protein sets: int64 arrays
    [n_q, n_db] (dctd_l1_protein_scores: the tiled SAD kernel of the search path + a per-pair reduction on the device).
    ``q_fps`` / ``db_fps``: int8-valued [n, d] arrays, or CUDA int8 tensors; protein i owns rows off[i] .. off[i+1]-1."""
    dev = _device()
    L = _lib.lib()
    q_off = np.ascontiguousarray(q_off, dtype=np.int64)
    db_off = np.ascontiguousarray(db_off, dtype=np.int64)
    nq, nd = len(q_off) - 1, len(db_off) - 1
    d_q = q_fps if isinstance(q_fps, torch.Tensor) else torch.from_numpy(_as_int8(q_fps)).to(dev)
    d_db = db_fps if isinstance(db_fps, torch.Tensor) else torch.from_numpy(_as_int8(db_fps)).to(dev)
    d = int(d_q.shape[1]) if d_q.dim() == 2 and d_q.shape[0] else int(d_db.shape[1])
    mn = torch.empty((nq, nd), dtype=torch.int32, device=dev)
    last = torch.empty((nq, nd), dtype=torch.int32, device=dev)
    if nq and nd:
        n_dbf = int(d_db.shape[0])
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            packed = torch.empty(max(int(L.dctd_l1_packed_bytes(n_dbf, d)), 16), dtype=torch.uint8, device=dev)
            if n_dbf:
                _lib.check(L.dctd_l1_pack(d_db.contiguous().data_ptr(), n_dbf, d, 0, packed.data_ptr(), stream), 'dctd_l1_pack')
            need = workspace_bytes or int(L.dctd_l1_protein_scores_workspace_bytes(int(d_q.shape[0]), nq, n_dbf, nd, d))
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            rc = L.dctd_l1_protein_scores(d_q.contiguous().data_ptr(), q_off.ctypes.data, nq, packed.data_ptr(),
                                          db_off.ctypes.data, nd, d, mn.data_ptr(), last.data_ptr(), ws.data_ptr(),
                                          ws.numel(), stream)
        if rc == _lib.ERR_UNSUPPORTED:        # vectors too wide for the tiled kernel: one warp per protein pair
            cat = torch.cat([d_q, d_db]).cpu().numpy()
            off = np.concatenate([q_off, db_off[1:] + q_off[-1]])
            a, b = np.divmod(np.arange(nq * nd, dtype=np.int64), nd)
            m1, l1 = _pair_dists(cat, off, a.astype(np.int32), (b + nq).astype(np.int32))
            return m1.reshape(nq, nd), l1.reshape(nq, nd)
        _lib.check(rc, 'dctd_l1_protein_scores')
    return mn.cpu().numpy().astype(np.int64), last.cpu().numpy().astype(np.int64)


DIST_CLAMP = 17000                 # s(x) = 1 - min(x / 17000, 1) is 0 for every x >= 17000
HITS_MAX_CAP = 992                 # longest hit row dctd_l1_protein_hits fills


def _dist_cut(threshold: float) -> int:
    """The largest distance x whose similarity passes dct-sim's threshold (s(x) >= threshold), found by evaluating the
    float64 expression itself over 0 .. 17000 (it is strictly decreasing there).  -1: nothing passes; DIST_CLAMP: every
    database protein passes, those without fingerprints included (threshold <= 0, or NaN: ``s < nan`` never ends
    dct-sim's loop)."""
    threshold = float(threshold)
    if threshold != threshold:
        return DIST_CLAMP
    x = np.arange(DIST_CLAMP + 1, dtype=np.int64)
    ok = np.nonzero(1.0 - np.minimum(x / 17000, 1.0) >= threshold)[0]
    return int(ok[-1]) if len(ok) else -1


def protein_hits(q_fps, q_off, db_fps, db_off, top: int, threshold: float, cap: int = None,
                 workspace_bytes: int = None):
    """dct-sim's database-search hits (src/dct-sim.py:126-156) without the all-pairs matrices: for query protein a, the
    database proteins ranked by the similarity of the two proteins' last (global) fingerprints - ascending by
    (min(last, 17000), b) - cut after max(top, #{b : s(last) >= threshold}) entries, exactly the rows dct-sim prints.
    Returns CSR int arrays (hit_off [n_q + 1], hit_db, hit_min, hit_last): hits of query a are
    hit_off[a] .. hit_off[a+1]-1 in output order, with the min over all fingerprint pairs and the last-vs-last distance
    (INT32_MAX where a protein has no fingerprints).

    One dctd_l1_protein_hits call with rows of ``cap`` hits (default max(top, 32)); queries with more hits than that are
    rerun once with cap = their largest count.  Raises DctdError(ERR_UNSUPPORTED) where the device path cannot give the
    rows: vectors too wide for its tiles, or more than HITS_MAX_CAP hits for one query."""
    dev = _device()
    L = _lib.lib()
    q_off = np.ascontiguousarray(q_off, dtype=np.int64)
    db_off = np.ascontiguousarray(db_off, dtype=np.int64)
    nq, nd = len(q_off) - 1, len(db_off) - 1
    d_q = q_fps if isinstance(q_fps, torch.Tensor) else torch.from_numpy(_as_int8(q_fps)).to(dev)
    d_db = db_fps if isinstance(db_fps, torch.Tensor) else torch.from_numpy(_as_int8(db_fps)).to(dev)
    d_q, d_db = d_q.contiguous(), d_db.contiguous()
    d = int(d_q.shape[1]) if d_q.dim() == 2 and d_q.shape[0] else int(d_db.shape[1])
    top_ = min(max(int(top), 0), nd)
    cut = _dist_cut(threshold)
    if cap is None:
        cap = max(top_, 32)
    if cap > HITS_MAX_CAP:
        raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'protein_hits: {cap} hits per query (at most {HITS_MAX_CAP})')

    def run(q, qoff, cap):
        n = len(qoff) - 1
        count = torch.empty(n, dtype=torch.int32, device=dev)
        rows = torch.empty((3, n, cap), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            need = workspace_bytes or int(L.dctd_l1_protein_hits_workspace_bytes(int(q.shape[0]), n, int(d_db.shape[0]),
                                                                                 nd, d, top_, cap))
            ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
            rc = L.dctd_l1_protein_hits(q.data_ptr(), qoff.ctypes.data, n, d_db.data_ptr(), db_off.ctypes.data, nd, d,
                                        top_, DIST_CLAMP, cut, cap, count.data_ptr(), rows[0].data_ptr(),
                                        rows[1].data_ptr(), rows[2].data_ptr(), ws.data_ptr(), ws.numel(), stream)
        _lib.check(rc, 'dctd_l1_protein_hits')
        return count.cpu().numpy().astype(np.int64), rows.cpu().numpy()

    def scatter(out, off, count, rows, sel):
        """rows of the queries `sel` -> their CSR slots"""
        width = rows.shape[2]
        m = np.arange(width)[None, :] < count[sel][:, None]
        pos = (off[:-1][sel][:, None] + np.arange(width)[None, :])[m]
        for o, r in zip(out, rows[:, sel]):
            o[pos] = r[m]

    if nq == 0:
        count, rows = np.zeros(0, dtype=np.int64), np.zeros((3, 0, cap), dtype=np.int32)
    else:
        count, rows = run(d_q, q_off, cap)
    off = np.concatenate([[0], np.cumsum(count)]).astype(np.int64)
    out = [np.empty(int(off[-1]), dtype=np.int64) for _ in range(3)]
    scatter(out, off, count, rows, count <= cap)
    over = np.nonzero(count > cap)[0]
    if len(over):                          # longer hit lists: one more call for those queries only
        cap2 = int(count[over].max())
        if cap2 > HITS_MAX_CAP:
            raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'protein_hits: {cap2} hits for one query (at most {HITS_MAX_CAP})')
        lens = q_off[over + 1] - q_off[over]
        sub_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        idx = np.concatenate([np.arange(q_off[a], q_off[a + 1]) for a in over]).astype(np.int64)
        sub_q = d_q[torch.from_numpy(idx).to(dev)] if len(idx) else d_q[:0]
        count2, rows2 = run(sub_q.contiguous(), sub_off, cap2)
        full = np.zeros(nq, dtype=bool)
        full[over] = True
        rows_full = np.zeros((3, nq, cap2), dtype=np.int32)
        rows_full[:, over] = rows2
        count_full = count.copy()
        count_full[over] = count2
        scatter(out, off, count_full, rows_full, full)
    return off, out[0], out[1], out[2]


def _sim(dist):
    """dct-sim.py:23-26 in float64."""
    d = np.int64(dist)
    d = d / 17000
    d = min(d, 1)
    return 1 - d


def prostSimilarity(emb1: np.ndarray, emb2: np.ndarray) -> float:   # noqa: N802 (reference name)
    """Similarity of two fingerprints (reference src/dct-sim.py:12-26)."""
    fps = np.stack([np.asarray(emb1), np.asarray(emb2)])
    mn, _ = _pair_dists(fps, np.array([0, 1, 2]), np.array([0]), np.array([1]))
    return _sim(mn[0])


def _maxs_s(mn, last):
    s = _sim(last)
    best = _sim(mn)
    return (best if best > 0 else 0), s      # the reference's running max starts at int 0


def domain_sim(dct_i: np.ndarray, dct_j: np.ndarray) -> tuple:
    """(max similarity over all fingerprint pairs, similarity of the two last = global fingerprints)
    (reference src/dct-sim.py:28-50)."""
    ni = dct_i.shape[0]
    fps = np.concatenate([dct_i, dct_j])
    mn, last = _pair_dists(fps, np.array([0, ni, len(fps)]), np.array([0]), np.array([1]))
    return _maxs_s(mn[0], last[0])


def load_dct(filename: str, asmap=True) -> tuple:
    """reference src/dct-sim.py:52-84."""
    start = time.time()
    data = np.load(filename)
    seqid, domidx, dct_all = data['sid'], data['idx'], data['dct']
    dct = {} if asmap else []
    for i in range(len(seqid)):
        block = dct_all[domidx[i]:domidx[i + 1], :]
        if asmap:
            dct[seqid[i]] = block
        else:
            dct.append(block)
    print(f"dct loaded for {len(seqid)} sequences, time used: {time.time() - start:.1f}s")
    return (dct, seqid)


def _emit(line, output):
    if output:
        with open(output, 'a', encoding='utf8') as out:
            out.write(line + '\n')
    else:
        print(line)


def _blocks(dcts):
    """list of [n_i, d] blocks -> (concatenated, offsets)."""
    off = np.concatenate([[0], np.cumsum([b.shape[0] for b in dcts])]).astype(np.int64)
    cat = np.concatenate(dcts) if dcts else np.zeros((0, 480), dtype=np.int8)
    return cat, off


def pair_sim(npzfile: str, pairfile: str, pairfound: str, output: str):
    """reference src/dct-sim.py:86-124; all listed pairs are scored in one kernel launch."""
    dct, _ = load_dct(npzfile, asmap=True)
    names = list(dct.keys())
    slot = {s: i for i, s in enumerate(names)}
    cat, off = _blocks([dct[s] for s in names])
    tot, rows = 0, []
    with open(pairfile, 'r', encoding='utf8') as inf:
        lines = inf.readlines()
    kept = []
    for aline in lines:
        if aline[0] == '#':
            kept.append(aline)
            continue
        subs = aline.split()
        s1, s2 = subs[0], subs[1]
        tot += 1
        if (s1 in slot) and (s2 in slot):
            rows.append((s1, s2))
            kept.append(aline)
    mn, last = _pair_dists(cat, off, np.array([slot[a] for a, _ in rows], dtype=np.int32),
                           np.array([slot[b] for _, b in rows], dtype=np.int32))
    for (s1, s2), a, b in zip(rows, mn, last):
        maxs, s = _maxs_s(a, b)
        _emit(f"{s1} {s2} {maxs} {s}", output)
    print(f"total pair {pairfile} found {len(rows)} (not found: {tot - len(rows)})")
    if pairfound:
        with open(pairfound, 'w', encoding='utf8') as out2:
            out2.writelines(kept)
        print(f"pairs saved to file {pairfound}")


def db_search(npzfile: str, dbfile: str, top: int, threshold: float, output: str):
    """reference src/dct-sim.py:126-156."""
    dct, seqid = load_dct(npzfile, asmap=False)
    db_dct, db_seqid = load_dct(dbfile, asmap=False)
    nq, nd = len(seqid), len(db_seqid)
    qcat, qoff = _blocks(list(dct))
    dcat, doff = _blocks(list(db_dct))
    try:
        off, hit_db, hit_min, hit_last = protein_hits(qcat, qoff, dcat, doff, top, threshold)
    except _lib.DctdError as e:
        if e.code != _lib.ERR_UNSUPPORTED:
            raise
    else:
        for i in range(nq):
            for j in range(off[i], off[i + 1]):
                maxs, s = _maxs_s(hit_min[j], hit_last[j])
                _emit(f"{seqid[i]} {db_seqid[hit_db[j]]} {maxs} {s}", output)
        return
    # wide fingerprints or very long hit lists: score all pairs
    mn, last = protein_scores(qcat, qoff, dcat, doff)            # all pairs: one tiled pass on the device
    # the reference sorts every query's hits by the global similarity, descending and stable (sorted(..., reverse=True)
    # keeps the database order among equal keys), and prints until rank >= top and s < threshold
    s_all = 1.0 - np.minimum(last / 17000, 1.0)                   # float64, the values _sim() produces
    order = np.argsort(-s_all, axis=1, kind='stable')
    for i in range(nq):
        for rank in range(nd):
            q = int(order[i, rank])
            if (rank >= top) and (s_all[i, q] < threshold):
                break
            maxs, s = _maxs_s(mn[i, q], last[i, q])               # exactly the reference's scalar arithmetic and types
            _emit(f"{seqid[i]} {db_seqid[q]} {maxs} {s}", output)


def all_sim(npzfile: str, output: str):
    """reference src/dct-sim.py:158-176."""
    dct, seqid = load_dct(npzfile, asmap=False)
    n = len(seqid)
    cat, off = _blocks(list(dct))
    mn, last = protein_scores(cat, off, cat, off)                 # the set against itself; the upper triangle is printed
    for i in range(n - 1):
        for j in range(i + 1, n):
            maxs, s = _maxs_s(mn[i, j], last[i, j])
            _emit(f"{seqid[i]} {seqid[j]} {maxs:.3f} {s:.3f}", output)


def main(argv=None):
    start = time.time()
    parser = argparse.ArgumentParser()
    parser.add_argument("--dct", help="dct in a npz file", required=True)
    parser.add_argument("--output", help="save results to a file", required=False)
    parser.add_argument("--pair", help="calculate distance between the proteins in the given file", required=False)
    parser.add_argument("--pairfound", help="pairs of proteins with similarity computed", required=False)
    parser.add_argument("--db", help="search query dct against this db", required=False)
    parser.add_argument("--top", help="report at most this many hits for database search", default=5, type=int)
    parser.add_argument("--threshold", help="similarity threshold for reporting hits for database search",
                        default=0.25, type=float)
    args = parser.parse_args(argv)

    header = "#prot1 prot2 sim-domain sim-global"
    if args.output:
        with open(args.output, "w", encoding='utf8') as out:
            out.write(header + "\n")
    else:
        print(header)
    nowt = time.time()
    if args.pair:
        pair_sim(args.dct, args.pair, args.pairfound, args.output)
    elif args.db:
        db_search(args.dct, args.db, args.top, args.threshold, args.output)
    else:
        all_sim(args.dct, args.output)
    if args.output:
        print("results saved to", args.output)
    end = time.time()
    print(f"total time used {end - start:.1f}s")
    print(f"distance calculation used {end - nowt:.1f}s")


if __name__ == '__main__':
    main()
