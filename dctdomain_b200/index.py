"""Drop-in for the faiss objects the reference uses on its search path.

Reference call sites:
    index = faiss.IndexFlatL2(d); index.add(fps); faiss.write_index(index, path)   src/database.py:241-243
    index = faiss.read_index(path); index.metric_type = faiss.METRIC_L1            src/query_db.py:75-76
    dm, im = index.search(que_arr, k)                                              src/query_db.py:87
so ``import dctdomain_b200.index as faiss`` keeps those lines unchanged.  The database is held on
the GPU as packed int8 (csrc/l1topk.cu); ``search`` is exhaustive L1 top-k with faiss' result
convention: float32 distances, int64 positions, k smallest by (distance, position) ascending,
(FLT_MAX, -1) padding.

Only the L1 metric is implemented (the reference never searches with anything else: it flips
``metric_type`` to METRIC_L1 right after ``read_index``); ``search`` with another metric raises.
Vectors must be integer valued in [-128, 127] - DCT fingerprints are int8 by construction
(src/database.py:240) - anything else raises instead of being rounded silently.
"""
from __future__ import annotations

import os
import struct

import numpy as np
import torch

from . import _lib
from .fingerprint import _device, _workspace

# faiss MetricType values
METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
METRIC_L1 = 2

FLT_MAX = float(np.finfo(np.float32).max)
_QUERY_BATCH = 8192     # queries per dctd_l1_topk call (bounds the candidate workspace: 64 KB per query)
K_HEAP_MAX = 992        # largest k of dctd_l1_topk / dctd_l1_topk_keys; larger k go to dctd_l1_topk_large
K_MAX = 8192            # largest k of dctd_l1_topk_large


def _as_int8(x, d=None) -> np.ndarray:
    a = np.asarray(x)
    if a.ndim != 2:
        raise ValueError('expected a [n, d] array')
    if d is not None and a.shape[1] != d:
        raise ValueError(f'vector dimension {a.shape[1]} != index dimension {d}')
    if a.dtype == np.int8:
        return np.ascontiguousarray(a)
    r = np.rint(a)
    if a.size and (not np.array_equal(r, a) or r.min() < -128 or r.max() > 127):
        raise ValueError('dctdomain_b200.index stores int8 fingerprints: values must be integers in [-128, 127]')
    return np.ascontiguousarray(r.astype(np.int8))


class IndexFlat:
    """Exhaustive index over int8 vectors resident on one GPU."""

    def __init__(self, d: int, metric: int = METRIC_L2, device=None):
        self.d = int(d)
        self.metric_type = metric
        self.is_trained = True
        self.ntotal = 0
        self._dev = _device(device)
        self._packed = None       # torch.uint8 device buffer in dctd_l1_pack layout
        self._cap = 0

    # -- storage --------------------------------------------------------------------------
    def _reserve(self, n: int):
        if n <= self._cap:
            return
        cap = max(n, int(self._cap * 1.5), 1024)
        nbytes = int(_lib.lib().dctd_l1_packed_bytes(cap, self.d))
        buf = torch.empty(nbytes, dtype=torch.uint8, device=self._dev)
        if self._packed is not None and self.ntotal:
            used = int(_lib.lib().dctd_l1_packed_bytes(self.ntotal, self.d))
            buf[:used].copy_(self._packed[:used])
        self._packed, self._cap = buf, cap

    def add(self, x):
        """Append vectors (faiss IndexFlat.add).  ``x``: [n, d] numpy array or int8 CUDA tensor."""
        if isinstance(x, torch.Tensor) and x.is_cuda:
            if x.dtype != torch.int8 or x.dim() != 2 or x.shape[1] != self.d:
                raise ValueError('CUDA input must be an int8 [n, d] tensor')
            rows = x.contiguous()
        else:
            rows = torch.from_numpy(_as_int8(x, self.d)).to(self._dev)
        n = int(rows.shape[0])
        if n == 0:
            return
        self._reserve(self.ntotal + n)
        with torch.cuda.device(self._dev):
            rc = _lib.lib().dctd_l1_pack(rows.data_ptr(), n, self.d, self.ntotal, self._packed.data_ptr(),
                                         torch.cuda.current_stream(self._dev).cuda_stream)
        _lib.check(rc, 'dctd_l1_pack')
        self.ntotal += n

    def reconstruct_n(self, i0: int = 0, n: int = -1) -> np.ndarray:
        """Stored vectors [i0, i0 + n) as int8 [n, d] (row-major); only the groups that hold them are unpacked."""
        if n < 0:
            n = self.ntotal - i0
        if i0 < 0 or n < 0 or i0 + n > self.ntotal:
            raise ValueError(f'range [{i0}, {i0 + n}) outside the index (ntotal = {self.ntotal})')
        if n == 0:
            return np.empty((0, self.d), dtype=np.int8)
        a = i0 // 32 * 32                                    # first vector of the first group touched
        out = torch.empty((i0 + n - a, self.d), dtype=torch.int8, device=self._dev)
        group_bytes = int(_lib.lib().dctd_l1_packed_bytes(32, self.d))
        with torch.cuda.device(self._dev):
            rc = _lib.lib().dctd_l1_unpack(self._packed.data_ptr() + (a // 32) * group_bytes, i0 + n - a, self.d,
                                           out.data_ptr(), torch.cuda.current_stream(self._dev).cuda_stream)
        _lib.check(rc, 'dctd_l1_unpack')
        return out[i0 - a:].cpu().numpy()

    def reserve(self, n: int):
        """Room for ``n`` vectors in total (avoids regrowing while a large database is added in pieces)."""
        self._reserve(int(n))

    # -- search ---------------------------------------------------------------------------
    def search_device(self, q: torch.Tensor, k: int, id_base: int = 0):
        """int8 CUDA queries [nq, d] -> (float32 [nq, k], int64 [nq, k]) CUDA tensors, stream ordered."""
        self._check_queries(q, k)
        L = _lib.lib()
        q = q.contiguous()
        nq = int(q.shape[0])
        dist = torch.empty((nq, k), dtype=torch.float32, device=self._dev)
        ids = torch.empty((nq, k), dtype=torch.int64, device=self._dev)
        if k > K_HEAP_MAX:
            self._topk_large(q, k, id_base, dist=dist, ids=ids)
            return dist, ids
        packed_ptr = self._packed.data_ptr() if self._packed is not None else 0
        with torch.cuda.device(self._dev):
            stream = torch.cuda.current_stream(self._dev).cuda_stream
            for b in range(0, nq, _QUERY_BATCH):
                e = min(nq, b + _QUERY_BATCH)
                need = int(L.dctd_l1_topk_workspace_bytes(e - b, self.ntotal, self.d, k))
                if need == 0:
                    raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'k={k}, d={self.d} not supported (k <= {K_MAX}, d <= 2048)')
                ws = _workspace(self._dev, need)
                rc = L.dctd_l1_topk(q[b:e].data_ptr(), e - b, packed_ptr, self.ntotal, self.d, k, id_base,
                                    dist[b:e].data_ptr(), ids[b:e].data_ptr(), ws.data_ptr(), ws.numel(), stream)
                _lib.check(rc, 'dctd_l1_topk')
        return dist, ids

    # -- pieces of a sharded search (dctdomain_b200.sharded; C ABI: dctd_l1_bound / dctd_l1_topk_keys) ---------------
    def _check_queries(self, q, k):
        if self.metric_type != METRIC_L1:
            raise NotImplementedError('only METRIC_L1 search is implemented (set index.metric_type = METRIC_L1, '
                                      'as reference src/query_db.py:76 does)')
        if q.dtype != torch.int8 or q.dim() != 2 or q.shape[1] != self.d or not q.is_cuda:
            raise ValueError('queries must be an int8 CUDA tensor [nq, d]')
        if k < 1:
            raise ValueError('k must be >= 1')

    def uses_bound(self, nq: int, n: int, k: int) -> bool:
        """Would a shard of ``n`` vectors honour an external distance bound for this (nq, k)?"""
        return bool(_lib.lib().dctd_l1_uses_bound(nq, n, self.d, k))

    def bound_device(self, q: torch.Tensor, k_local: int, sample_stride: int = 0) -> torch.Tensor:
        """int32 [nq]: upper bound of this shard's k_local-th best distance per query (INT32_MAX = none)."""
        self._check_queries(q, k_local)
        L = _lib.lib()
        q = q.contiguous()
        nq = int(q.shape[0])
        out = torch.empty(nq, dtype=torch.int32, device=self._dev)
        if nq == 0:
            return out
        packed_ptr = self._packed.data_ptr() if self._packed is not None else 0
        with torch.cuda.device(self._dev):
            stream = torch.cuda.current_stream(self._dev).cuda_stream
            for b in range(0, nq, _QUERY_BATCH):
                e = min(nq, b + _QUERY_BATCH)
                need = int(L.dctd_l1_bound_workspace_bytes(e - b, self.ntotal, self.d, k_local, sample_stride))
                if need == 0:
                    raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'k={k_local}, d={self.d} not supported (k <= 992, d <= 2048)')
                ws = _workspace(self._dev, need)
                rc = L.dctd_l1_bound(q[b:e].data_ptr(), e - b, packed_ptr, self.ntotal, self.d, k_local, sample_stride,
                                     out[b:e].data_ptr(), ws.data_ptr(), ws.numel(), stream)
                _lib.check(rc, 'dctd_l1_bound')
        return out

    def search_keys_device(self, q: torch.Tensor, k: int, id_base: int = 0, bound: torch.Tensor = None,
                           heap_only: bool = False) -> torch.Tensor:
        """int64 [nq, k] holding the packed keys (distance << 40 | id_base + position, ascending; -1 = empty slot) of this
        shard's k best among the vectors within ``bound`` (int32 [nq] CUDA tensor; None = no external bound)."""
        self._check_queries(q, k)
        L = _lib.lib()
        q = q.contiguous()
        nq = int(q.shape[0])
        keys = torch.empty((nq, k), dtype=torch.int64, device=self._dev)
        if k > K_HEAP_MAX:
            if bound is not None or heap_only:
                raise ValueError(f'bound and heap_only apply to k <= {K_HEAP_MAX} only')
            self._topk_large(q, k, id_base, keys=keys)
            return keys
        if bound is not None:
            if bound.dtype != torch.int32 or bound.shape != (nq,) or not bound.is_cuda:
                raise ValueError('bound must be an int32 CUDA tensor [nq]')
            bound = bound.contiguous()
        packed_ptr = self._packed.data_ptr() if self._packed is not None else 0
        with torch.cuda.device(self._dev):
            stream = torch.cuda.current_stream(self._dev).cuda_stream
            for b in range(0, nq, _QUERY_BATCH):
                e = min(nq, b + _QUERY_BATCH)
                need = int(L.dctd_l1_topk_workspace_bytes(e - b, self.ntotal, self.d, k))
                if need == 0:
                    raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'k={k}, d={self.d} not supported (k <= {K_MAX}, d <= 2048)')
                ws = _workspace(self._dev, need)
                rc = L.dctd_l1_topk_keys(q[b:e].data_ptr(), e - b, packed_ptr, self.ntotal, self.d, k, id_base,
                                         bound[b:e].data_ptr() if bound is not None else 0, keys[b:e].data_ptr(),
                                         ws.data_ptr(), ws.numel(), _lib.L1_HEAP_ONLY if heap_only else 0, stream)
                _lib.check(rc, 'dctd_l1_topk_keys')
        return keys

    def _topk_large(self, q, k, id_base, dist=None, ids=None, keys=None):
        """k > K_HEAP_MAX: dctd_l1_topk_large (radix selection) into (dist, ids) or keys."""
        if k > K_MAX:
            raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'k={k} not supported (k <= {K_MAX})')
        L = _lib.lib()
        nq = int(q.shape[0])
        packed_ptr = self._packed.data_ptr() if self._packed is not None else 0
        with torch.cuda.device(self._dev):
            stream = torch.cuda.current_stream(self._dev).cuda_stream
            for b in range(0, nq, _QUERY_BATCH):
                e = min(nq, b + _QUERY_BATCH)
                need = int(L.dctd_l1_topk_large_workspace_bytes(e - b, self.ntotal, self.d, k))
                if need == 0:
                    raise _lib.DctdError(_lib.ERR_UNSUPPORTED, f'k={k}, d={self.d} not supported (k <= {K_MAX}, d <= 2048)')
                ws = _workspace(self._dev, need)
                ptr = lambda t: t[b:e].data_ptr() if t is not None else 0   # noqa: E731
                rc = L.dctd_l1_topk_large(q[b:e].data_ptr(), e - b, packed_ptr, self.ntotal, self.d, k, id_base, ptr(dist),
                                          ptr(ids), ptr(keys), ws.data_ptr(), ws.numel(), stream)
                _lib.check(rc, 'dctd_l1_topk_large')

    def search(self, x, k: int):
        """faiss-style ``D, I = index.search(x, k)`` with host arrays."""
        q = torch.from_numpy(_as_int8(x, self.d)).to(self._dev)
        dist, ids = self.search_device(q, int(k))
        return dist.cpu().numpy(), ids.cpu().numpy()


def keys_merge(key_parts: torch.Tensor, want_keys: bool = False):
    """int64 [parts, nq, k] packed keys (each list ascending, -1 = empty) -> faiss' (float32 [nq, k], int64 [nq, k]),
    or the merged keys [nq, k] with ``want_keys`` (CUDA kernel dctd_l1_keys_merge)."""
    parts, nq, k = key_parts.shape
    dev = key_parts.device
    key_parts = key_parts.contiguous()
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        if want_keys:
            out = torch.empty((nq, k), dtype=torch.int64, device=dev)
            rc = _lib.lib().dctd_l1_keys_merge(key_parts.data_ptr(), parts, nq, k, 0, 0, out.data_ptr(), stream)
            _lib.check(rc, 'dctd_l1_keys_merge')
            return out
        out_d = torch.empty((nq, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
        rc = _lib.lib().dctd_l1_keys_merge(key_parts.data_ptr(), parts, nq, k, out_d.data_ptr(), out_i.data_ptr(), 0, stream)
    _lib.check(rc, 'dctd_l1_keys_merge')
    return out_d, out_i


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int, device=None):
        super().__init__(d, METRIC_L2, device)


class IndexFlatL1(IndexFlat):
    def __init__(self, d: int, device=None):
        super().__init__(d, METRIC_L1, device)


# ------------------------------------------------------------------------------------------
# .index files, faiss IndexFlat layout (SURVEY.md Appendix B):
#   fourcc "IxF2" ("IxFI" inner product, "IxFl" any other metric) | d int32 | ntotal int64 | 2 x int64 dummy (1 << 20) |
#   is_trained u8 | metric_type int32 | [metric_arg float32 if metric_type > 1] | n_floats uint64 | float32 data
# ------------------------------------------------------------------------------------------
_FOURCC = {METRIC_L2: b'IxF2', METRIC_INNER_PRODUCT: b'IxFI', METRIC_L1: b'IxFl'}     # IxFl: any other metric (+ metric_arg)


_SIDECAR_MAGIC = b'DCTDI8\x00\x02'
_DIGEST_SPAN = 4 << 20       # bytes hashed at either end of the float payload


def _sidecar_path(path: str) -> str:
    return path + '.i8'


def _payload_digest(f, payload_off: int, payload_bytes: int) -> bytes:
    """Content check of a .index float payload: blake2b over its first and last 4 MB (everything when smaller) and its
    length.  Cheap next to reading the file, and it changes whenever vectors at either end change - together with the
    full-size check this catches a rewritten index; the sidecar is then ignored and the float data is used."""
    import hashlib
    h = hashlib.blake2b(digest_size=16)
    h.update(struct.pack('<q', payload_bytes))
    f.seek(payload_off)
    if payload_bytes <= 2 * _DIGEST_SPAN:
        h.update(f.read(payload_bytes))
    else:
        h.update(f.read(_DIGEST_SPAN))
        f.seek(payload_off + payload_bytes - _DIGEST_SPAN)
        h.update(f.read(_DIGEST_SPAN))
    return h.digest()


def write_index(index: IndexFlat, path: str, sidecar: bool = None):
    """faiss.write_index for a flat index.  The file records the metric the index object carries (the reference builds
    IndexFlatL2 and flips to L1 only in memory, src/query_db.py:76, so its files say L2; an index whose metric_type is
    METRIC_L1 is written the way faiss writes it: fourcc 'IxFl', metric_type 2 and a float metric_arg).

    ``sidecar=True`` also writes ``<path>.i8``: the same vectors as raw int8 (a quarter of the bytes, no float
    round trip on load).  ``read_index`` uses it only if it matches the .index: d, ntotal, file size, mtime and a digest
    of the float payload (see ``_payload_digest``); the faiss-compatible .index stays the source of truth.  Default: off,
    or on with DCTD_INDEX_SIDECAR=1 in the environment (so that the reference's unchanged ``faiss.write_index(index,
    path)`` at src/database.py:243 produces one)."""
    if sidecar is None:
        sidecar = os.environ.get('DCTD_INDEX_SIDECAR') == '1'
    metric = index.metric_type if index.metric_type in _FOURCC else METRIC_L2
    rows = index.reconstruct_n()
    with open(path, 'wb') as f:
        f.write(_FOURCC[metric])
        f.write(struct.pack('<iqqqBi', index.d, index.ntotal, 1 << 20, 1 << 20, 1, metric))
        if metric > 1:
            f.write(struct.pack('<f', 0.0))         # metric_arg (faiss writes it for every metric beyond IP / L2)
        f.write(struct.pack('<Q', index.ntotal * index.d))
        payload_off = f.tell()
        f.write(rows.astype(np.float32).tobytes())
    side = _sidecar_path(path)
    if sidecar:
        with open(path, 'rb') as f:
            digest = _payload_digest(f, payload_off, index.ntotal * index.d * 4)
        with open(side, 'wb') as f:
            f.write(_SIDECAR_MAGIC)
            f.write(struct.pack('<iqq', index.d, index.ntotal, os.path.getsize(path)))
            f.write(digest)
            f.write(np.ascontiguousarray(rows, dtype=np.int8).tobytes())
    elif os.path.exists(side):
        os.remove(side)                     # a stale sidecar must not outlive a rewritten index


def read_index(path: str, device=None) -> IndexFlat:
    """faiss.read_index for a flat index file (written by faiss or by write_index above)."""
    with open(path, 'rb') as f:
        fourcc = f.read(4)
        if fourcc not in (b'IxF2', b'IxFI', b'IxFl'):
            raise ValueError(f'{path}: not a flat faiss index (fourcc {fourcc!r})')
        d, ntotal, _, _, _trained, metric = struct.unpack('<iqqqBi', f.read(4 + 8 * 3 + 1 + 4))
        if metric > 1:
            f.read(4)                       # metric_arg
        (n_floats,) = struct.unpack('<Q', f.read(8))
        if n_floats != ntotal * d:
            raise ValueError(f'{path}: inconsistent header ({n_floats} floats for {ntotal} x {d})')
        payload_off = f.tell()
        data = _read_sidecar(path, d, ntotal, f, payload_off)
        if data is None:
            f.seek(payload_off)
            data = np.frombuffer(f.read(n_floats * 4), dtype='<f4').reshape(ntotal, d)
    index = IndexFlat(d, metric, device)
    index.add(data)
    return index


def _read_sidecar(path: str, d: int, ntotal: int, index_file, payload_off: int):
    """int8 rows of ``<path>.i8`` if that file belongs to this .index (same d, ntotal, .index size AND the digest of the
    .index float payload recorded when the sidecar was written), else None."""
    side = _sidecar_path(path)
    if not os.path.exists(side):
        return None
    with open(side, 'rb') as f:
        if f.read(len(_SIDECAR_MAGIC)) != _SIDECAR_MAGIC:
            return None
        sd, sn, size = struct.unpack('<iqq', f.read(4 + 8 + 8))
        digest = f.read(16)
        if (sd, sn, size) != (d, ntotal, os.path.getsize(path)):
            return None
        if digest != _payload_digest(index_file, payload_off, ntotal * d * 4):
            return None                                                 # same shape, different vectors: stale sidecar
        rows = np.fromfile(f, dtype=np.int8, count=ntotal * d)      # writable: torch.from_numpy takes it as is
    if rows.size != ntotal * d:
        return None
    return rows.reshape(ntotal, d)
