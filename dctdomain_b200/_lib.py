"""ctypes binding of libdctd.so (C ABI: include/dctd.h).

There is deliberately no fallback: if the CUDA library is missing or a call fails, this module
raises.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DCTD_LIB') or os.path.join(_HERE, 'libdctd.so')   # DCTD_LIB: e.g. the instrumented build

OK = 0
ERR_ARG, ERR_CUDA, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_NOMEM = -1, -2, -3, -4, -5
FP_TABLES_RESIDENT = 1
FP_PLAN_NO_FUSION, FP_PLAN_GENERAL_KERNEL, FP_PLAN_LONGEST_FIRST = 1, 2, 4
L1_HEAP_ONLY = 1


class DctdError(RuntimeError):
    def __init__(self, code: int, what: str):
        self.code = code
        super().__init__(what)


class FpGeometry(C.Structure):
    _fields_ = [
        ('n_layers', C.c_int32), ('D', C.c_int32), ('n', C.c_int32), ('m', C.c_int32),
        ('maxlen', C.c_int32), ('overlap', C.c_int32),
        ('n_src', C.c_int32), ('src_rows', C.c_void_p),
        ('n_prot', C.c_int32), ('prot_src0', C.c_void_p), ('prot_nsrc', C.c_void_p),
        ('n_dom', C.c_int32), ('dom_prot', C.c_void_p), ('dom_seg_off', C.c_void_p),
        ('seg_beg', C.c_void_p), ('seg_end', C.c_void_p),
    ]


_lib = None


def build(verbose: bool = False) -> str:
    """Compile libdctd.so in-tree with nvcc for sm_100a (dctdomain_b200/csrc/Makefile)."""
    import subprocess
    out = None if verbose else subprocess.DEVNULL
    subprocess.run(['make', '-C', os.path.join(_HERE, 'csrc'), '-j4'], check=True, stdout=out)
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DctdError(ERR_ARG, f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; '
                                 f'g.build()"` (nvcc, sm_100a). There is no CPU fallback.')
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, sz, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t, C.c_uint32
    sig = {
        'dctd_version': (C.c_int, []),
        'dctd_strerror': (C.c_char_p, [C.c_int]),
        'dctd_last_cuda_error': (C.c_int, []),
        'dctd_last_cuda_error_string': (C.c_char_p, []),
        'dctd_launch_count': (i64, [C.c_int]),
        'dctd_h2d_rows': (C.c_int, [vp, vp, i64, vp, vp, vp]),
        'dctd_h2d_gather': (C.c_int, [vp, i64, vp]),
        'dctd_h2d_rows_staged': (C.c_int, [vp, vp, i64, vp, vp, vp, i64, C.c_int32, C.c_int32, vp]),
        'dctd_parse_domains': (C.c_int, [vp, i64, i32, vp, vp, i32, vp, vp, vp, vp, i64, C.POINTER(i32), C.POINTER(i32)]),
        'dctd_fp_plan_create': (C.c_int, [C.POINTER(FpGeometry), C.POINTER(vp)]),
        'dctd_fp_plan_create_ex': (C.c_int, [C.POINTER(FpGeometry), u32, C.POINTER(vp)]),
        'dctd_fp_plan_destroy': (None, [vp]),
        'dctd_fp_workspace_bytes': (sz, [vp]),
        'dctd_fp_algorithmic_bytes': (i64, [vp]),
        'dctd_fp_num_items': (i32, [vp]),
        'dctd_fp_execute': (C.c_int, [vp, vp, i64, vp, i64, vp, sz, u32, vp]),
        'dctd_fp_set_variant': (C.c_int, [C.c_int]),
        'dctd_fp_timing_read': (C.c_int, [vp, vp, vp]),
        'dctd_fp_plan_dump': (C.c_int, [vp, vp, i64, vp, i64, C.POINTER(i64), C.POINTER(i64)]),
        'dctd_fp_plan_dump_records': (C.c_int, [vp, vp, i64]),
        'dctd_scale_f64': (C.c_int, [vp, i64, vp, vp]),
        'dctd_idct_quant_f64': (C.c_int, [vp, i32, i32, i32, vp, vp]),
        'dctd_l1_packed_bytes': (sz, [i64, i32]),
        'dctd_l1_set_mode': (C.c_int, [C.c_int]),
        'dctd_l1_stream_stamps': (C.c_int, [vp, i64, i64, i32, i32, vp]),
        'dctd_l1_pack': (C.c_int, [vp, i64, i32, i64, vp, vp]),
        'dctd_l1_unpack': (C.c_int, [vp, i64, i32, vp, vp]),
        'dctd_l1_topk_workspace_bytes': (sz, [i64, i64, i32, i32]),
        'dctd_l1_topk': (C.c_int, [vp, i64, vp, i64, i32, i32, i64, vp, vp, vp, sz, vp]),
        'dctd_l1_topk_merge': (C.c_int, [vp, vp, i32, i64, i32, vp, vp, vp]),
        'dctd_l1_bound_workspace_bytes': (sz, [i64, i64, i32, i32, i32]),
        'dctd_l1_bound': (C.c_int, [vp, i64, vp, i64, i32, i32, i32, vp, vp, sz, vp]),
        'dctd_l1_uses_bound': (C.c_int, [i64, i64, i32, i32]),
        'dctd_l1_topk_keys': (C.c_int, [vp, i64, vp, i64, i32, i32, i64, vp, vp, vp, sz, u32, vp]),
        'dctd_l1_keys_merge': (C.c_int, [vp, i32, i64, i32, vp, vp, vp, vp]),
        'dctd_l1_topk_large_workspace_bytes': (sz, [i64, i64, i32, i32]),
        'dctd_l1_topk_large': (C.c_int, [vp, i64, vp, i64, i32, i32, i64, vp, vp, vp, vp, sz, vp]),
        'dctd_l1_pair_scores': (C.c_int, [vp, i32, vp, vp, vp, i64, vp, vp, vp]),
        'dctd_l1_protein_scores_workspace_bytes': (sz, [i64, i64, i64, i64, i32]),
        'dctd_l1_protein_scores': (C.c_int, [vp, vp, i64, vp, vp, i64, i32, vp, vp, vp, sz, vp]),
        'dctd_l1_protein_hits_workspace_bytes': (sz, [i64, i64, i64, i64, i32, i32, i32]),
        'dctd_l1_protein_hits': (C.c_int, [vp, vp, i64, vp, vp, i64, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, sz,
                                           vp]),
    }
    hooks = {'dctd_fp_set_variant', 'dctd_fp_timing_read', 'dctd_l1_set_mode', 'dctd_l1_stream_stamps'}   # tuning builds only
    for name, (res, args) in sig.items():
        try:
            fn = getattr(L, name)      # AttributeError here = header / library mismatch
        except AttributeError:
            if name in hooks or os.environ.get('DCTD_LIB_LAX') == '1':   # tuning hooks are not part of the ABI; LAX: A/B runs against older builds
                continue
            raise
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(code: int, what: str = ''):
    if code == OK:
        return
    L = lib()
    msg = L.dctd_strerror(code).decode()
    if code == ERR_CUDA:
        msg += ': ' + L.dctd_last_cuda_error_string().decode()
    err = DctdError(code, f'{what}: {msg}' if what else msg)
    if code == ERR_ARG:
        raise ValueError(str(err)) from err
    raise err


def exported_symbols():
    """Names declared in include/dctd.h (used by the CPU test that checks the .so exports them)."""
    import re
    hdr = os.path.join(os.path.dirname(_HERE), 'include', 'dctd.h')
    text = open(hdr).read()
    return sorted(set(re.findall(r'\b(dctd_[a-z0-9_]+)\s*\(', text)))
