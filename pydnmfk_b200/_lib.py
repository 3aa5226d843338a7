"""ctypes binding of libdnmf.so (include/dnmf.h).

The product path has NO CPU fallback: if the shared library is missing the
import fails loudly, and every kernel call raises :class:`DnmfError` on a
non-zero status.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DNMF_LIB_PATH') or os.path.join(_HERE, 'libdnmf.so')   # override: A/B builds only

F32, F64, I64 = 0, 1, 2
A_F16, A_BF16 = 3, 4          # data shard stored in fp16 / bf16; factors and results fp32 (include/dnmf.h)
MATH_ACCURATE, MATH_TF32 = 0, 1
E_UNSUPPORTED = -2
OP_AH, OP_WTA, OP_KL_UHT, OP_KL_WTU, OP_GRAM, OP_RESIDUAL, OP_SUMS, OP_NNZ, OP_AH_RESIDUAL = range(9)
MAX_K = 64

i64, i32, dbl, vp = C.c_int64, C.c_int, C.c_double, C.c_void_p

# name -> (restype, argtypes); mirrors include/dnmf.h one to one
SIGNATURES = {
    'dnmf_version': (C.c_char_p, []),
    'dnmf_last_error': (C.c_char_p, []),
    'dnmf_last_path': (i32, []),
    'dnmf_launch_count': (i64, [i32]),
    'dnmf_pass_count': (i64, [i32, i32]),
    'dnmf_device_info': (i32, [C.POINTER(i32)] * 3),
    'dnmf_set_force_generic': (i32, [i32]),
    'dnmf_set_tc_min_elems': (i32, [i64]),
    'dnmf_set_tc_profile': (i32, [vp]),
    'dnmf_set_tc_debug': (i32, [i32]),
    'dnmf_set_tc_residual': (i32, [i32]),
    'dnmf_workspace_bytes': (i64, [i32, i64, i64, i64, i32]),
    'dnmf_ah': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, i32, i32, vp, i64, vp]),
    'dnmf_wta': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, i32, i32, i32, vp, i64, vp]),
    'dnmf_kl_uht': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i64, i64, i64, dbl, i32, i32, vp, i64, vp]),
    'dnmf_kl_wtu': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i64, i64, i64, dbl, i32, i32, i32, vp, i64, vp]),
    'dnmf_gram': (i32, [vp, i64, i64, i64, i32, vp, i32, vp, i64, vp]),
    'dnmf_mu_update_w': (i32, [vp, i64, vp, i64, vp, i64, i64, dbl, i32, vp]),
    'dnmf_mu_update_h': (i32, [vp, i64, vp, i64, i64, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_kl_update_w': (i32, [vp, i64, vp, i64, vp, i64, i64, dbl, i32, vp]),
    'dnmf_kl_update_h': (i32, [vp, i64, vp, i64, i64, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_clamp_min': (i32, [vp, i64, i64, i64, dbl, i32, vp]),
    'dnmf_colsum': (i32, [vp, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_rowsum': (i32, [vp, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_sqnorm': (i32, [vp, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_normalize': (i32, [vp, i64, i64, vp, i64, i64, i64, vp, dbl, i32, vp]),
    'dnmf_ah_p': (i32, [vp, i64, vp, i64, i64, i64, i64, i32, i32, vp, i64, vp, vp]),
    'dnmf_wta_p': (i32, [vp, i64, vp, i64, i64, i64, i64, i32, i32, vp, i64, vp, vp]),
    'dnmf_kl_uht_p': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, dbl, i32, i32, vp, i64, vp, vp]),
    'dnmf_kl_wtu_p': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, dbl, i32, i32, vp, i64, vp, vp]),
    'dnmf_mu_update_w_p': (i32, [vp, i64, vp, vp, i64, i64, dbl, i32, vp]),
    'dnmf_mu_update_h_p': (i32, [vp, i64, vp, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_kl_update_w_p': (i32, [vp, i64, vp, vp, i64, i64, dbl, i32, vp]),
    'dnmf_kl_update_h_p': (i32, [vp, i64, vp, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_trace_terms_workspace_bytes': (i64, []),
    'dnmf_trace_terms': (i32, [vp, i64, vp, i64, i64, vp, vp, i64, vp, vp, i64, i32, vp, i64, vp]),
    'dnmf_residual_sqnorm': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_ah_residual': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_column_err': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, vp, vp, i32, vp]),
    'dnmf_hals_w_col': (i32, [vp, i64, vp, i64, vp, i64, i64, i64, dbl, vp, i32, vp, i64, vp]),
    'dnmf_div_col': (i32, [vp, i64, i64, i64, vp, i32, vp]),
    'dnmf_hals_h': (i32, [vp, i64, vp, i64, i64, vp, i64, i64, dbl, i32, vp]),
    'dnmf_bcd_pg_w': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i64, dbl, i32, vp]),
    'dnmf_bcd_pg_h': (i32, [vp, i64, vp, i64, vp, i64, i64, vp, i64, i64, dbl, i32, vp]),
    'dnmf_bcd_pg_w_dev': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i64, vp, i32, vp]),
    'dnmf_bcd_pg_h_dev': (i32, [vp, i64, vp, i64, vp, i64, i64, vp, i64, i64, vp, i32, vp]),
    'dnmf_bcd_state': (i32, [i32, vp, vp, vp]),
    'dnmf_bcd_advance': (i32, [vp, vp, vp, i64, vp, i32, i32, vp]),
    'dnmf_bcd_keep': (i32, [vp, vp, i64, vp, i32, vp]),
    'dnmf_div_cols': (i32, [vp, i64, i64, i64, vp, i32, vp]),
    'dnmf_axpby': (i32, [vp, vp, vp, dbl, dbl, i64, i32, vp]),
    'dnmf_nnz_counts': (i32, [vp, i64, i64, i64, vp, vp, i32, vp]),
    'dnmf_compact': (i32, [vp, i64, vp, i64, vp, i64, vp, i64, i32, vp]),
    'dnmf_scatter_rows': (i32, [vp, i64, vp, i64, i64, vp, i64, i32, vp]),
    'dnmf_scatter_cols': (i32, [vp, i64, vp, i64, i64, vp, i64, i32, vp]),
    'dnmf_perturb_uniform': (i32, [vp, vp, vp, i64, dbl, i32, vp]),
    # NMFk-level rows
    'dnmf_colsumsq': (i32, [vp, i64, i64, i64, vp, i32, vp, i64, vp]),
    'dnmf_colsum_workspace_bytes': (i64, [i64, i64]),
    'dnmf_scale_groups': (i32, [vp, i64, i64, i64, vp, i64, i64, i64, i32, dbl, i32, vp]),
    'dnmf_greedy_lsa': (i32, [vp, i64, i64, i64, vp, i32, vp]),
    'dnmf_permute_groups': (i32, [vp, vp, i64, i64, i64, i32, vp, i32, i32, vp]),
    'dnmf_median_last': (i32, [vp, i64, i64, vp, vp, i32, vp]),
    'dnmf_silhouettes': (i32, [vp, i64, i64, i64, vp, i32, vp]),
    'dnmf_rank1_sub': (i32, [vp, i64, i64, i64, vp, vp, vp, i32, vp]),
    'dnmf_matvec_workspace_bytes': (i64, [i64, i64, i32]),
    'dnmf_matvec_f64': (i32, [vp, i64, i64, i64, vp, vp, i32, i32, vp, i64, vp]),
    'dnmf_power_normalize': (i32, [vp, vp, vp, vp, i64, vp]),
    'dnmf_power_iterate': (i32, [vp, i64, i64, vp, dbl, i32, i32, vp, vp, i32, vp]),
    'dnmf_div_store': (i32, [vp, vp, vp, i64, i64, vp]),
    'dnmf_posneg_colsumsq': (i32, [vp, i64, i64, i64, vp, vp]),
    'dnmf_nnsvd_pick': (i32, [vp, i64, i64, i64, vp, vp, vp, i64, i32, vp]),
    # communicators (NCCL owned by the library), peer-mapped memory, fused half-step exchange
    'dnmf_comm_load': (i32, [C.c_char_p]),
    'dnmf_comm_nccl_version': (i32, [C.POINTER(i32)]),
    'dnmf_comm_unique_id': (i32, [vp]),
    'dnmf_comm_init_rank': (i32, [vp, i32, i32, C.POINTER(vp)]),
    'dnmf_comm_split': (i32, [vp, i32, i32, C.POINTER(vp)]),
    'dnmf_comm_rank': (i32, [vp, C.POINTER(i32), C.POINTER(i32)]),
    'dnmf_comm_destroy': (i32, [vp]),
    'dnmf_allreduce': (i32, [vp, vp, i64, i32, vp]),
    'dnmf_allgather': (i32, [vp, vp, vp, i64, i32, vp]),
    'dnmf_reduce_scatter': (i32, [vp, vp, vp, i64, i32, vp]),
    'dnmf_bcast': (i32, [vp, vp, i64, i32, i32, vp]),
    'dnmf_group_start': (i32, []),
    'dnmf_group_end': (i32, []),
    'dnmf_symm_alloc': (i32, [i64, C.POINTER(vp), vp]),
    'dnmf_symm_open': (i32, [vp, C.POINTER(vp)]),
    'dnmf_symm_close': (i32, [vp]),
    'dnmf_symm_free': (i32, [vp]),
    'dnmf_xchg_bytes': (i64, [i32, i64, i64, i32]),
    'dnmf_xchg_error': (i32, [vp, C.POINTER(i32), vp]),
    'dnmf_xchg_update_h': (i32, [C.POINTER(vp), i32, i32, i32, vp, i64, vp, i64, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_xchg_update_h_p': (i32, [C.POINTER(vp), i32, i32, i32, vp, i64, vp, vp, i64, i64, dbl, i32, i32, vp]),
    'dnmf_hals_w_sweep': (i32, [vp, i64, vp, i64, vp, i64, i64, dbl, C.POINTER(vp), i32, i32, i64, vp, i64, i32, vp]),
    'dnmf_mu_fit_resident_smem_bytes': (i64, [i64, i64, i64, i32, i32]),
    'dnmf_mu_fit_resident_cluster_size': (i32, [i64, i64, i64, i32, i32]),
    'dnmf_mu_fit_resident': (i32, [vp, i64, vp, vp, i64, i64, i64, i64, i32, i32, i64, i64, dbl, i32, vp]),
}

_NO_STATUS = {'dnmf_trace_terms_workspace_bytes', 'dnmf_xchg_bytes', 'dnmf_pass_count', 'dnmf_version', 'dnmf_last_error', 'dnmf_last_path', 'dnmf_launch_count', 'dnmf_workspace_bytes',
              'dnmf_set_force_generic', 'dnmf_set_tc_min_elems', 'dnmf_set_tc_profile', 'dnmf_set_tc_debug', 'dnmf_set_tc_residual', 'dnmf_colsum_workspace_bytes',
              'dnmf_matvec_workspace_bytes', 'dnmf_mu_fit_resident_smem_bytes', 'dnmf_mu_fit_resident_cluster_size'}


class DnmfError(RuntimeError):
    def __init__(self, name, status, message):
        super().__init__('%s failed with status %d: %s' % (name, status, message))
        self.status = status


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'pydnmfk_b200: %s is missing. Build it with `python __graft_entry__.py` (or '
            'pydnmfk_b200/csrc/build.sh). There is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = _load()


def raw():
    return _lib


def call(name, *args):
    """Call a status-returning entry point; raise DnmfError on failure."""
    rc = getattr(_lib, name)(*args)
    if name not in _NO_STATUS and rc != 0:
        raise DnmfError(name, rc, _lib.dnmf_last_error().decode())
    return rc


def version():
    return _lib.dnmf_version().decode()


def workspace_bytes(op, m, n, k, dtype):
    b = _lib.dnmf_workspace_bytes(op, m, n, k, dtype)
    if b < 0:
        raise DnmfError('dnmf_workspace_bytes', -1, _lib.dnmf_last_error().decode())
    return b


def last_path():
    return _lib.dnmf_last_path()


def launch_count(reset=False):
    return _lib.dnmf_launch_count(1 if reset else 0)


def pass_count(tensor_path, reset=False):
    """A-streaming passes issued since the last reset through the tcgen05 (True) or generic (False) kernels."""
    return _lib.dnmf_pass_count(1 if tensor_path else 0, 1 if reset else 0)


def set_force_generic(on):
    _lib.dnmf_set_force_generic(1 if on else 0)


def set_tc_min_elems(elems):
    _lib.dnmf_set_tc_min_elems(int(elems))
