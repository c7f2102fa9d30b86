"""ctypes binding of libscanb200.so -- the same `extern "C"` surface a Rust build.rs links
(include/scanb200.h).  There is no CPU fallback: a missing library is an ImportError with the
build command, and a missing GPU surfaces as SB_ERR_CUDA from sb_init."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libscanb200.so")

SB_OK, SB_ERR_INVALID_SHAPE, SB_ERR_INVALID_K, SB_ERR_CANCELLED, SB_ERR_CUDA, SB_ERR_NCCL, SB_ERR_OOM, \
    SB_ERR_INVALID_ARG, SB_ERR_UNSUPPORTED, SB_ERR_LINALG = range(10)
SB_GENE_MAJOR, SB_CELL_MAJOR = 0, 1

PROGRESS_CB = C.CFUNCTYPE(C.c_int, C.c_double, C.c_void_p)


class SbProfile(C.Structure):
    _fields_ = [("spmm_t_ms", C.c_double), ("spmm_n_ms", C.c_double), ("moments_ms", C.c_double),
                ("reduce_ms", C.c_double), ("dense_ms", C.c_double), ("comm_ms", C.c_double),
                ("spmm_t_bytes", C.c_double), ("spmm_n_bytes", C.c_double),
                ("spmm_t_flops", C.c_double), ("spmm_n_flops", C.c_double),
                ("spmm_t_launches", C.c_uint64), ("spmm_n_launches", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("own_kernel_launches", C.c_uint64),
                ("upload_ms", C.c_double), ("build_ms", C.c_double), ("output_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ScanB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


class CancellationError(ScanB200Error):
    """snoop::CancellationError (snoop/src/lib.rs:5-18)."""


# every symbol include/scanb200.h declares (tests/test_host_abi.py checks the export list)
SYMBOLS = [
    "sb_version", "sb_last_error", "sb_init", "sb_shutdown", "sb_comm_unique_id", "sb_comm_init", "sb_sync", "sb_set_option", "sb_host_alloc", "sb_host_free",
    "sb_upload", "sb_upload_compact", "sb_pack_csc_count", "sb_pack_csc_fill", "sb_upload_packed", "sb_adaptive_decode_vec", "sb_upload_adaptive", "sb_mat_shape", "sb_download", "sb_free_mat", "sb_cell_totals", "sb_gene_totals", "sb_gene_nnz",
    "sb_median_cell_total", "sb_partition", "sb_select_rows", "sb_select_cols", "sb_hvg_select",
    "sb_normalize", "sb_log_normalize", "sb_normalize_like", "sb_normalize_fixed_point", "sb_nmat_params", "sb_nmat_to_dense",
    "sb_nmat_dot", "sb_nmat_rdot", "sb_nmat_frobenius_sq", "sb_free_nmat", "sb_omega", "sb_bksvd", "sb_bksvd_run_pca", "sb_pca_diagnostics", "sb_randsvd",
    "sb_randsvd_run_pca", "sb_profile_enable", "sb_profile_reset", "sb_profile_get", "sb_timer_begin",
    "sb_timer_end", "sb_flush_l2", "sb_synth_generate", "sb_knn",
    "sb_irlba", "sb_irlba_start", "sb_mean_var_axis", "sb_mean_var_rows", "sb_sum_rows", "sb_sum_cols", "sb_sum_rows_dual", "sb_size_factors", "sb_upload_unsorted", "sb_filter_genes", "sb_multi_init", "sb_multi_size", "sb_multi_ctx", "sb_multi_run", "sb_multi_shutdown",
    "sb_sseq_compute_params", "sb_sseq_diff_exp", "sb_sseq_one_vs_rest", "sb_sseq_pairs",
    "sb_snn_graph", "sb_louvain", "sb_cluster_knn", "sb_leiden", "sb_cluster_knn_leiden", "sb_linkage_complete", "sb_merge_clusters",
    "sb_umap_graph", "sb_umap_layout", "sb_umap", "sb_umap_transform_graph", "sb_umap_transform_layout", "sb_umap_transform", "sb_tsne_affinities", "sb_tsne_layout", "sb_tsne",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C scan_rs_b200/csrc`).  scan_rs_b200 has no CPU fallback.")
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _lib.sb_last_error.restype = C.c_char_p
        for name in SYMBOLS:
            fn = getattr(_lib, name)
            if name not in ("sb_last_error", "sb_shutdown", "sb_free_mat", "sb_free_nmat", "sb_host_free", "sb_multi_shutdown"):
                fn.restype = C.c_int
        _lib.sb_shutdown.restype = None
        _lib.sb_free_mat.restype = None
        _lib.sb_free_nmat.restype = None
        _lib.sb_host_free.restype = None
        _lib.sb_multi_shutdown.restype = None
        _lib.sb_multi_shutdown.argtypes = [C.c_void_p]
        _lib.sb_host_free.argtypes = [C.c_void_p]
    return _lib


def check(rc: int):
    if rc == SB_OK:
        return
    msg = lib().sb_last_error().decode("utf-8", "replace")
    if rc == SB_ERR_CANCELLED:
        raise CancellationError(rc, msg)
    raise ScanB200Error(rc, msg)


def vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class _Pinned:
    """Owner of one page-locked allocation (freed when the last array view dies)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        check(lib().sb_host_alloc(C.c_size_t(max(int(nbytes), 1)), C.byref(self.ptr)))
        self.nbytes = int(nbytes)

    def __del__(self):
        try:
            if self.ptr:
                lib().sb_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype):
    """numpy array in page-locked host memory (sb_host_alloc); freed with its last view."""
    import numpy as np
    dt = np.dtype(dtype)
    n = int(np.prod(shape))
    owner = _Pinned(n * dt.itemsize)
    buf = (C.c_char * max(n * dt.itemsize, 1)).from_address(owner.ptr.value)
    buf._owner = owner  # the ctypes buffer is the array's base object and keeps the allocation alive
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)
