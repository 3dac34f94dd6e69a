"""ctypes binding of libpoolgen_cuda.so (include/poolgen_cuda.h).

This is the host-side mirror of the reference's per-locus callback interface
(`ChunkyReadAnalyseWrite::read_analyse_write(&FilterStats, out, n_threads, function)`,
src/base/structs_and_traits.rs:245-265) for the four analyses `ols_iterate`, `correlation`,
`chisq`, `fisher`.  There is no CPU fallback: without the shared library or without a B200 every
call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from .build import LIB_PATH, SYNTH_LIB_PATH

PG_OK = 0
KIND_OLS, KIND_CORR, KIND_CHISQ, KIND_FISHER = 0, 1, 2, 3
KIND_OLS_KINSHIP = 4  # header selector of the writer only
KIND_MLE, KIND_GWALPHA_LS, KIND_GWALPHA_ML = 5, 6, 7  # Nelder-Mead analyses (mle_iter, gwalpha)
LOCUS_FILTERED, LOCUS_OK, LOCUS_FAILED, LOCUS_UNSUPPORTED, LOCUS_PANIC = 0, 1, 2, 3, 4
MAX_ALLELES = 6
MAX_SLOTS = 5
ALLELE_NAMES = "ATCGND"  # sync column order, src/base/sync.rs:134-137

# every symbol include/poolgen_cuda.h declares (tests check the library exports each of them)
ABI_SYMBOLS = [
    "pg_abi_version", "pg_init", "pg_destroy", "pg_last_error", "pg_device_info", "pg_device_mem_info", "pg_pinned_alloc",
    "pg_pinned_free", "pg_scan_open", "pg_scan_close", "pg_batch_create", "pg_batch_destroy",
    "pg_batch_upload_counts", "pg_batch_upload_counts_u16", "pg_batch_upload_counts_u8", "pg_batch_upload_freq", "pg_batch_upload_sync_text", "pg_batch_text_labels",
    "pg_scan_submit_sync_text", "pg_batch_synth",
    "pg_batch_run", "pg_batch_download", "pg_batch_sync", "pg_batch_results", "pg_batch_time_runs",
    "pg_batch_bytes", "pg_scan_stream_begin", "pg_scan_submit_counts", "pg_scan_submit_counts_u16",
    "pg_scan_submit_counts_u8", "pg_scan_submit_freq", "pg_scan_collect", "pg_scan_text_labels",
    "pg_kin_open", "pg_kin_close", "pg_kin_reset", "pg_kin_columns", "pg_kin_append_columns", "pg_kin_append_counts",
    "pg_kin_last_labels", "pg_kin_append_sync_text", "pg_kin_text_labels", "pg_kin_format_frequency_rows", "pg_kin_synth", "pg_kin_get_columns", "pg_kin_gram", "pg_kin_gram_accumulate", "pg_kin_gram_time", "pg_kin_partial",
    "pg_kin_partial_get", "pg_kin_partial_set", "pg_kin_eig_select", "pg_kin_eigvals", "pg_kin_set_covariates",
    "pg_kin_covar_scan", "pg_kin_mle_scan", "pg_format_header", "pg_format_rows", "pg_format_rows_ex", "pg_format_kinship_rows", "pg_format_f64", "pg_sort_loci",
    "pg_format_frequency_header", "pg_format_frequency_rows",
    "pg_shard_range", "pg_nccl_version", "pg_init_multi", "pg_comm_unique_id", "pg_comm_init_rank", "pg_comm_info",
    "pg_comm_destroy", "pg_kin_allreduce", "pg_kin_copy_covariates",
]
# include/poolgen_synth.h (libpoolgen_synth.so: host replay of the synthetic workload, no CUDA)
SYNTH_SYMBOLS = ["pg_synth_counts_host", "pg_synth_phen_host", "pg_synth_sync_text_host"]
COMM_ID_BYTES = 128
STREAM_DEPTH = 3  # PG_STREAM_DEPTH: text slabs a scan keeps in flight


class PgError(RuntimeError):
    pass


class _Filter(C.Structure):
    _fields_ = [
        ("remove_ns", C.c_int32),
        ("min_coverage_depth", C.c_uint64),
        ("min_allele_frequency", C.c_double),
        ("max_missingness_rate", C.c_double),
        ("n_pool_sizes", C.c_int32),
        ("pool_sizes", C.POINTER(C.c_double)),
    ]


def _filter(fs) -> tuple:
    """pg_filter of a FilterStats + the pool sizes array it points into, which must outlive its use"""
    ps = np.ascontiguousarray(fs.pool_sizes, dtype=np.float64)
    return _Filter(int(fs.remove_ns), int(fs.min_coverage_depth), float(fs.min_allele_frequency),
                   float(fs.max_missingness_rate), int(ps.size), ps.ctypes.data_as(C.POINTER(C.c_double))), ps


class _Results(C.Structure):
    _fields_ = [
        ("n_loci", C.c_int64),
        ("n_slots", C.c_int32),
        ("n_phen", C.c_int32),
        ("meta", C.POINTER(C.c_uint64)),
        ("freq_mean", C.POINTER(C.c_double)),
        ("stats", C.POINTER(C.c_double)),
    ]


class _RowLabels(C.Structure):
    _fields_ = [
        ("positions", C.POINTER(C.c_uint64)),
        ("text", C.c_char_p),
        ("line_offsets", C.POINTER(C.c_uint64)),
        ("chr_names", C.POINTER(C.c_char_p)),
        ("chr_index", C.POINTER(C.c_uint32)),
    ]


_lib = None


def lib():
    """Load the CUDA library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PgError(f"{LIB_PATH} is missing: run `python -m poolgen_b200.build` (nvcc, sm_100a); "
                          "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        vp, i, i64, u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
        pvp = C.POINTER(C.c_void_p)
        sig = {
            "pg_abi_version": (i, []),
            "pg_init": (i, [i, pvp]),
            "pg_destroy": (None, [vp]),
            "pg_last_error": (C.c_char_p, [vp]),
            "pg_device_info": (i, [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(C.c_size_t)]),
            "pg_device_mem_info": (i, [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
            "pg_pinned_alloc": (i, [vp, C.c_size_t, pvp]),
            "pg_pinned_free": (i, [vp, vp]),
            "pg_scan_open": (i, [vp, i, C.POINTER(_Filter), i, i, C.POINTER(C.c_uint8), C.POINTER(C.c_double), i, pvp]),
            "pg_scan_close": (i, [vp]),
            "pg_batch_create": (i, [vp, i64, pvp]),
            "pg_batch_destroy": (i, [vp]),
            "pg_batch_upload_counts": (i, [vp, vp, i64]),
            "pg_batch_upload_counts_u16": (i, [vp, vp, i64]),
            "pg_batch_upload_counts_u8": (i, [vp, vp, i64]),
            "pg_batch_upload_freq": (i, [vp, vp, vp, i64]),
            "pg_batch_upload_sync_text": (i, [vp, vp, C.c_size_t, C.POINTER(i64)]),
            "pg_batch_text_labels": (i, [vp, pvp, pvp]),
            "pg_scan_submit_sync_text": (i, [vp, vp, C.c_size_t, C.POINTER(i), C.POINTER(i64)]),
            "pg_batch_synth": (i, [vp, u64, i64, i64]),
            "pg_batch_run": (i, [vp]),
            "pg_batch_download": (i, [vp]),
            "pg_batch_sync": (i, [vp]),
            "pg_batch_results": (i, [vp, C.POINTER(_Results)]),
            "pg_batch_time_runs": (i, [vp, i, C.POINTER(C.c_float), C.POINTER(i)]),
            "pg_batch_bytes": (i, [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
            "pg_scan_stream_begin": (i, [vp, i64]),
            "pg_scan_submit_counts": (i, [vp, vp, i64, C.POINTER(i)]),
            "pg_scan_submit_counts_u16": (i, [vp, vp, i64, C.POINTER(i)]),
            "pg_scan_submit_counts_u8": (i, [vp, vp, i64, C.POINTER(i)]),
            "pg_scan_submit_freq": (i, [vp, vp, vp, i64, C.POINTER(i)]),
            "pg_scan_collect": (i, [vp, i, C.POINTER(_Results)]),
            "pg_scan_text_labels": (i, [vp, i, pvp, pvp]),
            "pg_kin_open": (i, [vp, i, i64, pvp]),
            "pg_kin_close": (i, [vp]),
            "pg_kin_reset": (i, [vp]),
            "pg_kin_columns": (i64, [vp]),
            "pg_kin_append_columns": (i, [vp, vp, i64]),
            "pg_kin_append_counts": (i, [vp, C.POINTER(_Filter), i, C.POINTER(C.c_uint8), vp, i64, i, C.POINTER(i64)]),
            "pg_kin_last_labels": (i, [vp, i64, vp, vp]),
            "pg_kin_append_sync_text": (i, [vp, C.POINTER(_Filter), vp, C.c_size_t, i64, i, C.POINTER(i64), C.POINTER(i64)]),
            "pg_kin_text_labels": (i, [vp, pvp, pvp]),
            "pg_kin_format_frequency_rows": (i, [vp, i64, i64, vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(i64)]),
            "pg_kin_synth": (i, [vp, u64, i64, i64]),
            "pg_kin_get_columns": (i, [vp, i64, i64, vp]),
            "pg_kin_gram": (i, [vp]),
            "pg_kin_gram_accumulate": (i, [vp]),
            "pg_kin_gram_time": (i, [vp, i, C.POINTER(C.c_float)]),
            "pg_kin_partial": (i, [vp, pvp, C.POINTER(C.c_size_t)]),
            "pg_kin_partial_get": (i, [vp, vp]),
            "pg_kin_partial_set": (i, [vp, vp]),
            "pg_kin_eig_select": (i, [vp, i64, C.c_double, C.POINTER(i)]),
            "pg_kin_eigvals": (i, [vp, vp, i]),
            "pg_kin_set_covariates": (i, [vp, vp, i]),
            "pg_kin_covar_scan": (i, [vp, vp, i, i, C.POINTER(C.c_float), pvp, pvp, pvp]),
            "pg_kin_mle_scan": (i, [vp, vp, i, C.POINTER(C.c_float), pvp, pvp, pvp]),
            "pg_shard_range": (i, [i64, i, i, C.POINTER(i64), C.POINTER(i64)]),
            "pg_nccl_version": (i, [C.POINTER(i)]),
            "pg_init_multi": (i, [C.POINTER(i), i, pvp, pvp]),
            "pg_comm_unique_id": (i, [vp]),
            "pg_comm_init_rank": (i, [vp, vp, i, i, pvp]),
            "pg_comm_info": (i, [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i)]),
            "pg_comm_destroy": (i, [vp]),
            "pg_kin_allreduce": (i, [vp, pvp, i, C.POINTER(i64), C.POINTER(C.c_float)]),
            "pg_kin_copy_covariates": (i, [vp, vp]),
            "pg_format_header": (i, [i, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
            "pg_format_rows": (i, [i, C.POINTER(_Results), C.POINTER(_RowLabels), i, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
            "pg_format_rows_ex": (i, [i, C.POINTER(_Results), C.POINTER(_RowLabels), i, i, i, vp, C.c_size_t,
                                      C.POINTER(C.c_size_t)]),
            "pg_format_kinship_rows": (i, [i64, i, C.POINTER(C.c_char_p), vp, C.POINTER(C.c_char_p), vp, vp, i, vp,
                                           C.c_size_t, C.POINTER(C.c_size_t)]),
            "pg_format_f64": (i, [C.c_double, i, vp, C.c_size_t]),
            "pg_sort_loci": (i, [C.POINTER(_RowLabels), i64, vp]),
            "pg_format_frequency_header": (i, [C.POINTER(C.c_char_p), i, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
            "pg_format_frequency_rows": (i, [i64, i, vp, vp, vp, C.POINTER(_RowLabels), vp, i64, i, vp, C.c_size_t,
                                             C.POINTER(C.c_size_t)]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


_synth = None


def synth_lib():
    """libpoolgen_synth.so: the host replay of the synthetic workload (plain C++, no CUDA)."""
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_LIB_PATH):
            raise PgError(f"{SYNTH_LIB_PATH} is missing: run `python -m poolgen_b200.build`")
        L = C.CDLL(SYNTH_LIB_PATH)
        i, i64, u64, vp = C.c_int, C.c_int64, C.c_uint64, C.c_void_p
        L.pg_synth_counts_host.restype, L.pg_synth_counts_host.argtypes = i, [u64, i64, i64, i, i, vp]
        L.pg_synth_phen_host.restype, L.pg_synth_phen_host.argtypes = i, [u64, i, i, vp]
        L.pg_synth_sync_text_host.restype = i
        L.pg_synth_sync_text_host.argtypes = [u64, i64, i64, i, i, vp, C.c_size_t, C.POINTER(C.c_size_t)]
        _synth = L
    return _synth


@dataclass
class FilterStats:
    """FilterStats of the reference (src/base/structs_and_traits.rs:69-78), sync-path fields only.
    pool_sizes as the phenotype loader hands them over (normalised to sum 1, src/base/phen.rs:82-84)."""
    pool_sizes: np.ndarray
    remove_ns: bool = True
    min_coverage_depth: int = 1
    min_allele_frequency: float = 0.001
    max_missingness_rate: float = 0.0


@dataclass
class ScanResults:
    """Numeric records of a batch (see pg_results in include/poolgen_cuda.h)."""
    status: np.ndarray     # uint8 [L]
    n_out: np.ndarray      # uint8 [L]
    alleles: np.ndarray    # uint8 [L, 6] allele codes of the output rows (0xff = unused)
    freq_mean: np.ndarray  # f64 [L, S]
    stats: np.ndarray      # f64 [L, S, k, 4] = (statistic, se | raw r, t, p)

    @staticmethod
    def from_c(r: _Results) -> "ScanResults":
        L, S, k = int(r.n_loci), int(r.n_slots), int(r.n_phen)
        if L == 0:
            return ScanResults(np.zeros(0, np.uint8), np.zeros(0, np.uint8), np.zeros((0, 6), np.uint8),
                               np.zeros((0, S)), np.zeros((0, S, k, 4)))
        meta = np.ctypeslib.as_array(r.meta, shape=(L,)).copy()
        fm = np.ctypeslib.as_array(r.freq_mean, shape=(L, S)).copy()
        st = np.ctypeslib.as_array(r.stats, shape=(L, S, k, 4)).copy()
        status = (meta & 0xFF).astype(np.uint8)
        n_out = ((meta >> 8) & 0xFF).astype(np.uint8)
        alle = np.full((L, 6), 0xFF, dtype=np.uint8)
        for s in range(6):
            code = ((meta >> (16 + 8 * s)) & 0xFF).astype(np.uint8)
            alle[:, s] = np.where(s < n_out, code, 0xFF)
        return ScanResults(status, n_out, alle, fm, st)


    def to_c(self):
        """a pg_results over numpy copies of these records (for the writer); returns (struct, keep-alive tuple)"""
        L = int(self.status.shape[0])
        S = int(self.freq_mean.shape[1]) if self.freq_mean.ndim == 2 else 1
        k = int(self.stats.shape[2]) if self.stats.ndim == 4 else 1
        meta = self.status.astype(np.uint64) | (self.n_out.astype(np.uint64) << np.uint64(8))
        for s in range(6):
            code = np.where(s < self.n_out, self.alleles[:, s], 0).astype(np.uint64)
            meta |= code << np.uint64(16 + 8 * s)
        meta = np.ascontiguousarray(meta)
        fm = np.ascontiguousarray(self.freq_mean, dtype=np.float64)
        st = np.ascontiguousarray(self.stats, dtype=np.float64)
        r = _Results(L, S, k, meta.ctypes.data_as(C.POINTER(C.c_uint64)), fm.ctypes.data_as(C.POINTER(C.c_double)),
                     st.ctypes.data_as(C.POINTER(C.c_double)))
        return r, (meta, fm, st)


def format_header(kind: int) -> bytes:
    """the header line of the reference's output file (src/base/sync.rs:766,950, src/gwas/ols.rs:409)"""
    buf = C.create_string_buffer(128)
    n = C.c_size_t()
    _check(lib().pg_format_header(int(kind), buf, 128, C.byref(n)), None, "pg_format_header")
    return buf.raw[:n.value]


def format_f64(x: float, n_digits: int = 0) -> str:
    """f64::to_string() (n_digits = 0) or parse_f64_roundup_and_own(x, n_digits) (src/base/helpers.rs:103-117)"""
    buf = C.create_string_buffer(512)
    n = lib().pg_format_f64(float(x), int(n_digits), buf, 512)
    if n < 0:
        raise PgError("pg_format_f64 failed")
    return buf.raw[:n].decode()


FORMAT_EXACT_P = 1


def _formatted(fn, what: str, *args) -> bytes:
    """the text of a writer call fn(*args, out, capacity, &n_bytes): once with no buffer for the size, then to fill"""
    need = C.c_size_t()
    rc = fn(*args, None, 0, C.byref(need))
    if need.value == 0:
        if rc != PG_OK:
            raise PgError(f"{what}: bad arguments")
        return b""
    buf = C.create_string_buffer(need.value)
    _check(fn(*args, buf, need.value, C.byref(need)), None, what)
    return buf.raw[:need.value]


def format_rows(kind: int, results, positions, text=None, line_offsets=None, chr_names=None, chr_index=None,
                n_threads: int = 0, exact_p_pools: int = 0) -> bytes:
    """CSV rows of the per-locus callbacks for a slab of records (`results`: ScanResults or the raw pg_results of
    Scan.collect(copy=False)).  Chromosome names come from the sync text the loci were parsed from (text as bytes or a
    uint8 array, + line_offsets, as Batch.upload_sync_text returns them) or from chr_names[chr_index[locus]].
    exact_p_pools = n_pools > 0: PG_FORMAT_EXACT_P, the printed p-values are re-derived from t with the reference's own
    arithmetic (ols_iter / pearson_corr)."""
    keep = None
    if isinstance(results, ScanResults):
        results, keep = results.to_c()
    lab, keep_lab = _row_labels(positions, text, line_offsets, chr_names, chr_index)
    flags = FORMAT_EXACT_P if exact_p_pools > 0 else 0
    return _formatted(lib().pg_format_rows_ex, "pg_format_rows_ex", int(kind), C.byref(results), C.byref(lab), flags,
                      int(exact_p_pools), n_threads or (os.cpu_count() or 1))


def _text_arg(text):
    """sync text as the library takes it: (bytes object or address of a C-contiguous uint8 array, length), no copy"""
    if isinstance(text, np.ndarray):
        assert text.dtype == np.uint8 and text.flags["C_CONTIGUOUS"]
        return text.ctypes.data, int(text.size)
    buf = bytes(text)
    return buf, len(buf)


def _row_labels(positions, text=None, line_offsets=None, chr_names=None, chr_index=None):
    """pg_row_labels + the objects that must stay alive while it is used"""
    pos = np.ascontiguousarray(positions, dtype=np.uint64)
    lab = _RowLabels()
    lab.positions = pos.ctypes.data_as(C.POINTER(C.c_uint64))
    keep = [pos]
    if text is not None:
        off = np.ascontiguousarray(line_offsets, dtype=np.uint64)
        lab.text = _text_arg(text)[0]
        lab.line_offsets = off.ctypes.data_as(C.POINTER(C.c_uint64))
        keep += [text, off]
    else:
        names = (C.c_char_p * len(chr_names))(*[n.encode() if isinstance(n, str) else n for n in chr_names])
        idx = np.ascontiguousarray(chr_index, dtype=np.uint32)
        lab.chr_names = names
        lab.chr_index = idx.ctypes.data_as(C.POINTER(C.c_uint32))
        keep += [names, idx]
    return lab, keep


def sort_loci(positions, **label_kw) -> np.ndarray:
    """the order LoadAll::load leaves the loci in: stable sort by (chromosome bytes, position), src/base/sync.rs:1092-1101"""
    lab, keep = _row_labels(positions, **label_kw)
    n = len(keep[0])
    order = np.empty(n, dtype=np.int64)
    _check(lib().pg_sort_loci(C.byref(lab), n, order.ctypes.data), None, "pg_sort_loci")
    return order


def format_frequency_header(pool_names) -> bytes:
    names = (C.c_char_p * len(pool_names))(*[n.encode() if isinstance(n, str) else n for n in pool_names])
    return _formatted(lib().pg_format_frequency_header, "pg_format_frequency_header", names, len(pool_names))


def format_frequency_rows(columns, col_locus, col_allele, positions, locus_order=None, n_threads: int = 0, **label_kw) -> bytes:
    """sync2csv rows (src/base/sync.rs:1243-1260): columns f64 [P, n_pools] with their (locus ordinal, allele code)
    labels as the column loader returns them; locus_order from sort_loci for the reference's row order."""
    cols = np.ascontiguousarray(columns, dtype=np.float64)
    cl = np.ascontiguousarray(col_locus, dtype=np.int64)
    ca = np.ascontiguousarray(col_allele, dtype=np.uint8)
    lab, keep = _row_labels(positions, **label_kw)
    order = None if locus_order is None else np.ascontiguousarray(locus_order, dtype=np.int64)
    P, n = (cols.shape if cols.ndim == 2 else (0, 1))
    return _formatted(lib().pg_format_frequency_rows, "pg_format_frequency_rows", P, n, cols.ctypes.data,
                      cl.ctypes.data, ca.ctypes.data, C.byref(lab), None if order is None else order.ctypes.data,
                      0 if order is None else order.size, n_threads or (os.cpu_count() or 1))


def format_kinship_rows(chromosome, position, allele, beta, pval, n_threads: int = 0) -> bytes:
    """rows of ols_with_covariate's writer (src/gwas/ols.rs:410-433): beta / pval [k, P]; the label sequences are
    indexed by the column ordinal exactly like the reference indexes GenotypesAndPhenotypes' label vectors."""
    b = np.ascontiguousarray(beta, dtype=np.float64)
    p = np.ascontiguousarray(pval, dtype=np.float64)
    k, P = b.shape
    enc = lambda v: v.encode() if isinstance(v, str) else v
    cn = (C.c_char_p * P)(*[enc(v) for v in chromosome[:P]])
    an = (C.c_char_p * P)(*[enc(v) for v in allele[:P]])
    pos = np.ascontiguousarray(position[:P], dtype=np.uint64)
    return _formatted(lib().pg_format_kinship_rows, "pg_format_kinship_rows", P, k, cn, pos.ctypes.data, an,
                      b.ctypes.data, p.ctypes.data, n_threads or (os.cpu_count() or 1))


def _check(rc: int, ctx=None, what: str = ""):
    if rc != PG_OK:
        msg = lib().pg_last_error(ctx)
        raise PgError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")


def _parse_labels(n_loci: int, rc_of, ctx, what: str):
    """(line byte offsets, positions) of the n_loci loci of a text parse, copied out of the library's arrays, which
    rc_of(&offsets, &positions) points at"""
    po, pp = C.c_void_p(), C.c_void_p()
    _check(rc_of(C.byref(po), C.byref(pp)), ctx, what)
    if n_loci == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    return tuple(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(n_loci,)).copy() for p in (po, pp))


class Context:
    """One context per GPU (pg_init)."""

    def __init__(self, device: int = 0, _handle=None):
        if _handle is not None:  # a context pg_init_multi created
            self._h = _handle
            self.device = device
            return
        self._h = C.c_void_p()
        rc = lib().pg_init(int(device), C.byref(self._h))
        if rc != PG_OK:
            raise PgError(f"pg_init({device}) failed ({rc}): {lib().pg_last_error(None).decode()}")
        self.device = device

    def info(self):
        sm, ma, mi, mem = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        _check(lib().pg_device_info(self._h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)), self._h, "pg_device_info")
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "total_mem": mem.value}

    def mem_info(self):
        """(free, total) device bytes now; free is what other processes on a shared GPU left"""
        f, t = C.c_size_t(), C.c_size_t()
        _check(lib().pg_device_mem_info(self._h, C.byref(f), C.byref(t)), self._h, "pg_device_mem_info")
        return int(f.value), int(t.value)

    def pinned_empty(self, shape, dtype):
        """numpy array over a library-owned pinned host slab (freed with the returned handle's .free())."""
        dt = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dt.itemsize
        p = C.c_void_p()
        _check(lib().pg_pinned_alloc(self._h, nbytes, C.byref(p)), self._h, "pg_pinned_alloc")
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
        return arr, p

    def pinned_free(self, p):
        _check(lib().pg_pinned_free(self._h, p), self._h, "pg_pinned_free")

    def close(self):
        if self._h:
            lib().pg_destroy(self._h)
            self._h = C.c_void_p()


class Scan:
    """A configured per-locus analysis = (callback kind, FilterStats, phenotypes)."""

    def __init__(self, ctx: Context, kind: int, fs: FilterStats, n_pools: int, allele_codes, phen=None):
        self.ctx = ctx
        self.kind = kind
        codes = np.ascontiguousarray(allele_codes, dtype=np.uint8)
        f, ps = _filter(fs)
        self._keep = (codes, ps)
        if phen is not None:
            y = np.ascontiguousarray(phen, dtype=np.float64)
            if y.ndim == 1:
                y = y[:, None].copy()
            k = y.shape[1]
            if kind in (KIND_GWALPHA_LS, KIND_GWALPHA_ML):
                # the gwalpha_fmt matrix [rows, 3]: column 0 bins, column 1 q, column 2 = sig, MIN, MAX, then -inf
                assert y.shape[1] == 3, y.shape
                k = y.shape[0]
            yp = y.ctypes.data_as(C.POINTER(C.c_double))
        else:
            y, k, yp = None, 0, None
        self.n_pools, self.n_alleles = int(n_pools), int(codes.size)
        self.k = 1 if kind in (KIND_GWALPHA_LS, KIND_GWALPHA_ML) else k
        self._h = C.c_void_p()
        _check(lib().pg_scan_open(ctx._h, int(kind), C.byref(f), int(n_pools), int(codes.size),
                                  codes.ctypes.data_as(C.POINTER(C.c_uint8)), yp, int(k), C.byref(self._h)),
               ctx._h, "pg_scan_open")

    def batch(self, capacity: int) -> "Batch":
        return Batch(self, capacity)

    def run_counts(self, counts) -> ScanResults:
        """counts: uint32 (or uint16) [L, A, n_pools] -> records, synchronously."""
        c = np.ascontiguousarray(counts)
        b = self.batch(max(1, c.shape[0]))
        try:
            b.upload_counts(c)
            b.run()
            return b.fetch()
        finally:
            b.close()

    # streaming: pg_scan_stream_begin / submit / collect
    def stream_begin(self, max_loci: int):
        _check(lib().pg_scan_stream_begin(self._h, int(max_loci)), self.ctx._h, "pg_scan_stream_begin")

    def submit_counts(self, counts) -> int:
        t = C.c_int()
        c = counts
        assert c.flags["C_CONTIGUOUS"]
        assert c.dtype in (np.uint32, np.uint16, np.uint8)
        fn = {4: lib().pg_scan_submit_counts, 2: lib().pg_scan_submit_counts_u16, 1: lib().pg_scan_submit_counts_u8}[c.dtype.itemsize]
        _check(fn(self._h, c.ctypes.data, int(c.shape[0]), C.byref(t)), self.ctx._h, "pg_scan_submit_counts")
        return t.value

    def submit_freq(self, freq, depth) -> int:
        t = C.c_int()
        assert freq.dtype == np.float64 and depth.dtype == np.uint32
        assert freq.flags["C_CONTIGUOUS"] and depth.flags["C_CONTIGUOUS"]
        _check(lib().pg_scan_submit_freq(self._h, freq.ctypes.data, depth.ctypes.data, int(freq.shape[0]), C.byref(t)),
               self.ctx._h, "pg_scan_submit_freq")
        return t.value

    def collect(self, ticket: int, copy: bool = True):
        r = _Results()
        _check(lib().pg_scan_collect(self._h, int(ticket), C.byref(r)), self.ctx._h, "pg_scan_collect")
        return ScanResults.from_c(r) if copy else r

    def close(self):
        if self._h:
            lib().pg_scan_close(self._h)
            self._h = C.c_void_p()


class Batch:
    def __init__(self, scan: Scan, capacity: int):
        self.scan = scan
        self._h = C.c_void_p()
        self._keep = None
        _check(lib().pg_batch_create(scan._h, int(capacity), C.byref(self._h)), scan.ctx._h, "pg_batch_create")

    def _ck(self, rc, what):
        _check(rc, self.scan.ctx._h, what)

    def upload_counts(self, counts):
        c = np.ascontiguousarray(counts)
        if c.dtype not in (np.uint32, np.uint16, np.uint8):
            c = c.astype(np.uint32)
        assert c.ndim == 3 and c.shape[1] == self.scan.n_alleles and c.shape[2] == self.scan.n_pools, c.shape
        self._keep = c
        fn = {4: lib().pg_batch_upload_counts, 2: lib().pg_batch_upload_counts_u16, 1: lib().pg_batch_upload_counts_u8}[c.dtype.itemsize]
        self._ck(fn(self._h, c.ctypes.data, int(c.shape[0])), "pg_batch_upload_counts")

    def upload_freq(self, freq, depth):
        f = np.ascontiguousarray(freq, dtype=np.float64)
        d = np.ascontiguousarray(depth, dtype=np.uint32)
        self._keep = (f, d)
        self._ck(lib().pg_batch_upload_freq(self._h, f.ctypes.data, d.ctypes.data, int(f.shape[0])), "pg_batch_upload_freq")

    def synth(self, seed: int, first_locus: int, n_loci: int):
        self._ck(lib().pg_batch_synth(self._h, int(seed), int(first_locus), int(n_loci)), "pg_batch_synth")

    def upload_sync_text(self, text: bytes):
        """a line-aligned chunk of a sync file, parsed on the device; returns (n_loci, line byte offsets, positions)"""
        buf = bytes(text)
        self._keep = buf
        n = C.c_int64()
        self._ck(lib().pg_batch_upload_sync_text(self._h, buf, len(buf), C.byref(n)), "pg_batch_upload_sync_text")
        L = int(n.value)
        off, pos = _parse_labels(L, lambda po, pp: lib().pg_batch_text_labels(self._h, po, pp), self.scan.ctx._h,
                                 "pg_batch_text_labels")
        return L, off, pos

    def run(self):
        self._ck(lib().pg_batch_run(self._h), "pg_batch_run")

    def sync(self):
        self._ck(lib().pg_batch_sync(self._h), "pg_batch_sync")

    def time_runs(self, iters: int):
        ms, nl = C.c_float(), C.c_int()
        self._ck(lib().pg_batch_time_runs(self._h, int(iters), C.byref(ms), C.byref(nl)), "pg_batch_time_runs")
        return float(ms.value), int(nl.value)

    def bytes(self):
        a, b = C.c_size_t(), C.c_size_t()
        self._ck(lib().pg_batch_bytes(self._h, C.byref(a), C.byref(b)), "pg_batch_bytes")
        return int(a.value), int(b.value)

    def download(self):
        self._ck(lib().pg_batch_download(self._h), "pg_batch_download")

    def results_view(self) -> _Results:
        r = _Results()
        self._ck(lib().pg_batch_results(self._h, C.byref(r)), "pg_batch_results")
        return r

    def fetch(self) -> ScanResults:
        self.download()
        self.sync()
        return ScanResults.from_c(self.results_view())

    def close(self):
        if self._h:
            lib().pg_batch_destroy(self._h)
            self._h = C.c_void_p()


class Kinship:
    """ols_with_covariate (src/gwas/ols.rs:278-436) over this GPU's shard of allele columns (pg_kin_*)."""

    def __init__(self, ctx: Context, n_pools: int, max_columns: int):
        self.ctx, self.n = ctx, int(n_pools)
        self._h = C.c_void_p()
        _check(lib().pg_kin_open(ctx._h, int(n_pools), int(max_columns), C.byref(self._h)), ctx._h, "pg_kin_open")

    def _ck(self, rc, what):
        _check(rc, self.ctx._h, what)

    @property
    def columns(self) -> int:
        return int(lib().pg_kin_columns(self._h))

    def reset(self):
        self._ck(lib().pg_kin_reset(self._h), "pg_kin_reset")

    def append_columns(self, cols):
        """cols: f64 [P_add, n_pools] (one allele column per row)."""
        c = np.ascontiguousarray(cols, dtype=np.float64)
        assert c.ndim == 2 and c.shape[1] == self.n, c.shape
        self._ck(lib().pg_kin_append_columns(self._h, c.ctypes.data, int(c.shape[0])), "pg_kin_append_columns")

    def append_counts(self, counts, allele_codes, fs: FilterStats, keep_p_minus_1: bool = False):
        """counts: uint32 [L, A, n_pools]; returns (col_locus int64 [P_add], col_allele uint8 [P_add])."""
        c = np.ascontiguousarray(counts, dtype=np.uint32)
        codes = np.ascontiguousarray(allele_codes, dtype=np.uint8)
        f, _ps = _filter(fs)
        added = C.c_int64()
        self._ck(lib().pg_kin_append_counts(self._h, C.byref(f), int(codes.size),
                                            codes.ctypes.data_as(C.POINTER(C.c_uint8)), c.ctypes.data, int(c.shape[0]),
                                            int(keep_p_minus_1), C.byref(added)), "pg_kin_append_counts")
        n_add = int(added.value)
        loc = np.empty(n_add, dtype=np.int64)
        alle = np.empty(n_add, dtype=np.uint8)
        self._ck(lib().pg_kin_last_labels(self._h, n_add, loc.ctypes.data, alle.ctypes.data), "pg_kin_last_labels")
        return loc, alle

    def append_sync_text(self, text, fs: FilterStats, max_loci: int, keep_p_minus_1: bool = False):
        """a line-aligned chunk of sync text (bytes or a uint8 array) through the device parser and LoadAll: returns
        (n_loci, line offsets, positions, col_locus, col_allele)"""
        buf, size = _text_arg(text)
        f, _ps = _filter(fs)
        nl, added = C.c_int64(), C.c_int64()
        self._ck(lib().pg_kin_append_sync_text(self._h, C.byref(f), buf, size, int(max_loci), int(keep_p_minus_1),
                                               C.byref(nl), C.byref(added)), "pg_kin_append_sync_text")
        L, n_add = int(nl.value), int(added.value)
        off, pos = _parse_labels(L, lambda po, pp: lib().pg_kin_text_labels(self._h, po, pp), self.ctx._h,
                                 "pg_kin_text_labels")
        loc = np.empty(n_add, dtype=np.int64)
        alle = np.empty(n_add, dtype=np.uint8)
        self._ck(lib().pg_kin_last_labels(self._h, n_add, loc.ctypes.data, alle.ctypes.data), "pg_kin_last_labels")
        return L, off, pos, loc, alle

    def format_frequency_rows(self, first: int, count: int, out) -> tuple:
        """sync2csv rows of columns [first, first + count) of the last append_sync_text, formatted on the device into
        `out` (a writable uint8 array, ideally Context.pinned_empty): returns (bytes, rows) of the whole rows that fit"""
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"] and out.flags["WRITEABLE"]
        nb, nr = C.c_size_t(), C.c_int64()
        self._ck(lib().pg_kin_format_frequency_rows(self._h, int(first), int(count), out.ctypes.data, out.size,
                                                    C.byref(nb), C.byref(nr)), "pg_kin_format_frequency_rows")
        return int(nb.value), int(nr.value)

    def synth(self, seed: int, first_locus: int, n_loci: int):
        self._ck(lib().pg_kin_synth(self._h, int(seed), int(first_locus), int(n_loci)), "pg_kin_synth")

    def get_columns(self, first: int, count: int) -> np.ndarray:
        out = np.empty((count, self.n), dtype=np.float64)
        self._ck(lib().pg_kin_get_columns(self._h, int(first), int(count), out.ctypes.data), "pg_kin_get_columns")
        return out

    def gram(self, accumulate: bool = False):
        """K = G G' of the resident columns; with accumulate, K += G G' (a later block of a column set larger than the
        device: reset() keeps K)"""
        if accumulate:
            self._ck(lib().pg_kin_gram_accumulate(self._h), "pg_kin_gram_accumulate")
        else:
            self._ck(lib().pg_kin_gram(self._h), "pg_kin_gram")

    def gram_time(self, iters: int) -> float:
        ms = C.c_float()
        self._ck(lib().pg_kin_gram_time(self._h, int(iters), C.byref(ms)), "pg_kin_gram_time")
        return float(ms.value)

    def partial_device_ptr(self):
        """(device pointer, element count) of the n x n partial Gram matrix, for an NCCL all-reduce by the caller."""
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(lib().pg_kin_partial(self._h, C.byref(p), C.byref(n)), "pg_kin_partial")
        return int(p.value), int(n.value)

    def partial_get(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.float64)
        self._ck(lib().pg_kin_partial_get(self._h, out.ctypes.data), "pg_kin_partial_get")
        return out

    def partial_set(self, K):
        k = np.ascontiguousarray(K, dtype=np.float64)
        assert k.shape == (self.n, self.n)
        self._ck(lib().pg_kin_partial_set(self._h, k.ctypes.data), "pg_kin_partial_set")

    def copy_covariates_from(self, src: "Kinship"):
        """the outcome of another handle's eigen step (one process, several GPUs: the step is replicated work)"""
        self._ck(lib().pg_kin_copy_covariates(self._h, src._h), "pg_kin_copy_covariates")

    def eig_select(self, P_total: int, variance_explained: float) -> int:
        m = C.c_int()
        self._ck(lib().pg_kin_eig_select(self._h, int(P_total), float(variance_explained), C.byref(m)), "pg_kin_eig_select")
        return int(m.value)

    def eigvals(self, count: int) -> np.ndarray:
        out = np.empty(count, dtype=np.float64)
        self._ck(lib().pg_kin_eigvals(self._h, out.ctypes.data, int(count)), "pg_kin_eigvals")
        return out

    def set_covariates(self, cov):
        c = np.ascontiguousarray(cov, dtype=np.float64).reshape(self.n, -1)
        self._ck(lib().pg_kin_set_covariates(self._h, c.ctypes.data if c.size else None, int(c.shape[1])), "pg_kin_set_covariates")

    def covar_scan(self, phen, iters: int = 0):
        """phen [n_pools, k] -> (beta, var, pval) each [k, columns] (+ milliseconds of `iters` launches if iters > 0)."""
        y = np.ascontiguousarray(phen, dtype=np.float64)
        if y.ndim == 1:
            y = y[:, None].copy()
        k = y.shape[1]
        ms = C.c_float()
        pb, pv, pp = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._ck(lib().pg_kin_covar_scan(self._h, y.ctypes.data, int(k), int(iters), C.byref(ms), C.byref(pb), C.byref(pv),
                                         C.byref(pp)), "pg_kin_covar_scan")
        out = self._records(k, (pb, pv, pp))
        return out + (float(ms.value),) if iters > 0 else out

    def mle_scan(self, phen, timed: bool = False):
        """mle_with_covariate (gwas/mle.rs:307-463): phen [n_pools, k] -> (beta, var, pval) each [k, columns]
        (+ kernel milliseconds if timed)."""
        y = np.ascontiguousarray(phen, dtype=np.float64)
        if y.ndim == 1:
            y = y[:, None].copy()
        k = y.shape[1]
        ms = C.c_float()
        pb, pv, pp = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._ck(lib().pg_kin_mle_scan(self._h, y.ctypes.data, int(k), C.byref(ms), C.byref(pb), C.byref(pv), C.byref(pp)),
                 "pg_kin_mle_scan")
        out = self._records(k, (pb, pv, pp))
        return out + (float(ms.value),) if timed else out

    def _records(self, k: int, ptrs) -> tuple:
        """copies of the scan's [k, columns] f64 record arrays behind ptrs"""
        P = self.columns
        if P == 0:
            return tuple(np.zeros((k, 0)) for _ in ptrs)
        return tuple(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(k, P)).copy() for p in ptrs)

    def close(self):
        if self._h:
            lib().pg_kin_close(self._h)
            self._h = C.c_void_p()


def _pin_nccl_library():
    """One libnccl.so.2 per process: the dynamic loader keeps a single object per SONAME, so when this Python process
    will also import torch (whose bundled NCCL may be newer than the system's), the library must map that same file --
    PG_NCCL_LIB tells it which (see pg_comm.cu).  A no-op when the variable is set or no bundled NCCL exists."""
    if os.environ.get("PG_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
            cand = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["PG_NCCL_LIB"] = cand
                return
    except (ImportError, ValueError, AttributeError):
        pass


def shard_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """pg_shard_range: the contiguous [begin, end) of `rank` (earlier ranks take the larger shards)"""
    b, e = C.c_int64(), C.c_int64()
    _check(lib().pg_shard_range(int(total), int(rank), int(world), C.byref(b), C.byref(e)), None, "pg_shard_range")
    return int(b.value), int(e.value)


def nccl_version() -> int:
    _pin_nccl_library()
    v = C.c_int()
    _check(lib().pg_nccl_version(C.byref(v)), None, "pg_nccl_version")
    return int(v.value)


class Comm:
    """The library's NCCL communicator (pg_comm): `Comm.init_multi(devices)` for one process driving several GPUs
    (what the Rust CLI does, src/main.rs:280-298), `Comm.init_rank(ctx, id, rank, world)` for one process per GPU."""

    def __init__(self, handle, contexts):
        self._h = handle
        self.contexts = contexts

    @staticmethod
    def init_multi(devices) -> "Comm":
        _pin_nccl_library()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        ctxs = (C.c_void_p * len(devices))()
        h = C.c_void_p()
        _check(lib().pg_init_multi(devs, len(devices), ctxs, C.byref(h)), None, "pg_init_multi")
        return Comm(h, [Context(int(d), _handle=C.c_void_p(c)) for d, c in zip(devices, ctxs)])

    @staticmethod
    def unique_id() -> bytes:
        _pin_nccl_library()
        buf = C.create_string_buffer(COMM_ID_BYTES)
        _check(lib().pg_comm_unique_id(buf), None, "pg_comm_unique_id")
        return buf.raw

    @staticmethod
    def init_rank(ctx: Context, uid: bytes, rank: int, world: int) -> "Comm":
        assert len(uid) == COMM_ID_BYTES
        _pin_nccl_library()
        h = C.c_void_p()
        _check(lib().pg_comm_init_rank(ctx._h, uid, int(rank), int(world), C.byref(h)), ctx._h, "pg_comm_init_rank")
        return Comm(h, [ctx])

    def info(self):
        w, n, f = C.c_int(), C.c_int(), C.c_int()
        _check(lib().pg_comm_info(self._h, C.byref(w), C.byref(n), C.byref(f)), None, "pg_comm_info")
        return {"world": w.value, "n_local": n.value, "first_rank": f.value}

    def kin_allreduce(self, kins, timed: bool = False):
        """sum the partial Gram matrices (and the column counts) of `kins` (one per local rank) over the communicator;
        returns the total column count (and the device milliseconds of the exchange step when timed)"""
        arr = (C.c_void_p * len(kins))(*[k._h for k in kins])
        tot, ms = C.c_int64(), C.c_float()
        _check(lib().pg_kin_allreduce(self._h, arr, len(kins), C.byref(tot), C.byref(ms) if timed else None),
               kins[0].ctx._h, "pg_kin_allreduce")
        return (int(tot.value), float(ms.value)) if timed else int(tot.value)

    def close(self):
        if self._h:
            lib().pg_comm_destroy(self._h)
            self._h = C.c_void_p()


def submit_sync_text(scan: "Scan", text: bytes, deferred: bool = False):
    """pg_scan_submit_sync_text: parse + scan + download of one text slab; returns (ticket, n_loci).
    deferred=True passes n_loci = NULL: the call only enqueues the copy and the parse (n_loci comes back as None, the
    count is in the collected records) and the slab's scan is launched by the next submit or by its collect."""
    t, n = C.c_int(), C.c_int64()
    buf, size = _text_arg(text)
    if not hasattr(scan, "_keep_text"):
        scan._keep_text = {}
    _check(lib().pg_scan_submit_sync_text(scan._h, buf, size, C.byref(t), None if deferred else C.byref(n)),
           scan.ctx._h, "pg_scan_submit_sync_text")
    scan._keep_text[t.value] = (text, buf)  # the chunk must stay alive until its ticket is collected
    return t.value, (None if deferred else int(n.value))


def text_labels(scan: "Scan", ticket: int, n_loci: int):
    """pg_scan_text_labels after the collect of `ticket`: (line byte offsets, positions) of its loci"""
    return _parse_labels(int(n_loci), lambda po, pp: lib().pg_scan_text_labels(scan._h, int(ticket), po, pp),
                         scan.ctx._h, "pg_scan_text_labels")


def synth_counts_host(seed: int, first_locus: int, n_loci: int, n_pools: int, n_alleles: int) -> np.ndarray:
    out = np.empty((n_loci, n_alleles, n_pools), dtype=np.uint32)
    rc = synth_lib().pg_synth_counts_host(int(seed), int(first_locus), int(n_loci), int(n_pools), int(n_alleles), out.ctypes.data)
    if rc != PG_OK:
        raise PgError(f"pg_synth_counts_host failed ({rc})")
    return out


def synth_sync_text_host(seed: int, first_locus: int, n_loci: int, n_pools: int, n_alleles: int, out: np.ndarray) -> int:
    """writes the synthetic counts as sync text into `out` (uint8 array, e.g. over pinned memory); returns the bytes"""
    nb = C.c_size_t()
    rc = synth_lib().pg_synth_sync_text_host(int(seed), int(first_locus), int(n_loci), int(n_pools), int(n_alleles),
                                       out.ctypes.data, int(out.size), C.byref(nb))
    if rc != PG_OK:
        raise PgError(f"pg_synth_sync_text_host failed ({rc}): needs {nb.value} bytes, has {out.size}")
    return int(nb.value)


def synth_phen_host(seed: int, n_pools: int, k: int) -> np.ndarray:
    out = np.empty((n_pools, k), dtype=np.float64)
    rc = synth_lib().pg_synth_phen_host(int(seed), int(n_pools), int(k), out.ctypes.data)
    if rc != PG_OK:
        raise PgError(f"pg_synth_phen_host failed ({rc})")
    return out
