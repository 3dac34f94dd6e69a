"""File-level mirror of the reference's chunked readers for the hot path: `FilePhen::lparse` (src/base/phen.rs:21-98),
`find_file_splits` (src/base/helpers.rs:16-27, 74-91) and `ChunkyReadAnalyseWrite::read_analyse_write` of `FileSyncPhen`
/ `FileSync` (src/base/sync.rs:606-786, 788-970), with the same names and argument meaning.

What differs is where the work happens: a reader thread does not parse its lines and call a per-locus callback, it hands
line-aligned blocks of raw bytes to the library (`pg_scan_submit_sync_text`: parse + filter + regression on the GPU) and
appends the rows `pg_format_rows` returns.  Nothing here computes on the CPU; without the CUDA library every call raises.
"""
from __future__ import annotations

import os
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np

from . import capi
from .capi import (KIND_CHISQ, KIND_CORR, KIND_FISHER, KIND_GWALPHA_LS, KIND_GWALPHA_ML, KIND_MLE, KIND_OLS, Context,
                   FilterStats, PgError, Scan)

_MISSING = {"", "NA", "NAN", "NaN", "na", "nan"}  # src/base/phen.rs:66-72


@dataclass
class Phen:
    """src/base/structs_and_traits.rs: Phen { pool_names, pool_sizes (normalised to sum 1), phen_matrix n x k }"""
    pool_names: list
    pool_sizes: np.ndarray
    phen_matrix: np.ndarray


@dataclass
class FilePhen:
    """src/base/structs_and_traits.rs: FilePhen; only the "default" delimited format (the GWAlpha format feeds
    `gwalpha`, which is not part of this path)"""
    filename: str
    delim: str = ","
    names_column_id: int = 0
    sizes_column_id: int = 1
    trait_values_column_ids: list = field(default_factory=lambda: [2])
    format: str = "default"

    def lparse(self) -> Phen:
        """src/base/phen.rs:21-98: '#' lines skipped, fields trimmed, missing values -> NaN, pool sizes divided by their
        sequential sum"""
        if self.format != "default":
            raise PgError("Invalid phenotype format for this path: only 'default' (src/base/phen.rs:24-98)")
        names, sizes, vals = [], [], []
        with open(self.filename, "r", newline="") as fh:
            for line in fh:
                line = line.rstrip("\n").rstrip("\r")
                if line[:1] == "#":  # the reference indexes byte 0: an empty line panics there
                    continue
                if line == "":
                    raise PgError("empty line in the phenotype file (the reference panics: index out of bounds)")
                f = [x.strip() for x in line.split(self.delim)]
                names.append(f[self.names_column_id])
                try:
                    sizes.append(float(f[self.sizes_column_id]))
                except ValueError:
                    raise PgError(f"T_T Pool sizes column (column index: {self.sizes_column_id}) is not a valid number. "
                                  f"Line: {line}.") from None
                for j in self.trait_values_column_ids:
                    vals.append(float("nan") if f[j] in _MISSING else float(f[j]))
        total = 0.0
        for s in sizes:  # `pool_sizes.iter().sum()`: sequential
            total = total + s
        k = len(self.trait_values_column_ids)
        n = len(vals) // k
        return Phen(names, np.array([s / total for s in sizes], dtype=np.float64),
                    np.array(vals, dtype=np.float64).reshape(n, k))


def _find_start_of_next_line(fname: str, pos: int) -> int:
    """src/base/helpers.rs:16-27: for pos > 0 the rest of the line at pos is skipped (a full line when pos is a start)"""
    if pos <= 0:
        return 0
    with open(fname, "rb") as fh:
        fh.seek(pos)
        fh.readline()
        return fh.tell()


def find_file_splits(fname: str, n_threads: int) -> list:
    """src/base/helpers.rs:74-91: (0..end).step_by(end / n_threads) + end, each moved to the start of the next line,
    consecutive duplicates removed"""
    if not os.path.exists(fname):
        raise PgError(f"The input file: {fname} does not exist. Please make sure you are entering the correct filename "
                      "and/or the correct path.")
    end = os.path.getsize(fname)
    step = end // n_threads
    if step == 0:
        raise PgError("more threads than bytes in the input file (the reference panics: step_by(0))")
    out = list(range(0, end, step)) + [end]
    out = [_find_start_of_next_line(fname, p) for p in out]
    dedup = [out[0]]
    for p in out[1:]:
        if p != dedup[-1]:
            dedup.append(p)
    return dedup


def _kind_of(function) -> int:
    """the reference passes the callback itself (gwas::ols_iterate, gwas::correlation, tables::chisq, tables::fisher)"""
    if isinstance(function, int):
        return function
    name = getattr(function, "__name__", str(function))
    table = {"ols_iterate": KIND_OLS, "correlation": KIND_CORR, "chisq": KIND_CHISQ, "fisher": KIND_FISHER,
             "mle_iterate": KIND_MLE, "gwalpha_ls": KIND_GWALPHA_LS, "gwalpha_ml": KIND_GWALPHA_ML}
    if name not in table:
        raise PgError(f"unknown per-locus function {name!r}")
    return table[name]


def _default_out(fname: str, test: str) -> str:
    """src/base/sync.rs:885-903: <name without its last extension>-<seconds>-<test>.csv"""
    bname = ".".join(fname.split(".")[:-1])
    return f"{bname}-{time.time()}-{test}.csv"


def _last_line_end(view) -> int:
    """the length of view up to and including its last newline, 0 if it has none; searched back from the end"""
    hi = view.size
    while hi:
        lo = max(hi - (1 << 16), 0)
        nl = np.flatnonzero(view[lo:hi] == 10)
        if nl.size:
            return lo + int(nl[-1]) + 1
        hi = lo
    return 0


def _line_blocks(fname: str, start: int, end: int, block_bytes: int, bufs: list):
    """(absolute byte offset, uint8 view) of line-aligned blocks of at most block_bytes bytes over [start, end) of the
    file, read into the arrays `bufs` in turn.  While bytes of the range remain, a block ends at its last newline and
    the rest moves to the head of the next buffer; the last block takes what is left, so a last line without a newline
    joins it where it fits.  Block i + len(bufs) reuses the buffer of block i: the caller is done with block i before
    it asks for that one (with one buffer, before it asks for the next block)."""
    with open(fname, "rb", buffering=0) as fh:
        fh.seek(start)
        at, left, tail, i = start, end - start, bufs[0][:0], 0
        while left > 0 or tail.size:
            buf, nc = bufs[i % len(bufs)], tail.size
            buf[:nc] = tail
            got = fh.readinto(memoryview(buf)[nc:nc + min(left, block_bytes - nc)]) if left > 0 else 0
            left = left - got if got else 0  # the file ended before the range did
            fill = cut = nc + got
            if left:
                cut = _last_line_end(buf[:fill])
                if cut == 0:
                    raise PgError(f"a line of {fname} is longer than the block size {block_bytes}")
            if cut:
                yield at, buf[:cut]
            at, tail, i = at + cut, buf[cut:fill], i + 1


def _chunk_worker(ctx: Context, kind: int, fs: FilterStats, n_pools: int, phen, fname: str, start: int, end: int,
                  block_bytes: int, fmt_threads: int, sink: list, errors: list):
    """the body of `per_chunk` (src/base/sync.rs:794-870 / 612-687) for the byte range [start, end)"""
    scan = None
    pinned = []
    try:
        scan = Scan(ctx, kind, fs, n_pools, np.arange(6, dtype=np.uint8), phen)
        scan.stream_begin(_max_loci(block_bytes, n_pools))
        bufs = []
        for _ in range(capi.STREAM_DEPTH):
            arr, h = ctx.pinned_empty((block_bytes,), np.uint8)
            pinned.append(h)
            bufs.append(arr)
        out = bytearray()
        pending = []  # (ticket, block)

        def finish(ticket, block):
            res = scan.collect(ticket, copy=False)
            if res.n_loci:
                off, pos = capi.text_labels(scan, ticket, res.n_loci)
                # the output file carries the reference's own p-value digits (PG_FORMAT_EXACT_P)
                out.extend(capi.format_rows(kind, res, pos, text=block, line_offsets=off, n_threads=fmt_threads,
                                            exact_p_pools=n_pools))

        for _, block in _line_blocks(fname, start, end, block_bytes, bufs):
            pending.append((capi.submit_sync_text(scan, block, deferred=True)[0], block))
            if len(pending) == len(bufs):
                finish(*pending.pop(0))
        while pending:
            finish(*pending.pop(0))
        sink.append((start, bytes(out)))
    except Exception as e:  # noqa: BLE001 -- re-raised by the caller, like a panicking reader thread
        errors.append(e)
    finally:
        if scan is not None:
            scan.close()
        for h in pinned:
            ctx.pinned_free(h)


def _read_analyse_write(ctx, kind, fs, n_pools, phen, fname, test, out, n_threads, block_bytes):
    if out == "":
        out = _default_out(fname, test)
    if os.path.exists(out):
        raise PgError("Cannot write to output file")  # create_new(true), src/base/sync.rs:905
    chunks = find_file_splits(fname, n_threads)
    if len(chunks) - 1 < n_threads:
        # the reference indexes chunks[n_threads] unguarded (src/base/sync.rs:909) and panics
        raise PgError(f"{n_threads} threads but only {len(chunks) - 1} line-aligned chunks in {fname}")
    sink, errors, threads = [], [], []
    fmt_threads = max(1, (os.cpu_count() or 1) // n_threads)
    for i in range(n_threads):
        t = threading.Thread(target=_chunk_worker, args=(ctx, kind, fs, n_pools, phen, fname, chunks[i], chunks[i + 1],
                                                         block_bytes, fmt_threads, sink, errors))
        t.start()
        threads.append(t)
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    with open(out, "xb") as fo:
        fo.write(capi.format_header(kind))
        for _, rows in sorted(sink):  # chunk files are concatenated in name order = start offset order (sync.rs:953-967)
            fo.write(rows)
    return out


@dataclass
class FileSyncPhen:
    """src/base/structs_and_traits.rs: FileSyncPhen { filename_sync, pool_names, pool_sizes, phen_matrix, test }"""
    filename_sync: str
    pool_names: list
    pool_sizes: np.ndarray
    phen_matrix: np.ndarray
    test: str = "ols_iter"

    def read_analyse_write(self, ctx: Context, filter_stats: FilterStats, out: str, n_threads: int, function,
                           block_bytes: int = 32 << 20) -> str:
        """`read_analyse_write(&self, &FilterStats, out, n_threads, function)` (src/base/sync.rs:872-970) for
        function = ols_iterate | correlation | mle_iterate | gwalpha_ls | gwalpha_ml (for the last two phen_matrix is
        the gwalpha_fmt matrix, src/main.rs:335-358): returns the output file name"""
        kind = _kind_of(function)
        if kind not in (KIND_OLS, KIND_CORR, KIND_MLE, KIND_GWALPHA_LS, KIND_GWALPHA_ML):
            raise PgError("FileSyncPhen::read_analyse_write takes gwas::ols_iterate, correlation, mle_iterate or gwalpha_ls / _ml")
        return _read_analyse_write(ctx, kind, filter_stats, len(self.pool_names), self.phen_matrix, self.filename_sync,
                                   self.test, out, n_threads, block_bytes)


@dataclass
class FileSync:
    """src/base/structs_and_traits.rs: FileSync { filename, test } -- the count tests need no phenotypes, only the pool
    sizes that travel in FilterStats"""
    filename: str
    test: str = "chisq_test"

    def read_analyse_write(self, ctx: Context, filter_stats: FilterStats, out: str, n_threads: int, function,
                           block_bytes: int = 32 << 20) -> str:
        """src/base/sync.rs:689-786 for function = chisq | fisher"""
        kind = _kind_of(function)
        if kind not in (KIND_CHISQ, KIND_FISHER):
            raise PgError("FileSync::read_analyse_write takes tables::chisq or tables::fisher")
        return _read_analyse_write(ctx, kind, filter_stats, int(np.asarray(filter_stats.pool_sizes).size), None,
                                   self.filename, self.test, out, n_threads, block_bytes)


# ---- whole-matrix entries: sync2csv (SaveCsv::write_csv, src/base/sync.rs:1182-1262) and ols_iter_with_kinship
# (into_genotypes_and_phenotypes + ols_with_covariate, src/base/sync.rs:1106-1179, src/gwas/ols.rs:278-436) ----------
@dataclass
class _LoadedColumns:
    col_locus: np.ndarray  # int64 [P] locus ordinal (over the kept loci of the whole file) of every column
    col_allele: np.ndarray # uint8 [P]
    chr_names: list        # distinct chromosome names
    chr_index: np.ndarray  # uint32 [L]
    positions: np.ndarray  # uint64 [L]


# ---- columns beyond one device: the handle holds a device block of columns at a time -------------------------------
_COLS_PER_LINE = 6  # a locus emits at most six allele columns (--keep-ns with MAF 0 and no --keep-p-minus-1)
_KIN_RESERVE_BYTES = 1 << 30  # outside the handle: cuSOLVER's and cuBLAS' handles, kernel modules loaded on first use


def _line_min_bytes(n_pools: int) -> int:
    """a locus line holds at least "c\\t0\\tN" + n_pools * "\\t0:0:0:0:0:0" bytes"""
    return 12 * n_pools + 5


def _max_loci(block_bytes: int, n_pools: int) -> int:
    """the loci a text block of block_bytes bytes can hold at most: the max_loci of the device loaders"""
    return block_bytes // _line_min_bytes(n_pools) + 2


def text_block_columns(n_bytes: int, n_pools: int, n_lines: int = None) -> int:
    """an upper bound of the allele columns a text block of n_bytes bytes (n_lines newlines, if known) can emit: six
    per line, as many lines as the bytes can hold"""
    lines = n_bytes // _line_min_bytes(n_pools) + 1
    if n_lines is not None:
        lines = min(lines, n_lines + 1)
    return _COLS_PER_LINE * lines


def _grow(need: int, elem: int) -> int:
    """bytes of a text-scratch buffer of `need` elements (pg_text.cu: grow() keeps an eighth and 64 Ki elements spare)"""
    return (need + need // 8 + 65536) * elem


def kin_device_bytes(n_pools: int, columns: int, k: int, block_bytes: int, sm_count: int) -> int:
    """Device bytes (plus the pinned copy of the records) a pg_kin handle of `columns` columns takes at most when it is
    filled from text blocks of at most block_bytes bytes, its Gram matrix formed, its eigen step run and k phenotypes
    scanned (pg_kinship.cu, pg_text.cu; every buffer at its largest)"""
    n, ldg = int(n_pools), (int(n_pools) + 3) & ~3
    cap = -(-max(int(columns), 1) // 16) * 16  # pg_kin_open rounds up to kKC = 16 columns
    nt = -(-ldg // 128)
    ntiles = nt * (nt + 1) // 2
    tile = 128 * 128 * 8
    # G (+ one tile of slack) and K
    total = (cap * ldg + 128) * 8 + n * n * 8
    # Gram workspace: one partial tile per (column slice, tile); slices of >= 16 columns, ~8 waves over the SMs
    total += min(-(-8 * sm_count // ntiles), cap // 16) * ntiles * tile
    # eigen step: the matrix, the eigenvalues, syevd's workspace (1 + 6 n + 2 n^2 doubles), info
    total += n * n * 8 + n * 8 + (1 + 6 * n + 2 * n * n) * 8 + 4
    # loader scratch of one text block (max_loci loci of six columns) and the device parser's buffers
    L = _max_loci(block_bytes, n)
    total += L * 4 + (L + 1) * 8 + L * 6 * 8 + L * 6 + (8 * L + (64 << 10)) + L * 6 * n * 4 + n * 8
    nb = block_bytes + 1
    total += _grow(nb + 32, 1) + _grow(nb, 4) + _grow(-(-nb // 4096) + 1, 8)
    total += nb * (4 + 1 + 4 + 8) + (nb // 256 + 2) * 4 + 2 * L * 8 + (8 * nb // 4096 + (64 << 10)) + 16
    # records [3][k][columns] on the device and pinned, the list of deferred columns (one entry per column and
    # phenotype pass), the partial sums of the DMMA scan's pool passes, Q and y~, the Student-t table, the MLE moments
    total += 2 * 3 * k * cap * 8 + (cap * k + 2) * 8 + -(-cap // 8) * 17 * 64
    total += (n + 1 + k) * ldg * 8 + (8 << 20) + ((13 + k) * ldg + 13 + 2 * 13 * 13 + k * 15) * 8
    return total


def kin_block_columns(device_bytes: int, n_pools: int, k: int, block_bytes: int, sm_count: int) -> int:
    """the most columns a handle can hold within device_bytes (kin_device_bytes), 0 if not even one"""
    lo, hi = 0, max(int(device_bytes), 0) // ((n_pools + 3 & ~3) * 8) + 16
    while lo < hi:  # kin_device_bytes grows with the columns: the largest count that fits
        mid = (lo + hi + 1) // 2
        if kin_device_bytes(n_pools, mid, k, block_bytes, sm_count) <= device_bytes:
            lo = mid
        else:
            hi = mid - 1
    return lo


def _chr_index(block, off, index_of: dict) -> np.ndarray:
    """uint32 chromosome index of the lines that start at `off` in block (uint8): the name is the text up to the
    line's first tab, numbered in order of first appearance in index_of (name -> index), which spans the blocks"""
    end = np.array(off, dtype=np.int64)
    todo = np.arange(end.size)
    while todo.size:  # every name to its tab at once, a byte a step (a locus line holds tabs)
        todo = todo[block[end[todo]] != 9]
        end[todo] += 1
    mv = memoryview(block)
    return np.array([index_of.setdefault(mv[a:b].tobytes(), len(index_of))
                     for a, b in zip(np.asarray(off, dtype=np.int64).tolist(), end.tolist())], dtype=np.uint32)


class _Labels:
    """labels of the loaded loci over the text blocks of a file, in file order"""

    def __init__(self):
        self.index_of = {}
        self.chr_index, self.positions, self.col_locus, self.col_allele = [], [], [], []
        self.base = 0

    def add(self, block, L, off, pos, loc, alle):
        self.chr_index.append(_chr_index(block, off, self.index_of))
        self.positions.append(pos)
        self.col_locus.append(loc + self.base)
        self.col_allele.append(alle)
        self.base += L

    def finish(self) -> _LoadedColumns:
        cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
        return _LoadedColumns(cat(self.col_locus, np.int64), cat(self.col_allele, np.uint8), list(self.index_of),
                              cat(self.chr_index, np.uint32), cat(self.positions, np.uint64))


def _count_columns_bound(fname: str) -> int:
    """an upper bound of the allele columns LoadAll can emit: six per line"""
    with open(fname, "rb") as fh:
        lines = sum(chunk.count(b"\n") for chunk in iter(lambda: fh.read(1 << 24), b"")) + 1
    return _COLS_PER_LINE * lines


_FMT_CHUNK_BYTES = 16 << 20  # rows per device formatter call: each of the two pinned buffers holds this many bytes


def _kept_lines(block, at: int, off, pos, loc, index_of: dict):
    """pass 1 of sync2csv over one text block: for every locus that emitted columns, the absolute byte offset of its
    line, the bytes pass 2 gathers for it (its line, plus a newline where the file's last line has none), its
    chromosome index, its position and its column count"""
    keep, cols = np.unique(loc, return_counts=True)  # the loader emits columns grouped by ascending locus
    o = off[keep].astype(np.int64)
    nl = np.flatnonzero(block == 10)
    k = np.searchsorted(nl, o)
    ends = nl[np.minimum(k, nl.size - 1)] + 1 if nl.size else np.zeros(o.size, np.int64)
    ends = np.where(k < nl.size, ends, block.size)
    size = ends - o + (ends == block.size) * int(block[-1] != 10)
    return at + o, size, _chr_index(block, o, index_of), pos[keep], cols


def write_csv(self, ctx: Context, filter_stats: FilterStats, keep_p_minus_1: bool, out: str, n_threads: int,
              block_bytes: int = 32 << 20, timings: dict = None) -> str:
    """sync2csv: `SaveCsv::write_csv(&self, &FilterStats, keep_p_minus_1, out, n_threads)` of FileSyncPhen
    (src/base/sync.rs:1182-1262): header `#chr,pos,allele,<pool names>`, one row per kept allele of every kept locus,
    loci in LoadAll's order (stable by chromosome, position), frequencies through parse_f64_roundup_and_own(x, 6).

    One code path for any file size; the kinship handle holds one text block's columns at most.  Pass 1 loads every
    text block on the device and keeps, per locus that emits columns, where its line is, its chromosome, position and
    column count; no column leaves the device.  The loci are sorted on the host (pg_sort_loci).  Pass 2 gathers the
    kept lines in that order into line-aligned blocks of at most block_bytes (contiguous runs of the file in one
    read), loads each block again, checks that every line gives its pass-1 column count, and formats the rows on the
    device into two pinned buffers in turn; a writer thread writes one while the next is formatted.  The rows of a
    block are the sorted loci's rows: within a locus, the columns keep the loader's order.
    `timings` (measurement only): filled with wall seconds per phase."""
    if out == "":
        out = _default_out(self.filename_sync, "allele_frequencies")
    if os.path.exists(out):
        raise PgError("Cannot write to output file")
    fname = self.filename_sync
    n = len(self.pool_names)
    max_loci = _max_loci(block_bytes, n)
    clock = time.perf_counter
    tm = {"pass1_s": 0.0, "sort_s": 0.0, "gather_s": 0.0, "parse_s": 0.0, "format_s": 0.0, "write_wait_s": 0.0}
    kin = capi.Kinship(ctx, n, text_block_columns(block_bytes, n))
    pinned = []
    try:
        t0 = clock()
        index_of, parts = {}, []
        for at, block in _line_blocks(fname, 0, os.path.getsize(fname), block_bytes, [np.empty(block_bytes, np.uint8)]):
            kin.reset()
            _L, off, pos, loc, _alle = kin.append_sync_text(block, filter_stats, max_loci, keep_p_minus_1)
            if loc.size:
                parts.append(_kept_lines(block, at, off, pos, loc, index_of))
        if not parts:
            raise PgError("No data passed the filtering variables. Please decrease minimum depth, and/or minimum "
                          "allele frequency.")  # assert at src/base/sync.rs:1219
        line_at, size, chr_idx, positions, cols = (np.concatenate(x) for x in zip(*parts))
        del parts
        tm["pass1_s"] = clock() - t0
        t0 = clock()
        order = capi.sort_loci(positions, chr_names=list(index_of), chr_index=chr_idx)
        line_at, size, positions, cols = line_at[order], size[order], positions[order], cols[order]
        tm["sort_s"] = clock() - t0
        row_max = max(map(len, index_of)) + 25 + 19 * n  # chr,pos,allele + n numbers of at most 19 bytes + newline
        bufs = []
        for _ in range(2):
            arr, h = ctx.pinned_empty((max(_FMT_CHUNK_BYTES, row_max),), np.uint8)
            pinned.append(h)
            bufs.append(arr)
        _sync2csv_pass2(kin, fname, out, self.pool_names, filter_stats, keep_p_minus_1, block_bytes, max_loci,
                        line_at, size, positions, cols, bufs, tm)
    finally:
        kin.close()
        for h in pinned:
            ctx.pinned_free(h)
    if timings is not None:
        timings.update(tm, loci=int(cols.size), columns=int(cols.sum()))
    return out


def _sync2csv_pass2(kin, fname, out, pool_names, fs, keep_p_minus_1, block_bytes, max_loci, line_at, size, positions,
                    cols, bufs, tm):
    """pass 2 of write_csv over the loci in output order; the output file is removed again if anything fails"""
    clock = time.perf_counter
    cum = np.cumsum(size)
    # the lines [i, j) of a run are contiguous in the file
    brk = np.flatnonzero(line_at[1:] != line_at[:-1] + size[:-1]) + 1
    writer = ThreadPoolExecutor(max_workers=1)
    pending = [None, None]
    fo = open(out, "xb")
    try:
        fo.write(capi.format_frequency_header(pool_names))
        with open(fname, "rb") as fh:
            i, N, b = 0, int(size.size), 0
            while i < N:
                t0 = clock()
                j = int(np.searchsorted(cum, (cum[i - 1] if i else 0) + block_bytes, side="right"))
                if j == i:
                    raise PgError(f"a line of {fname} is longer than the block size {block_bytes}")
                block = bytearray()
                starts = [i] + brk[np.searchsorted(brk, i, side="right"):np.searchsorted(brk, j)].tolist() + [j]
                for s, e in zip(starts[:-1], starts[1:]):
                    want = int(line_at[e - 1] + size[e - 1] - line_at[s])
                    fh.seek(int(line_at[s]))
                    data = fh.read(want)
                    if len(data) == want - 1 and not data.endswith(b"\n") and not fh.read(1):
                        data += b"\n"  # the file's last line, which has no newline
                    if len(data) != want:
                        raise PgError(f"{fname} changed between passes: {len(data)} of the {want} bytes at offset "
                                      f"{int(line_at[s])}")
                    block += data
                tm["gather_s"] += clock() - t0
                t0 = clock()
                kin.reset()
                try:
                    L, _off, pos, loc, _alle = kin.append_sync_text(block, fs, max_loci, keep_p_minus_1)
                except PgError as e:  # these lines parsed in pass 1
                    raise PgError(f"{fname} changed between passes: {e}") from None
                tm["parse_s"] += clock() - t0
                got = np.bincount(loc, minlength=L) if loc.size else np.zeros(L, np.int64)
                if L != j - i or not np.array_equal(got, cols[i:j]) or not np.array_equal(pos, positions[i:j]):
                    raise PgError(f"{fname} changed between passes: the {j - i} kept lines from offset "
                                  f"{int(line_at[i])} on no longer give the loci and columns of pass 1")
                P, first = int(loc.size), 0
                while first < P:
                    if pending[b] is not None:
                        t0 = clock()
                        pending[b].result()
                        tm["write_wait_s"] += clock() - t0
                    t0 = clock()
                    nb, nr = kin.format_frequency_rows(first, P - first, bufs[b])
                    tm["format_s"] += clock() - t0
                    pending[b] = writer.submit(fo.write, memoryview(bufs[b])[:nb])
                    first += nr
                    b ^= 1
                i = j
        t0 = clock()
        for p in pending:
            if p is not None:
                p.result()
        tm["write_wait_s"] += clock() - t0
        fo.close()
    except BaseException:
        writer.shutdown(wait=True)
        fo.close()
        os.remove(out)
        raise
    writer.shutdown(wait=True)


def _iter_with_kinship(self, ctx: Context, filter_stats: FilterStats, keep_p_minus_1: bool,
                       xxt_eigen_variance_explained: float, out: str, n_threads: int, block_bytes: int, method: str,
                       device_bytes: int = None, timings: dict = None) -> str:
    """One code path for any file size.  The handle holds up to the columns `device_bytes` allows (None: the free device
    memory less a reserve for the library's fixed allocations).  Pass 1 loads text blocks into the handle and, before
    a block whose column bound does not fit, forms the Gram matrix of what is resident (pg_kin_gram on the first device
    block, pg_kin_gram_accumulate on the later ones) and resets the columns.  The eigen step runs once over the sum.
    With more than one device block, pass 2 scans the block still resident, then re-reads the byte ranges of the others
    and scans them; their records go to their columns' place.  With one block this is load, Gram, eigen step, scan.
    `timings` (measurement only): filled with wall seconds per phase; the stream is synchronised after every Gram."""
    if out != "" and os.path.exists(out):
        raise PgError("Cannot write to output file")
    if np.isnan(self.phen_matrix).any():
        raise PgError("pools with missing phenotypes: remove them before the scan (the reference's remove_missing, "
                      "src/gwas/ols.rs:286)")
    n = len(self.pool_names)
    k = int(np.asarray(self.phen_matrix).reshape(n, -1).shape[1])
    sm_count = ctx.info()["sm_count"]
    if device_bytes is None:
        device_bytes = ctx.mem_info()[0] - _KIN_RESERVE_BYTES
    file_cols = _count_columns_bound(self.filename_sync)
    need = min(text_block_columns(block_bytes, n), file_cols)
    cap = min(kin_block_columns(device_bytes, n, k, block_bytes, sm_count), file_cols)
    if cap < need:
        raise PgError(f"device_bytes {device_bytes} cannot hold one text block of {block_bytes} bytes: its "
                      f"{need} columns take {kin_device_bytes(n, need, k, block_bytes, sm_count)} bytes")
    max_loci = _max_loci(block_bytes, n)
    clock = time.perf_counter
    tm = {"pass1_load_s": 0.0, "pass1_gram_s": 0.0, "eig_s": 0.0, "pass2_load_s": 0.0, "scan_s": 0.0}
    kin = capi.Kinship(ctx, n, cap)
    lab = _Labels()
    dev_blocks = [[]]  # per device block: (byte offset, bytes, columns) of its text blocks
    try:
        def flush():
            t0 = clock()
            kin.gram(accumulate=len(dev_blocks) > 1)
            if timings is not None:
                kin.partial_device_ptr()  # synchronises the handle's stream
            tm["pass1_gram_s"] += clock() - t0

        for at, block in _line_blocks(self.filename_sync, 0, os.path.getsize(self.filename_sync), block_bytes,
                                      [np.empty(block_bytes, np.uint8)]):
            if kin.columns + text_block_columns(block.size, n, int(np.count_nonzero(block == 10))) > cap:
                flush()
                kin.reset()
                dev_blocks.append([])
            t0 = clock()
            L, off, pos, loc, alle = kin.append_sync_text(block, filter_stats, max_loci, keep_p_minus_1)
            tm["pass1_load_s"] += clock() - t0
            lab.add(block, L, off, pos, loc, alle)
            dev_blocks[-1].append((at, block.size, int(loc.size)))
        ld = lab.finish()
        P = int(ld.col_locus.size)
        if P == 0:
            raise PgError("No data passed the filtering variables.")
        flush()
        t0 = clock()
        n_eigenvecs = kin.eig_select(P, float(xxt_eigen_variance_explained))
        tm["eig_s"] = clock() - t0
        scan = kin.covar_scan if method == "ols" else kin.mle_scan
        if len(dev_blocks) == 1:
            t0 = clock()
            beta, _var, pval = scan(self.phen_matrix)   # [k, P] in file order
            tm["scan_s"] = clock() - t0
        else:
            beta, pval = np.empty((k, P)), np.empty((k, P))
            offsets = np.cumsum([0] + [sum(c for _, _, c in tb) for tb in dev_blocks])
            order = [len(dev_blocks) - 1] + list(range(len(dev_blocks) - 1))  # the last block is still resident
            with open(self.filename_sync, "rb") as fh:
                for d in order:
                    if d != order[0]:
                        t0 = clock()
                        kin.reset()
                        for at, nbytes, cols in dev_blocks[d]:
                            fh.seek(at)
                            block = fh.read(nbytes)
                            got = kin.append_sync_text(block, filter_stats, max_loci, keep_p_minus_1)[3].size
                            if len(block) != nbytes or got != cols:
                                raise PgError(f"{self.filename_sync} changed between passes: the {nbytes} bytes at "
                                              f"offset {at} gave {got} columns, {cols} before")
                        tm["pass2_load_s"] += clock() - t0
                    t0 = clock()
                    b, _var, pv = scan(self.phen_matrix)
                    tm["scan_s"] += clock() - t0
                    beta[:, offsets[d]:offsets[d + 1]] = b
                    pval[:, offsets[d]:offsets[d + 1]] = pv
    finally:
        kin.close()
    t0 = clock()
    # the matrix columns follow the loci sorted by (chromosome, position): permute the records into that order
    order = capi.sort_loci(ld.positions, chr_names=ld.chr_names, chr_index=ld.chr_index)
    first = np.full(int(ld.positions.size) + 1, -1, dtype=np.int64)
    count = np.zeros(int(ld.positions.size) + 1, dtype=np.int64)
    for c, l in enumerate(ld.col_locus):
        if first[l] < 0:
            first[l] = c
        count[l] += 1
    seq = np.concatenate([np.arange(first[l], first[l] + count[l]) for l in order if first[l] >= 0]).astype(np.int64)
    names = [n.decode() for n in ld.chr_names]
    chromosome = ["intercept"] + [names[ld.chr_index[ld.col_locus[c]]] for c in seq]
    position = [0] + [int(ld.positions[ld.col_locus[c]]) for c in seq]
    allele = ["intercept"] + [capi.ALLELE_NAMES[ld.col_allele[c]] for c in seq]
    rows = capi.format_kinship_rows(chromosome, position, allele, beta[:, seq], pval[:, seq], n_threads=max(1, n_threads))
    if out == "":  # src/gwas/ols.rs:374-398, src/gwas/mle.rs:409-433
        bname = ".".join(self.filename_sync.split(".")[:-1])
        out = f"{bname}-{method}_iterative_xxt_{n_eigenvecs + 1}_eigens-{time.time()}.csv"
    with open(out, "xb") as fo:
        fo.write(capi.format_header(capi.KIND_OLS_KINSHIP))
        fo.write(rows)
    if timings is not None:
        tm["write_s"] = clock() - t0
        tm["device_blocks"] = len(dev_blocks)
        tm["columns"] = P
        tm["capacity"] = cap
        timings.update(tm)
    return out


def ols_iter_with_kinship(self, ctx: Context, filter_stats: FilterStats, keep_p_minus_1: bool,
                          xxt_eigen_variance_explained: float, out: str, n_threads: int,
                          block_bytes: int = 32 << 20, device_bytes: int = None) -> str:
    """`poolgen ols_iter_with_kinship` (src/main.rs:280-298): into_genotypes_and_phenotypes (src/base/sync.rs:1106-1179)
    then ols_with_covariate (src/gwas/ols.rs:278-436) and its writer, including the label indexing of
    src/gwas/ols.rs:421-424 (row i of the allele columns carries entry i of the label vectors, whose entry 0 is the
    intercept's)"""
    return _iter_with_kinship(self, ctx, filter_stats, keep_p_minus_1, xxt_eigen_variance_explained, out, n_threads,
                              block_bytes, "ols", device_bytes)


def mle_iter_with_kinship(self, ctx: Context, filter_stats: FilterStats, keep_p_minus_1: bool,
                          xxt_eigen_variance_explained: float, out: str, n_threads: int,
                          block_bytes: int = 32 << 20, device_bytes: int = None) -> str:
    """`poolgen mle_iter_with_kinship` (src/main.rs:316-326): the same loader, then mle_with_covariate
    (src/gwas/mle.rs:307-463) -- kinship matrix, PCs by the same rule, one maximum-likelihood fit per column and
    phenotype -- and its writer (same header and row layout, labels indexed the same way, mle.rs:449-460)"""
    return _iter_with_kinship(self, ctx, filter_stats, keep_p_minus_1, xxt_eigen_variance_explained, out, n_threads,
                              block_bytes, "mle", device_bytes)


FileSyncPhen.write_csv = write_csv
FileSyncPhen.ols_iter_with_kinship = ols_iter_with_kinship
FileSyncPhen.mle_iter_with_kinship = mle_iter_with_kinship
