"""sync2csv at any file size: the device formatter of frequency rows (pg_kin_format_frequency_rows) against the host's
pg_format_frequency_rows, and the two-pass FileSyncPhen.write_csv against rows built from the oracle's loader, with
its memory bound to one text block."""
import os

import numpy as np
import pytest

import poolgen_b200 as pb
from oracle import pgo
from poolgen_b200 import capi, sync_io
from tests import helpers as H

pytestmark = pytest.mark.gpu


def _sync_lines(counts, chroms, positions):
    """counts [L, 6, n] -> sync lines (no newline)"""
    out = []
    for l in range(counts.shape[0]):
        pools = "\t".join(":".join(str(int(v)) for v in counts[l, :, i]) for i in range(counts.shape[2]))
        out.append(f"{chroms[l]}\t{positions[l]}\tN\t{pools}")
    return out


def _formatter_counts(rng, n, L):
    """[L, 6, n] counts whose frequencies cover 0, 1, NaN (pools without coverage), the doubles nearest to and just
    beside the ties (k + 0.5) / 1e6, and random ratios"""
    c = np.zeros((L, 6, n), dtype=np.uint64)
    for l in range(L):
        kind = l % 5
        if kind == 0:  # random small counts over all six alleles: zeros, ones, short ratios
            c[l] = rng.integers(0, 6, (6, n)) * (rng.random((6, n)) < 0.6)
        elif kind == 1:  # exact ties (2k + 1) / 2e6 and their neighbours ((2k + 1) m +- 1) / (2e6 m)
            k = rng.integers(0, 10 ** 6, n)
            m = rng.choice([1, 1000, 2000], n)
            d = rng.choice([-1, 0, 1], n) * (m > 1)
            a = (2 * k + 1) * m + d
            c[l, 0], c[l, 1] = a, 2_000_000 * m - a
        elif kind == 2:  # large random depths: long ratios
            c[l, :4] = rng.integers(0, 1 << 30, (4, n))
        elif kind == 3:  # one allele per pool (frequencies 0 and 1), some pools without coverage (NaN)
            a = rng.integers(0, 6, n)
            c[l, a, np.arange(n)] = rng.integers(1, 50, n)
            c[l, :, rng.random(n) < 0.2] = 0
        else:  # biallelic, tiny minor counts
            c[l, 2] = rng.integers(0, 3, n)
            c[l, 3] = rng.integers(1_000_000, 4_000_000_000, n)
        c[l, :, 0] += (c[l, :, 0].sum() == 0)  # the first pool keeps some coverage
    return c


def _chrom_names(rng, L):
    """1 to 200 bytes, some a prefix of another"""
    base = ["c", "chr", "chr1", "chr10", "chr1_random", "X" * 200, "X" * 199, "scaffold_" + "7" * 150]
    return [base[i] if i < len(base) else "s" + "".join(rng.choice(list("abcXYZ0129_"), int(rng.integers(0, 199))))
            for i in rng.integers(0, len(base) + 4, L)]


@pytest.mark.parametrize("n", [2, 5, 31, 32, 33, 100, 1000, 2000, 4099])
def test_device_rows_equal_the_host_rows(ctx, n):
    rng = np.random.default_rng(n)
    L = max(10, min(200, 200_000 // n))
    counts = _formatter_counts(rng, n, L)
    chroms = _chrom_names(rng, L)
    pos = [int(p) for p in rng.integers(0, 1 << 62, L)]
    pos[0], pos[1 % L] = 0, 2 ** 64 - 1
    text = ("\n".join(_sync_lines(counts, chroms, pos)) + "\n").encode()
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), remove_ns=False, min_coverage_depth=0,
                        min_allele_frequency=0.0, max_missingness_rate=1.0)
    kin = pb.Kinship(ctx, n, 6 * L)
    try:
        nl, off, p, loc, alle = kin.append_sync_text(text, fs, L)
        P = kin.columns
        assert nl == L and P == loc.size and P >= L and set(alle.tolist()) == set(range(6))
        G = kin.get_columns(0, P)
        assert np.isnan(G).any() and (G == 0).any() and (G == 1).any()
        host = pb.format_frequency_rows(G, loc, alle, p, text=text, line_offsets=off)
        buf = np.empty(len(host) + 64, np.uint8)
        nb, nr = kin.format_frequency_rows(0, P, buf)
        assert (nb, nr) == (len(host), P)
        assert bytes(buf[:nb]) == host
        # a capacity of a few rows: whole rows only, then the rest from where the call stopped
        rows = host.splitlines(keepends=True)
        small = np.empty(2 * max(len(r) for r in rows) + 1, np.uint8)
        fit = int(np.searchsorted(np.cumsum([len(r) for r in rows]), small.size, side="right"))
        nb, nr = kin.format_frequency_rows(0, P, small)
        assert fit >= 2 and (nr, bytes(small[:nb])) == (fit, b"".join(rows[:fit]))
        got, first = [], 0
        while first < P:
            nb, nr = kin.format_frequency_rows(first, P - first, small)
            assert nr >= 1
            got.append(bytes(small[:nb]))
            first += nr
        assert b"".join(got) == host
        # a sub-range: the rows of those columns
        nb, nr = kin.format_frequency_rows(3, 4, buf)
        assert bytes(buf[:nb]) == b"".join(rows[3:7]) and nr == 4
        # a capacity below one row is refused
        with pytest.raises(pb.PgError, match=r"\(-1\)"):
            kin.format_frequency_rows(0, P, np.empty(len(rows[0]) - 1, np.uint8))
        with pytest.raises(pb.PgError, match=r"\(-1\)"):
            kin.format_frequency_rows(P - 1, 2, buf)
    finally:
        kin.close()


def test_formatter_needs_a_text_append(ctx):
    n = 4
    kin = pb.Kinship(ctx, n, 64)
    buf = np.empty(1 << 16, np.uint8)
    try:
        with pytest.raises(pb.PgError, match=r"\(-3\)"):  # nothing appended yet
            kin.format_frequency_rows(0, 0, buf)
        # a column outside the loader's range (|x * 1e6| >= 9e14), appended as numbers: not text
        kin.append_columns(np.array([[0.5, 9e8, 1.0, float("inf")]]))
        with pytest.raises(pb.PgError, match=r"\(-3\)"):
            kin.format_frequency_rows(0, 1, buf)
        text = b"chr1\t7\tA\t" + b"\t".join([b"1:2:0:0:0:0"] * n) + b"\n"
        fs = pb.FilterStats(pool_sizes=np.full(n, 0.25), min_allele_frequency=0.0)
        kin.append_sync_text(text, fs, 4)
        nb, nr = kin.format_frequency_rows(0, 2, buf)   # the text's two columns, after the appended one
        assert bytes(buf[:nb]) == b"chr1,7,A" + b",0.333333" * n + b"\nchr1,7,T" + b",0.666667" * n + b"\n"
        kin.reset()
        with pytest.raises(pb.PgError, match=r"\(-3\)"):
            kin.format_frequency_rows(0, 0, buf)
    finally:
        kin.close()


# ---- file level ---------------------------------------------------------------------------------------------------
def _c1_file(tmp_path, L=2400, last_newline=False):
    """C1's counts as a sync file that exercises LoadAll's order and the reader: chromosomes shuffled (chr1, chr10,
    chr9), positions that decrease within a chromosome, duplicate (chromosome, position) pairs, CRLF lines, comment lines,
    a line whose position is not an integer, no newline after the last line.  Returns (path, counts, chroms, pos) of
    the locus lines."""
    c1 = H.load_c1()
    counts = c1["counts"][:L]
    names = ["chr1", "chr10", "chr9"]
    chroms = [names[(l * 7 // 50) % 3] for l in range(L)]
    pos = [int(10_000 - (l % 900) * 3) for l in range(L)]
    for l in range(0, L, 97):  # duplicates of the previous locus' (chromosome, position)
        if l:
            chroms[l], pos[l] = chroms[l - 1], pos[l - 1]
    lines = _sync_lines(counts, chroms, pos)
    out = []
    for l, ln in enumerate(lines):
        if l % 31 == 5:
            out.append("#a comment\n")
        if l % 53 == 7:
            out.append("chr1\tnot_a_number\tN\t" + "\t".join(["1:2:3:4:0:0"] * 5) + "\r\n")
        out.append(ln + ("\r\n" if l % 3 == 1 else "\n"))
    if not last_newline:
        out[-1] = out[-1].rstrip("\r\n")
    path = str(tmp_path / "t.sync")
    with open(path, "w", newline="") as fh:
        fh.write("".join(out))
    return path, counts, chroms, pos


def _expected(counts, chroms, pos, fs, keep_p_minus_1, names):
    from tests.test_writer import _oracle_sync2csv_rows
    ocols, olabels = pgo.load_columns(counts.transpose(0, 2, 1).astype(np.uint64), np.arange(6, dtype=np.uint8),
                                      H.oracle_fs(fs), keep_p_minus_1)
    head = "#chr,pos,allele," + ",".join(names) + "\n"
    return head + _oracle_sync2csv_rows(ocols, olabels, chroms, pos), len(olabels)


@pytest.mark.parametrize("keep_p_minus_1", [False, True])
def test_write_csv_many_blocks_equals_the_oracle_rows(ctx, tmp_path, keep_p_minus_1):
    path, counts, chroms, pos = _c1_file(tmp_path)
    names = ["G1", "G2", "G3", "G4", "G5"]
    sizes = np.full(5, 0.2)
    fs = pb.FilterStats(pool_sizes=sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(path, names, sizes, np.zeros((5, 1)), "sync2csv")
    timings = {}
    out = src.write_csv(ctx, fs, keep_p_minus_1, str(tmp_path / "freq.csv"), 2, block_bytes=6 << 10, timings=timings)
    expect, P = _expected(counts, chroms, pos, fs, keep_p_minus_1, names)
    got = open(out, "rb").read().decode()
    assert got == expect and P > 1000
    assert timings["columns"] == P and timings["loci"] < len(pos)   # some loci were filtered out
    with pytest.raises(pb.PgError, match="Cannot write"):
        src.write_csv(ctx, fs, keep_p_minus_1, out, 2, block_bytes=6 << 10)
    auto = src.write_csv(ctx, fs, keep_p_minus_1, "", 2)  # default name, one block
    assert auto.startswith(str(tmp_path / "t-")) and auto.endswith("-allele_frequencies.csv")
    assert open(auto, "rb").read().decode() == expect


def test_write_csv_keep_ns_six_columns(ctx, tmp_path):
    """--keep-ns with MAF 0: loci emit six columns (the loader's largest), with and without a last newline"""
    for last_newline in (True, False):
        d = tmp_path / str(last_newline)
        d.mkdir()
        path, counts, chroms, pos = _c1_file(d, L=900, last_newline=last_newline)
        counts = counts.copy()
        counts[::4, :, 0] += 1  # every allele seen: six columns
        with open(path, "rb") as fh:
            raw = fh.read()
        # rewrite the locus lines with the changed counts (same layout, comments and CRLF kept)
        lines = raw.split(b"\n")
        body = [i for i, ln in enumerate(lines) if ln and not ln.startswith(b"#") and b"not_a_number" not in ln]
        new = _sync_lines(counts, chroms, pos)
        for i, ln in zip(body, new):
            lines[i] = ln.encode() + (b"\r" if lines[i].endswith(b"\r") else b"")
        with open(path, "wb") as fh:
            fh.write(b"\n".join(lines))
        names = ["G1", "G2", "G3", "G4", "G5"]
        fs = pb.FilterStats(pool_sizes=np.full(5, 0.2), remove_ns=False, min_coverage_depth=0, min_allele_frequency=0.0,
                            max_missingness_rate=1.0)
        src = pb.FileSyncPhen(path, names, np.full(5, 0.2), np.zeros((5, 1)), "sync2csv")
        out = src.write_csv(ctx, fs, False, str(d / "freq.csv"), 1, block_bytes=4 << 10)
        expect, P = _expected(counts, chroms, pos, fs, False, names)
        assert open(out, "rb").read().decode() == expect
        assert P > 6 * 225 and expect.count(",N,") and expect.count(",D,")


def test_write_csv_memory_is_one_text_block(ctx, tmp_path, monkeypatch):
    """the handle is never opened for more than one text block's columns and no column is copied to the host, for
    any file size"""
    seen = []

    class Recording(capi.Kinship):
        def __init__(self, ctx, n_pools, max_columns):
            seen.append(int(max_columns))
            super().__init__(ctx, n_pools, max_columns)

        def get_columns(self, first, count):
            raise AssertionError("write_csv copied columns to the host")

    monkeypatch.setattr(sync_io.capi, "Kinship", Recording)
    path, counts, chroms, pos = _c1_file(tmp_path)
    fs = pb.FilterStats(pool_sizes=np.full(5, 0.2), min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(path, ["a", "b", "c", "d", "e"], np.full(5, 0.2), np.zeros((5, 1)), "sync2csv")
    for bb in (4 << 10, 16 << 10):
        src.write_csv(ctx, fs, True, str(tmp_path / f"o{bb}.csv"), 1, block_bytes=bb)
        assert seen and max(seen) <= sync_io.text_block_columns(bb, 5) < 6 * len(pos) // 4
        seen.clear()
    # the file's size does not move the bound
    big = str(tmp_path / "big.sync")
    with open(big, "wb") as fo:
        for _ in range(4):
            fo.write(open(path, "rb").read() + b"\n")
    src.filename_sync = big
    src.write_csv(ctx, fs, True, str(tmp_path / "big.csv"), 1, block_bytes=4 << 10)
    assert max(seen) <= sync_io.text_block_columns(4 << 10, 5)


def test_write_csv_refuses_a_file_changed_between_passes(ctx, tmp_path, monkeypatch):
    path, counts, chroms, pos = _c1_file(tmp_path)
    fs = pb.FilterStats(pool_sizes=np.full(5, 0.2), min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(path, ["a", "b", "c", "d", "e"], np.full(5, 0.2), np.zeros((5, 1)), "sync2csv")
    original = open(path, "rb").read()
    real_sort = capi.sort_loci

    def edit(change):
        def sort_then_change(*a, **kw):
            with open(path, "wb") as fh:
                fh.write(change(original))
            return real_sort(*a, **kw)
        return sort_then_change

    lines = original.split(b"\n")
    body = [i for i, ln in enumerate(lines) if ln and not ln.startswith(b"#") and b"not_a_number" not in ln]
    zeroed = list(lines)
    zeroed[body[10]] = b"\t".join(lines[body[10]].split(b"\t")[:3] + [b"0:0:0:0:0:0"] * 5)  # same line, filtered now
    shifted = list(lines)
    shifted[body[3]] = b"#" + lines[body[3]]  # one byte more: every later line moves
    for change in (lambda b: b[:len(b) // 2], lambda b: b"\n".join(zeroed), lambda b: b"\n".join(shifted)):
        monkeypatch.setattr(capi, "sort_loci", edit(change))
        out = str(tmp_path / "changed.csv")
        with pytest.raises(pb.PgError, match="changed between passes"):
            src.write_csv(ctx, fs, False, out, 1, block_bytes=8 << 10)
        assert not os.path.exists(out)
        with open(path, "wb") as fh:
            fh.write(original)
    monkeypatch.setattr(capi, "sort_loci", real_sort)
    # nothing passes the filter: the reference's error, and no output file
    strict = pb.FilterStats(pool_sizes=np.full(5, 0.2), min_coverage_depth=10 ** 9)
    out = str(tmp_path / "none.csv")
    with pytest.raises(pb.PgError, match="No data passed"):
        src.write_csv(ctx, strict, False, out, 1)
    assert not os.path.exists(out)
