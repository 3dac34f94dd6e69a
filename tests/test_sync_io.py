"""File-level mirror of the reference's readers (poolgen_b200/sync_io.py): FilePhen::lparse, find_file_splits on the CPU,
FileSyncPhen / FileSync::read_analyse_write on the GPU."""
import json
import os

import numpy as np
import pytest

import poolgen_b200 as pb
from tests import helpers as H


def _write_c1_phen(path):
    with open(os.path.join(H.HERE, "golden", "c1_phen.json")) as fh:
        ph = json.load(fh)
    lines = ["#name,poolSizes,Trait_A,Trait_B"]
    for name, size, row in zip(ph["pool_names"], ph["pool_sizes_raw"], ph["phen"]):
        lines.append(f"{name}, {size:g},{row[0]} ,{row[1]}")
    with open(path, "w") as fh:
        fh.write("\r\n".join(lines) + "\r\n")


def test_file_phen_known_answer(tmp_path):
    # src/base/phen.rs:208-236: tests/test.csv -> names G1..G5, pool sizes 0.2 each, traits columns 2 and 3
    p = str(tmp_path / "test.csv")
    _write_c1_phen(p)
    phen = pb.FilePhen(p, ",", 0, 1, [2, 3]).lparse()
    assert phen.pool_names == ["G1", "G2", "G3", "G4", "G5"]
    assert list(phen.pool_sizes) == [0.2, 0.2, 0.2, 0.2, 0.2]
    assert phen.phen_matrix.T.tolist() == [[0.1, 0.3, 0.5, 0.7, 0.9], [83.2, 75.3, 49.8, 23.9, 12.0]]
    with open(p, "a") as fh:
        fh.write("G6,10,NA,\n")
    phen = pb.FilePhen(p, ",", 0, 1, [2, 3]).lparse()
    assert np.isnan(phen.phen_matrix[5]).all() and abs(phen.pool_sizes.sum() - 1.0) < 1e-15
    assert phen.pool_sizes[5] == 10.0 / 110.0


def test_find_file_splits(tmp_path):
    # src/base/helpers.rs:74-91: split points move to the start of the NEXT line (a full line is skipped even when the
    # raw split already is a line start), duplicates collapse
    p = str(tmp_path / "x.sync")
    lines = [("chr1\t%d\tN\t" % i) + "\t".join(["1:2:3:4:0:0"] * 3) + "\n" for i in range(100)]
    with open(p, "w") as fh:
        fh.writelines(lines)
    size = os.path.getsize(p)
    starts = np.cumsum([0] + [len(l) for l in lines])
    for n_threads in (1, 2, 3, 7):
        s = pb.find_file_splits(p, n_threads)
        assert s[0] == 0 and s[-1] == size and s == sorted(set(s))
        assert all(x in starts for x in s)
        raw = list(range(0, size, size // n_threads)) + [size]
        expect = [0 if r == 0 else int(starts[np.searchsorted(starts, r, side="right")]) if r < size else size for r in raw]
        dedup = [expect[0]] + [b for a, b in zip(expect, expect[1:]) if a != b]
        assert s == dedup
    with pytest.raises(pb.PgError):
        pb.find_file_splits(str(tmp_path / "missing.sync"), 2)


@pytest.mark.gpu
@pytest.mark.parametrize("analysis", ["ols_iter", "pearson_corr", "chisq_test", "fisher_exact_test"])
def test_read_analyse_write_c1(ctx, tmp_path, analysis):
    """`poolgen <analysis> -f tests/test.sync -p tests/test.csv --n-threads 3` through the mirror: three reader threads
    over line-aligned byte ranges, blocks of 48 KB (so lines straddle block ends), rows concatenated in chunk order;
    the file equals header + rows of the same records computed from the parsed counts in one batch"""
    from tests.test_text_gpu import _sync_text
    c1 = H.load_c1()
    names = [str(s) for s in c1["chrom_names"]]
    chroms = [names[i] for i in c1["chrom_idx"]]
    pos = [int(p) for p in c1["pos"]]
    fsync = str(tmp_path / "test.sync")
    with open(fsync, "wb") as fh:
        fh.write(_sync_text(c1["counts"], chroms, pos))
    fphen = str(tmp_path / "test.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=10, min_allele_frequency=0.01)
    out = str(tmp_path / "out.csv")
    if analysis in ("ols_iter", "pearson_corr"):
        fn = pb.ols_iterate if analysis == "ols_iter" else pb.correlation
        src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, analysis)
        y = phen.phen_matrix
    else:
        fn = pb.chisq if analysis == "chisq_test" else pb.fisher
        src = pb.FileSync(fsync, analysis)
        y = None
    got_name = src.read_analyse_write(ctx, fs, out, 3, fn, block_bytes=48 << 10)
    assert got_name == out
    kind = {"ols_iter": pb.KIND_OLS, "pearson_corr": pb.KIND_CORR, "chisq_test": pb.KIND_CHISQ,
            "fisher_exact_test": pb.KIND_FISHER}[analysis]
    scan = pb.Scan(ctx, kind, fs, 5, c1["codes"], y)
    whole = scan.run_counts(c1["counts"])
    scan.close()
    expect = pb.format_header(kind) + pb.format_rows(kind, whole, c1["pos"], chr_names=names, chr_index=c1["chrom_idx"],
                                                     exact_p_pools=5)   # the file-level writer prints the reference's digits of p
    got = open(out, "rb").read()
    assert got == expect and got.count(b"\n") > 1500
    with pytest.raises(pb.PgError):   # create_new(true): the output file must not exist
        src.read_analyse_write(ctx, fs, out, 3, fn)
    # default output name: <sync name without extension>-<seconds>-<test>.csv (src/base/sync.rs:885-903)
    auto = src.read_analyse_write(ctx, fs, "", 2, fn)
    assert auto.startswith(str(tmp_path / "test-")) and auto.endswith(f"-{analysis}.csv")
    assert open(auto, "rb").read() == expect


@pytest.mark.gpu
@pytest.mark.parametrize("keep_p_minus_1", [False, True])
def test_sync2csv_file(ctx, tmp_path, keep_p_minus_1):
    """`poolgen sync2csv -f test.sync -p test.csv [--keep-p-minus-1]` through FileSyncPhen.write_csv: small blocks, the
    chromosomes of the file shuffled so that LoadAll's sort matters; against rows built from the oracle's loader"""
    from oracle import pgo
    from tests.test_text_gpu import _sync_text
    from tests.test_writer import _oracle_sync2csv_rows
    c1 = H.load_c1()
    L = 2500
    counts = c1["counts"][:L]
    names = ["chrB", "chrA", "chr10", "chr9"]
    chroms = [names[(l // 300) % 4] for l in range(L)]
    pos = [int(p) for p in c1["pos"][:L]]
    fsync = str(tmp_path / "t.sync")
    with open(fsync, "wb") as fh:
        fh.write(_sync_text(counts, chroms, pos))
    fphen = str(tmp_path / "t.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, "sync2csv")
    out = src.write_csv(ctx, fs, keep_p_minus_1, str(tmp_path / "freq.csv"), 2, block_bytes=40 << 10)
    got = open(out, "rb").read().decode()
    ocols, olabels = pgo.load_columns(counts.transpose(0, 2, 1).astype(np.uint64), c1["codes"], H.oracle_fs(fs),
                                      keep_p_minus_1)
    expect = "#chr,pos,allele,G1,G2,G3,G4,G5\n" + _oracle_sync2csv_rows(ocols, olabels, chroms, pos)
    assert got == expect and got.count("\n") == len(olabels) + 1 > 1000


@pytest.mark.gpu
def test_ols_iter_with_kinship_file(ctx, tmp_path):
    """`poolgen ols_iter_with_kinship` through FileSyncPhen.ols_iter_with_kinship: rows phenotype-outer / column-inner
    in LoadAll's locus order with the reference's label indexing (row i carries label i of the vectors that start with
    the intercept's entry), numbers against the oracle's ols_with_covariate"""
    from oracle import pgo
    from tests.test_text_gpu import _sync_text
    c1 = H.load_c1()
    L = 1200
    counts = c1["counts"][:L]
    names = ["chrB", "chrA"]
    chroms = [names[(l // 250) % 2] for l in range(L)]
    pos = [int(p) for p in c1["pos"][:L]]
    fsync = str(tmp_path / "k.sync")
    with open(fsync, "wb") as fh:
        fh.write(_sync_text(counts, chroms, pos))
    fphen = str(tmp_path / "k.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, "ols_iter_with_kinship")
    out = src.ols_iter_with_kinship(ctx, fs, True, 0.75, str(tmp_path / "kin.csv"), 2, block_bytes=40 << 10)
    lines = open(out).read().split("\n")
    assert lines[0] == "#chr,pos,alleles,phenotype,statistic,pvalue" and lines[-1] == ""
    rows = [ln.split(",") for ln in lines[1:-1]]
    # oracle: columns in LoadAll's order
    ocols, olabels = pgo.load_columns(counts.transpose(0, 2, 1).astype(np.uint64), c1["codes"], H.oracle_fs(fs), True)
    loci = sorted(range(L), key=lambda l: (chroms[l].encode(), pos[l]))
    by_locus = {}
    for c, (l, a) in enumerate(olabels):
        by_locus.setdefault(l, []).append((c, a))
    seq = [ca for l in loci for ca in by_locus.get(l, [])]
    P = len(seq)
    G = ocols[[c for c, _ in seq]]
    om, ob, ov, op = pgo.ols_with_covariate(G, phen.phen_matrix, 0.75)
    assert len(rows) == 2 * P
    labels = [("intercept", "0", "intercept")] + [(chroms[olabels[c][0]], str(pos[olabels[c][0]]), "ATCGND"[a]) for c, a in seq]
    for j in range(2):
        for i in range(P):
            r = rows[j * P + i]
            assert tuple(r[:3]) == labels[i] and r[3] == f"Pheno_{j}", (r, labels[i])   # the shifted labels of ols.rs:421-424
            for got, exp, tol in ((float(r[4]), ob[i, j], 1e-7), (float(r[5]), op[i, j], 1e-6)):
                assert (np.isnan(got) and np.isnan(exp)) or abs(got - exp) <= tol * max(abs(exp), 1e-3), (r, exp)


@pytest.mark.gpu
def test_mle_iter_with_kinship_file(ctx, tmp_path):
    """`poolgen mle_iter_with_kinship` (src/main.rs:316-326) through FileSyncPhen.mle_iter_with_kinship: the loader and
    the rows of the OLS entry, numbers against the oracle's mle_with_covariate (gwas/mle.rs:307-463) to the simplex
    search's convergence (tests/test_nm_gpu.py states the tolerance)"""
    from oracle import pgo
    from tests.test_text_gpu import _sync_text
    c1 = H.load_c1()
    L = 500
    counts = c1["counts"][:L]
    chroms = ["chr1"] * L
    pos = [int(p) for p in c1["pos"][:L]]
    fsync = str(tmp_path / "m.sync")
    with open(fsync, "wb") as fh:
        fh.write(_sync_text(counts, chroms, pos))
    fphen = str(tmp_path / "m.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, "mle_iter_with_kinship")
    out = src.mle_iter_with_kinship(ctx, fs, True, 0.75, str(tmp_path / "kin_mle.csv"), 2, block_bytes=40 << 10)
    lines = open(out).read().split("\n")
    assert lines[0] == "#chr,pos,alleles,phenotype,statistic,pvalue" and lines[-1] == ""
    rows = [ln.split(",") for ln in lines[1:-1]]
    ocols, olabels = pgo.load_columns(counts.transpose(0, 2, 1).astype(np.uint64), c1["codes"], H.oracle_fs(fs), True)
    loci = sorted(range(L), key=lambda l: (chroms[l].encode(), pos[l]))
    by_locus = {}
    for c, (l, a) in enumerate(olabels):
        by_locus.setdefault(l, []).append((c, a))
    seq = [ca for l in loci for ca in by_locus.get(l, [])]
    P = len(seq)
    G = ocols[[c for c, _ in seq]]
    om, ob, ov, op = pgo.mle_with_covariate(G, phen.phen_matrix, 0.75)
    assert om == 0 and len(rows) == 2 * P and P > 150     # raw frequencies: the first eigenvalue alone crosses 0.75
    labels = [("intercept", "0", "intercept")] + [(chroms[olabels[c][0]], str(pos[olabels[c][0]]), "ATCGND"[a]) for c, a in seq]
    worst = 0.0
    for j in range(2):
        for i in range(P):
            r = rows[j * P + i]
            assert tuple(r[:3]) == labels[i] and r[3] == f"Pheno_{j}", (r, labels[i])
            got_b, got_p = float(r[4]), float(r[5])
            if np.isnan(ob[i, j]):
                assert np.isnan(got_b) and np.isnan(got_p), r
                continue
            eb = abs(got_b - ob[i, j]) / max(abs(ob[i, j]), np.sqrt(ov[i, j]))
            ep = abs(got_p - op[i, j]) / max(op[i, j], 1e-12)
            worst = max(worst, eb, ep)
    assert worst < 1e-3, worst


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["write_csv", "ols_iter_with_kinship"])
def test_file_without_last_newline(ctx, tmp_path, entry):
    """the file-level entries on a file whose last line has no newline: the same output as with the newline, at a
    block size where that line is a block of its own and at one where it joins the block before it"""
    from tests.test_text_gpu import _sync_text
    c1 = H.load_c1()
    L = 1200
    chroms = [["chrB", "chrA"][(l // 250) % 2] for l in range(L)]
    text = _sync_text(c1["counts"][:L], chroms, [int(p) for p in c1["pos"][:L]])
    last = len(text) - 1 - text.rfind(b"\n", 0, len(text) - 1) - 1  # the last line without its newline
    files = {}
    for newline in (True, False):
        files[newline] = str(tmp_path / f"k{int(newline)}.sync")
        with open(files[newline], "wb") as fh:
            fh.write(text if newline else text[:-1])
    layouts = {}  # last line alone in its block -> block size
    for bb in range(32 << 10, 31 << 10, -1):
        sizes = [v.size for _, v in pb.sync_io._line_blocks(files[False], 0, len(text) - 1, bb,
                                                             [np.empty(bb, np.uint8)])]
        layouts.setdefault(len(sizes) > 1 and sizes[-1] == last, bb)
        if len(layouts) == 2:
            break
    assert set(layouts) == {True, False}
    fphen = str(tmp_path / "k.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    outs = {}
    for newline, fsync in files.items():
        src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, entry)
        for alone, bb in layouts.items():
            out = str(tmp_path / f"{entry}_{int(newline)}_{int(alone)}.csv")
            if entry == "write_csv":
                src.write_csv(ctx, fs, False, out, 2, block_bytes=bb)
            else:
                src.ols_iter_with_kinship(ctx, fs, True, 0.75, out, 2, block_bytes=bb)
            outs[newline, alone] = open(out, "rb").read()
    for alone in (True, False):
        assert outs[False, alone] == outs[True, alone] and outs[True, alone].count(b"\n") > 1000
