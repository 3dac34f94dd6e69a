"""Kinship analyses over more columns than one device block: the accumulated Gram matrix (pg_kin_gram_accumulate) and
the two-pass file-level driver of ols_iter_with_kinship / mle_iter_with_kinship (poolgen_b200/sync_io.py).  The
capacity test runs on the CPU; the others need a GPU."""
import os

import numpy as np
import pytest

import poolgen_b200 as pb
from poolgen_b200 import sync_io
from tests import helpers as H

SM_COUNT = 148  # B200


def test_block_capacity_from_a_byte_budget(tmp_path):
    """the columns a handle can hold grow with the budget, their footprint never exceeds it, one more column would,
    and a text block is bounded by six columns per line of at least 12 n + 5 bytes"""
    for n, k, bb in ((5, 2, 40 << 10), (60, 1, 32 << 10), (2000, 1, 32 << 20), (2000, 16, 32 << 20)):
        prev = 0
        for budget in np.unique(np.geomspace(1 << 16, 200 << 30, 60).astype(np.int64)):
            budget = int(budget)
            cap = sync_io.kin_block_columns(budget, n, k, bb, SM_COUNT)
            assert cap >= prev, (n, budget, cap, prev)
            prev = cap
            if cap:
                assert sync_io.kin_device_bytes(n, cap, k, bb, SM_COUNT) <= budget
            assert sync_io.kin_device_bytes(n, cap + 1, k, bb, SM_COUNT) > budget
        # the footprint covers G at ldg x 8 bytes per column at least
        ldg = (n + 3) & ~3
        assert sync_io.kin_device_bytes(n, 10 ** 6, k, bb, SM_COUNT) > 10 ** 6 * ldg * 8
    # 180 GB hold a 10 M-column block at 2,000 pools (C4: 5 M biallelic loci) with 32 MB text blocks
    assert sync_io.kin_block_columns(180 << 30, 2000, 1, 32 << 20, SM_COUNT) > 10_000_000
    # text blocks: six columns per line, lines of at least 12 n + 5 bytes; a known line count tightens the bound
    for n in (2, 5, 2000):
        w = 12 * n + 5
        for nb in (0, w - 1, w, 10 * w + 3, 1 << 20):
            assert sync_io.text_block_columns(nb, n) == 6 * (nb // w + 1)
            assert sync_io.text_block_columns(nb, n, n_lines=1) == min(12, 6 * (nb // w + 1))
        line = "c\t0\tN" + "\t0:0:0:0:0:0" * n + "\n"
        assert len(line) == w + 1
        for lines in (1, 7, 100):
            assert sync_io.text_block_columns(lines * len(line), n) >= 6 * lines
    # the whole-file bound: six per line
    p = tmp_path / "six.sync"
    p.write_bytes(b"a\n" * 41)
    assert sync_io._count_columns_bound(str(p)) == 6 * 42


# ---- device: K accumulated over blocks ----------------------------------------------------------------------------
def _gram_blocks(kin, G, splits):
    """pg_kin_gram on the first block, pg_kin_gram_accumulate on the others; returns K"""
    at = 0
    for i, s in enumerate(splits):
        kin.reset()
        kin.append_columns(G[at:at + s])
        kin.gram(accumulate=i > 0)
        at += s
    assert at == G.shape[0]
    return kin.partial_get()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [40, 257, 2000])
def test_gram_accumulate_matches_numpy(ctx, n):
    rng = np.random.default_rng(n)
    splits = [1, 15, 16, 17, 4093, 33]
    P = sum(splits)
    G = rng.random((P, n))
    kin = pb.Kinship(ctx, n, max(splits))
    K = _gram_blocks(kin, G, splits)
    ref = G.T @ G
    assert np.allclose(K, ref, rtol=1e-12, atol=1e-12 * P)
    assert np.array_equal(K, K.T)
    assert np.array_equal(_gram_blocks(kin, G, splits), K)  # the same split: the same bits
    # a new sequence on other data keeps nothing of the old K
    G2 = rng.random((500, n)) - 0.5
    K2 = _gram_blocks(kin, G2, [100, 17, 383])
    fresh = pb.Kinship(ctx, n, 383)
    assert np.array_equal(_gram_blocks(fresh, G2, [100, 17, 383]), K2)
    fresh.close()
    assert np.allclose(K2, G2.T @ G2, rtol=1e-12, atol=1e-12 * 500)
    # the eigen step over the accumulated K with the summed column count
    K = _gram_blocks(kin, G, splits)
    m_acc = kin.eig_select(P, 0.5)
    ev_acc = kin.eigvals(n)
    kin.close()
    whole = pb.Kinship(ctx, n, P)
    whole.append_columns(G)
    whole.gram()
    Kw = whole.partial_get()
    # one block is pg_kin_gram itself; accumulating onto a zero K gives the same bits
    assert np.array_equal(_gram_blocks(whole, G, [P]), Kw)
    whole.partial_set(np.zeros((n, n)))
    whole.gram(accumulate=True)
    assert np.array_equal(whole.partial_get(), Kw)
    m_one = whole.eig_select(P, 0.5)
    ev_one = whole.eigvals(n)
    whole.close()
    assert m_acc == m_one
    assert np.abs(ev_acc - ev_one).max() <= 1e-12 * ev_one[0]


# ---- file level ---------------------------------------------------------------------------------------------------
def _write_sync(path, counts, chroms, pos):
    from tests.test_text_gpu import _sync_text
    with open(path, "wb") as fh:
        fh.write(_sync_text(counts, chroms, pos))


def _run(src, ctx, method, fs, keep_p_minus_1, thr, out, block_bytes, device_bytes=None):
    """the file-level entry through the driver, with its phase record (device blocks used)"""
    tm = {}
    name = sync_io._iter_with_kinship(src, ctx, fs, keep_p_minus_1, thr, out, 2, block_bytes, method,
                                      device_bytes=device_bytes, timings=tm)
    return name, tm


def _one_text_block(ctx, n, k, block_bytes):
    """the smallest budget pass 1 accepts: the footprint of one text block's column bound"""
    return sync_io.kin_device_bytes(n, sync_io.text_block_columns(block_bytes, n), k, block_bytes, ctx.info()["sm_count"])


def _c1_file(tmp_path, L, chroms):
    c1 = H.load_c1()
    counts = c1["counts"][:L]
    pos = [int(p) for p in c1["pos"][:L]]
    fsync = str(tmp_path / "c.sync")
    _write_sync(fsync, counts, chroms, pos)
    from tests.test_sync_io import _write_c1_phen
    fphen = str(tmp_path / "c.csv")
    _write_c1_phen(fphen)
    phen = pb.FilePhen(fphen, ",", 0, 1, [2, 3]).lparse()
    fs = pb.FilterStats(pool_sizes=phen.pool_sizes, min_coverage_depth=5, min_allele_frequency=0.01)
    return c1, counts, pos, fsync, phen, fs


def _oracle_order(counts, codes, fs, keep_p_minus_1, chroms, pos):
    """the oracle's columns in the rows' order (loci sorted by chromosome and position) and their labels"""
    from oracle import pgo
    ocols, olabels = pgo.load_columns(counts.transpose(0, 2, 1).astype(np.uint64), codes, H.oracle_fs(fs), keep_p_minus_1)
    L = counts.shape[0]
    loci = sorted(range(L), key=lambda l: (chroms[l].encode(), pos[l]))
    by_locus = {}
    for c, (l, a) in enumerate(olabels):
        by_locus.setdefault(l, []).append((c, a))
    seq = [ca for l in loci for ca in by_locus.get(l, [])]
    labels = [("intercept", "0", "intercept")] + [(chroms[olabels[c][0]], str(pos[olabels[c][0]]), "ATCGND"[a]) for c, a in seq]
    return ocols[[c for c, _ in seq]], labels


def _rows(path):
    lines = open(path).read().split("\n")
    assert lines[0] == "#chr,pos,alleles,phenotype,statistic,pvalue" and lines[-1] == ""
    return [ln.split(",") for ln in lines[1:-1]]


def _check_ols_rows(rows, labels, ob, op, k, ov=None):
    """the assertions of tests/test_sync_io.py::test_ols_iter_with_kinship_file; with ov (PCs selected on the device),
    those of tests/test_kinship_gpu.py::test_c4_shape_gram_and_covariate_scan for the device's own PCs: beta to 1e-7 of
    max(|beta|, its standard error), p to 1e-6"""
    P = len(labels) - 1
    assert len(rows) == k * P
    for j in range(k):
        for i in range(P):
            r = rows[j * P + i]
            assert tuple(r[:3]) == labels[i] and r[3] == f"Pheno_{j}", (r, labels[i])
            got_b, got_p = float(r[4]), float(r[5])
            if ov is None:
                for got, exp, tol in ((got_b, ob[i, j], 1e-7), (got_p, op[i, j], 1e-6)):
                    assert (np.isnan(got) and np.isnan(exp)) or abs(got - exp) <= tol * max(abs(exp), 1e-3), (r, exp)
                continue
            if np.isnan(ob[i, j]):
                assert np.isnan(got_b), r
                continue
            assert abs(got_b - ob[i, j]) <= 1e-7 * max(abs(ob[i, j]), np.sqrt(ov[i, j])), (r, ob[i, j], ov[i, j])
            assert abs(got_p - op[i, j]) <= 1e-6 * op[i, j] + H.P_FLOOR, (r, op[i, j])


def _check_mle_rows(rows, labels, ob, ov, op, k):
    """the assertions of tests/test_sync_io.py::test_mle_iter_with_kinship_file"""
    P = len(labels) - 1
    assert len(rows) == k * P
    worst = 0.0
    for j in range(k):
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
@pytest.mark.parametrize("method", ["ols", "mle"])
def test_file_in_device_blocks_is_text_identical(ctx, tmp_path, method):
    """the C1-derived files of the file-level tests, forced into three or more device blocks: at the threshold of
    those tests (no PCs) the output equals the one-block run byte for byte, and the oracle's records"""
    from oracle import pgo
    L = 1200 if method == "ols" else 500
    chroms = [["chrB", "chrA"][(l // 250) % 2] for l in range(L)] if method == "ols" else ["chr1"] * L
    c1, counts, pos, fsync, phen, fs = _c1_file(tmp_path, L, chroms)
    src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, f"{method}_iter_with_kinship")
    bb = 3 << 10   # 14 to 32 text blocks, a few per device block
    one, tm1 = _run(src, ctx, method, fs, True, 0.75, str(tmp_path / "one.csv"), bb)
    many, tmb = _run(src, ctx, method, fs, True, 0.75, str(tmp_path / "many.csv"), bb, _one_text_block(ctx, 5, 2, bb))
    assert tm1["device_blocks"] == 1 and tmb["device_blocks"] >= 3, (tm1, tmb)
    assert open(many, "rb").read() == open(one, "rb").read()
    # the public entry takes the same budget
    entry = src.ols_iter_with_kinship if method == "ols" else src.mle_iter_with_kinship
    pub = entry(ctx, fs, True, 0.75, str(tmp_path / "pub.csv"), 2, block_bytes=bb, device_bytes=_one_text_block(ctx, 5, 2, bb))
    assert open(pub, "rb").read() == open(one, "rb").read()
    G, labels = _oracle_order(counts, c1["codes"], fs, True, chroms, pos)
    rows = _rows(many)
    if method == "ols":
        om, ob, ov, op = pgo.ols_with_covariate(G, phen.phen_matrix, 0.75)
        _check_ols_rows(rows, labels, ob, op, 2)
    else:
        om, ob, ov, op = pgo.mle_with_covariate(G, phen.phen_matrix, 0.75)
        assert om == 0 and len(labels) - 1 > 150
        _check_mle_rows(rows, labels, ob, ov, op, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("method,thr,m_expect", [("ols", 0.999, 55), ("mle", 0.9766, 4)])
def test_file_in_device_blocks_with_pcs(ctx, tmp_path, method, thr, m_expect):
    """a synthetic 60-pool file with principal components as covariates (m > 0; the simplex search converges within
    the reference's 1,000 iterations up to four covariates, tests/test_nm_gpu.py):
    the accumulated K differs from the one-block K in its last bits, so the records agree with the one-block run to the
    analysis' tolerance (OLS also with the oracle); the output names carry the same eigen count"""
    from oracle import pgo
    n, L, k = 60, 300, 2
    seed = 0x5EED0060
    counts = np.zeros((L, 6, n), dtype=np.uint32)
    counts[:, :4] = pb.synth_counts_host(seed, 0, L, n, 4)
    chroms = ["chr2" if l % 3 else "chr1" for l in range(L)]
    pos = [1000 + 7 * l for l in range(L)]
    phen = pb.synth_phen_host(seed, n, k)
    names = [f"p{i}" for i in range(n)]
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_coverage_depth=1, min_allele_frequency=0.01)
    bb = 32 << 10
    outs = {}
    for tag, budget in (("one", None), ("many", _one_text_block(ctx, n, k, bb))):
        d = tmp_path / tag
        d.mkdir()
        fsync = str(d / "s.sync")
        _write_sync(fsync, counts, chroms, pos)
        src = pb.FileSyncPhen(fsync, names, fs.pool_sizes, phen, f"{method}_iter_with_kinship")
        name, tm = _run(src, ctx, method, fs, True, thr, "", bb, budget)
        outs[tag] = (name, tm)
    (one, tm1), (many, tmb) = outs["one"], outs["many"]
    assert tm1["device_blocks"] == 1 and tmb["device_blocks"] >= 3, (tm1, tmb)
    strip = lambda p: os.path.basename(p).rsplit("-", 1)[0]   # <name>-<method>_iterative_xxt_<m + 1>_eigens
    assert strip(one) == strip(many) == f"s-{method}_iterative_xxt_{m_expect + 1}_eigens"
    r1, rb = _rows(one), _rows(many)
    assert [r[:4] for r in r1] == [r[:4] for r in rb]
    a1 = np.array([[float(x) for x in r[4:]] for r in r1])
    ab = np.array([[float(x) for x in r[4:]] for r in rb])
    assert (np.isnan(a1) == np.isnan(ab)).all()
    G, labels = _oracle_order(counts, np.arange(6, dtype=np.uint8), fs, True, chroms, pos)
    if method == "ols":
        ok = ~np.isnan(a1)
        err = np.abs(ab - a1)[ok] / np.maximum(np.abs(a1[ok]), 1e-3)
        assert err.max() <= 1e-9, err.max()
        om, ob, ov, op = pgo.ols_with_covariate(G, phen, thr)
        assert om == m_expect
        _check_ols_rows(rb, labels, ob, op, k, ov)
        return
    # the simplex search: errors relative to max(|beta|, its standard error) and to p, as tests/test_nm_gpu.py takes
    # them.  Where the reference's 1,000 iterations do not converge, where the search stops depends on the last bits
    # of the PCs (DESIGN.md section 11): such records are counted, not pinned (measured on a B200: 97 % of the 1,580
    # records within 1e-3, the rest within 4e-2 of the standard error)
    om, ob, ov, op = pgo.mle_with_covariate(G, phen, thr)
    assert om == m_expect
    se = np.sqrt(ov.T.reshape(-1))
    b1, bm, p1, pm = a1[:, 0], ab[:, 0], a1[:, 1], ab[:, 1]
    ok = ~np.isnan(b1) & ~np.isnan(se)
    eb = np.abs(bm - b1)[ok] / np.maximum(np.abs(b1[ok]), se[ok])
    ep = np.abs(pm - p1)[ok] / np.maximum(p1[ok], 1e-12)
    err = np.maximum(eb, ep)
    print(f"mle with {om} PCs, device blocks vs one block: median {np.median(err):.1e}, "
          f"{(err < 1e-3).mean():.4f} of {err.size} records within 1e-3, max {err.max():.1e}")
    assert np.median(err) < 5e-6 and (err < 1e-3).mean() >= 0.95 and err.max() < 0.2, (np.median(err), (err < 1e-3).mean())
    # no record-by-record oracle check here: the search is not invariant to the basis of the PCs, and the device's
    # eigenvectors are not numpy's; tests/test_nm_gpu.py holds pg_kin_mle_scan to the oracle with the same covariates
    # on both sides, and test_file_in_device_blocks_is_text_identical[mle] holds the file level to it at m = 0


@pytest.mark.gpu
def test_file_six_columns_per_locus(ctx, tmp_path):
    """--keep-ns, MAF 0, no --keep-p-minus-1: every locus emits six columns, more than a bound of five per line holds;
    the file-level entry runs and matches the oracle"""
    from oracle import pgo
    rng = np.random.default_rng(66)
    n, L, k = 7, 400, 2
    counts = rng.integers(1, 40, size=(L, 6, n)).astype(np.uint32)
    chroms = ["chr1"] * L
    pos = list(range(1, L + 1))
    fsync = str(tmp_path / "six.sync")
    _write_sync(fsync, counts, chroms, pos)
    phen = pb.synth_phen_host(0x51C, n, k)
    names = [f"p{i}" for i in range(n)]
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), remove_ns=False, min_allele_frequency=0.0)
    src = pb.FileSyncPhen(fsync, names, fs.pool_sizes, phen, "ols_iter_with_kinship")
    out = src.ols_iter_with_kinship(ctx, fs, False, 0.75, str(tmp_path / "six.csv"), 2)
    G, labels = _oracle_order(counts, np.arange(6, dtype=np.uint8), fs, False, chroms, pos)
    assert len(labels) - 1 > 5 * (L + 1)
    om, ob, ov, op = pgo.ols_with_covariate(G, phen, 0.75)
    _check_ols_rows(_rows(out), labels, ob, op, k)


@pytest.mark.gpu
def test_budget_below_one_text_block_is_refused(ctx, tmp_path):
    L = 300
    chroms = ["chr1"] * L
    c1, counts, pos, fsync, phen, fs = _c1_file(tmp_path, L, chroms)
    src = pb.FileSyncPhen(fsync, phen.pool_names, phen.pool_sizes, phen.phen_matrix, "ols_iter_with_kinship")
    bb = 12 << 10
    budget = _one_text_block(ctx, 5, 2, bb) - 1
    before = sorted(os.listdir(tmp_path))
    for entry in (src.ols_iter_with_kinship, src.mle_iter_with_kinship):
        for out in ("", str(tmp_path / "x.csv")):
            with pytest.raises(pb.PgError) as e:
                entry(ctx, fs, True, 0.75, out, 2, block_bytes=bb, device_bytes=budget)
            assert str(budget) in str(e.value) and str(bb) in str(e.value)
    assert sorted(os.listdir(tmp_path)) == before
    # one byte more is enough
    out = src.ols_iter_with_kinship(ctx, fs, True, 0.75, str(tmp_path / "y.csv"), 2, block_bytes=bb,
                                    device_bytes=budget + 1)
    assert os.path.exists(out)
