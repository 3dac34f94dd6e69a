"""GPU tests of the Nelder-Mead analyses (SURVEY.md 8f-3 / 8f-4): mle_iter (PG_KIND_MLE) and gwalpha
(PG_KIND_GWALPHA_LS / _ML) against the oracle's restatement of the reference (argmin's simplex search pinned by the
reference's own test_gwalpha lines, tests/test_oracle_golden.py).

Tolerance, declared up front: both sides run the same capped simplex search (1,000 iterations), whose path turns on
comparisons of nearly equal costs; the device evaluates the mle_iter cost as a quadratic form of centred moments
(O(p^2) per evaluation) where the reference walks the residuals (O(n p)), and its libm differs from the host's in the
last bit.  A path that splits ends at a different point of the flat valley around the optimum, so agreement is to the
solver's convergence: medians at 1e-6 or better, every value within 1e-3 (relative to the coefficient or its standard
error; measured maxima 4e-6) -- not the 1e-9 of the closed-form analyses.  The keep-mask, the allele order and the mean frequencies are bit-exact."""
import numpy as np
import pytest

import poolgen_b200 as pb
from oracle import pgo
from tests import helpers as H
from tests.test_nm_edges_gpu import check_mle_status

pytestmark = pytest.mark.gpu


def _gwalpha_fmt(n, rng):
    """a gwalpha_fmt matrix for n pools: bins sum to 1, increasing quantiles, sig / MIN / MAX in column 2"""
    bins = rng.dirichlet(np.full(n, 8.0))
    q = np.concatenate([[0.0], np.sort(rng.uniform(0.05, 0.95, size=n - 1))])
    rows = max(n, 3)
    fmt = np.full((rows, 3), -np.inf)
    fmt[:n, 0], fmt[:n, 1] = bins, q
    fmt[:3, 2] = (0.15, 0.0, 1.0)
    return fmt


def test_gwalpha_reference_example(ctx):
    """the reference's own known-answer test (src/gwas/gwalpha.rs:392-447) through the device path and the writer"""
    counts = np.array([5, 2, 6, 2, 2, 7, 3, 2, 5, 4, 3, 3, 5, 5, 0], dtype=np.uint32).reshape(5, 3)
    fmt = np.array([0.2, 0.2, 0.2, 0.2, 0.2, 0.0, 0.1, 0.4, 0.7, 0.9, 0.02, 0.0, 0.9, -np.inf, -np.inf]).reshape(3, 5).T.copy()
    fs = pb.FilterStats(pool_sizes=np.full(5, 20.0), min_allele_frequency=0.005)
    codes = np.array([0, 1, 5], dtype=np.uint8)
    dev_counts = np.ascontiguousarray(counts.T[None])           # [1, A, n]
    expect = {"LS": (5.816067, 9.176892), "ML": (-3.293261, -7.098985)}
    for method, kind in (("LS", pb.KIND_GWALPHA_LS), ("ML", pb.KIND_GWALPHA_ML)):
        rec = pb.gwalpha(ctx, dev_counts, fmt, fs, method, codes)
        assert rec.status[0] == pb.LOCUS_OK and rec.n_out[0] == 2 and list(rec.alleles[0][:2]) == [0, 1]
        alpha = rec.stats[0, :2, 0, 0]
        assert np.allclose(alpha, expect[method], rtol=0, atol=2e-5), (method, alpha)
        rows = pb.format_rows(kind, rec, [12345], chr_names=["Chromosome1"], chr_index=[0]).decode()
        lines = rows.strip().split("\n")
        assert len(lines) == 2 and lines[0].startswith("Chromosome1,12345,A,0.353287,Pheno_0,")
        assert lines[1].startswith("Chromosome1,12345,T,0.267133,Pheno_0,") and lines[1].endswith(",Unknown")
        got = [float(l.split(",")[5]) for l in lines]
        assert np.allclose(got, expect[method], atol=2e-5)


@pytest.mark.parametrize("n,A,L", [(5, 4, 300), (8, 6, 200), (12, 4, 150)])
@pytest.mark.parametrize("method", ["LS", "ML"])
def test_gwalpha_synthetic(ctx, method, n, A, L):
    rng = np.random.default_rng(100 * n + A)
    counts = pb.synth_counts_host(0x6A1 + n, 0, L, n, min(A, 4))
    full = np.zeros((L, A, n), dtype=np.uint32)
    full[:, :min(A, 4)] = counts
    fmt = _gwalpha_fmt(n, rng)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.01)
    codes = np.arange(A, dtype=np.uint8)
    dev = pb.gwalpha(ctx, full, fmt, fs, method, codes)
    okind = pgo.SCAN_GWALPHA_LS if method == "LS" else pgo.SCAN_GWALPHA_ML
    orc = pgo.scan_batch(okind, full, codes, fmt, H.oracle_fs(fs), 8)
    assert ((orc.status == pgo.FILTERED) == (dev.status == pb.LOCUS_FILTERED)).all()
    ok = orc.status == pgo.OK
    assert (dev.status[ok] == pb.LOCUS_OK).all() and ok.sum() > 0.5 * L
    assert (orc.n_out[ok] == dev.n_out[ok]).all() and (orc.allele[ok] == dev.alleles[ok]).all()
    S = dev.stats.shape[1]
    slot = np.arange(S)[None, :] < orc.n_out[ok][:, None]
    fm_o, fm_d = orc.freq_mean[ok][:, :S][slot], dev.freq_mean[ok][slot]
    assert np.allclose(fm_d, fm_o, rtol=1e-12, atol=0)
    a_o, a_d = orc.stat[ok][:, :S, 0][slot], dev.stats[ok][:, :, 0, 0][slot]
    err = np.abs(a_d - a_o) / np.maximum(np.abs(a_o), 1.0)
    print(f"gwalpha {method} n={n}: {slot.sum()} alphas, median err {np.median(err):.2e}, 99% {np.quantile(err, 0.99):.2e}, max {err.max():.2e}")
    # measured on B200 (profiles/README.md): medians 1e-8, maxima 2e-7
    assert np.median(err) < 1e-6 and err.max() < 1e-4


@pytest.mark.parametrize("n,A,k,L", [(30, 4, 2, 400), (100, 4, 1, 300), (6, 6, 3, 400), (1000, 4, 3, 60)])
def test_mle_iter_synthetic(ctx, n, A, k, L):
    counts = pb.synth_counts_host(0x31E + n, 0, L, n, min(A, 4))
    full = np.zeros((L, A, n), dtype=np.uint32)
    full[:, :min(A, 4)] = counts
    phen = pb.synth_phen_host(0x31E + n, n, k)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    codes = np.arange(A, dtype=np.uint8)
    dev = pb.mle_iterate(ctx, full, phen, fs, codes)
    orc = pgo.scan_batch(pgo.SCAN_MLE, full, codes, phen, H.oracle_fs(fs), 8)
    assert ((orc.status == pgo.FILTERED) == (dev.status == pb.LOCUS_FILTERED)).all()
    # statuses: UNSUPPORTED exactly where the reference's design has fewer pools than columns, OK against FAILED only
    # at a numerically singular X'X (cond > 1e12), nothing else
    both, why = check_mle_status(full, codes, fs, dev, orc, f"mle_iter n={n} k={k}")
    assert both.sum() > 0.5 * L, why
    assert (orc.n_out[both] == dev.n_out[both]).all() and (orc.allele[both] == dev.alleles[both]).all()
    S = dev.stats.shape[1]
    slot = np.broadcast_to((np.arange(S)[None, :] < orc.n_out[both][:, None])[:, :, None], (both.sum(), S, k))
    b_o, b_d = orc.stat[both][:, :S][slot], dev.stats[both][..., 0][slot]
    v_o, v_d = orc.var[both][:, :S][slot], dev.stats[both][..., 1][slot]
    p_o, p_d = orc.pval[both][:, :S][slot], dev.stats[both][..., 3][slot]
    # the OLS standard error of the coefficient is the natural scale: v_b = s2 diag, s2 = 2 RSS / n
    se = np.sqrt(np.abs(v_o) * n / (2.0 * np.maximum(n - (orc.n_out[both].astype(float)[:, None, None] + 1.0), 1.0) * np.ones((1, S, k)))[slot])
    eb = np.abs(b_d - b_o) / np.maximum(np.abs(b_o), se)
    ev = np.abs(v_d - v_o) / np.abs(v_o)
    ep = np.abs(p_d - p_o) / np.maximum(p_o, 1e-12)
    print(f"mle_iter n={n} k={k}: {slot.sum()} coefficients, beta err median {np.median(eb):.2e} max {eb.max():.2e}; "
          f"v_b err median {np.median(ev):.2e} max {ev.max():.2e}; p err median {np.median(ep):.2e} max {ep.max():.2e}")
    # measured on B200 (profiles/README.md): beta medians 1e-8 .. 3e-7, maxima 4e-6; p maxima 2.4e-6
    assert np.median(eb) < 5e-6 and eb.max() < 1e-3
    assert np.median(ev) < 1e-6 and ev.max() < 1e-3
    assert np.median(ep) < 5e-6 and ep.max() < 1e-3
    # rows text: beta rounded to 6 digits, p printed in full
    rows = pb.format_rows(pb.KIND_MLE, dev, np.arange(1, L + 1), chr_names=["chr1"], chr_index=np.zeros(L, np.uint32)).decode()
    first = rows.split("\n")[0].split(",")
    assert len(first) == 7 and first[4] == "Pheno_0"


def test_file_level_mle_iter_and_gwalpha(ctx, tmp_path):
    """`poolgen mle_iter` / `poolgen gwalpha` from a sync file (src/main.rs:299-358): FileSyncPhen::read_analyse_write with
    the new callbacks over the reference's tests/test.sync (5 pools), rows in file order"""
    from tests.test_text_gpu import _sync_text
    c1 = H.load_c1()
    L = 600
    counts = c1["counts"][:L]
    names = [str(s) for s in c1["chrom_names"]]
    chroms = [names[i] for i in c1["chrom_idx"][:L]]
    pos = [int(p) for p in c1["pos"][:L]]
    fsync = tmp_path / "t.sync"
    fsync.write_bytes(_sync_text(counts, chroms, pos))
    fs = pb.FilterStats(pool_sizes=c1["pool_sizes"], min_coverage_depth=10, min_allele_frequency=0.01)
    src = pb.FileSyncPhen(str(fsync), [f"p{i}" for i in range(5)], c1["pool_sizes"], c1["phen"], "mle_iter")
    out = src.read_analyse_write(ctx, fs, str(tmp_path / "mle.csv"), 2, pb.mle_iterate, block_bytes=16 << 10)
    lines = open(out).read().strip().split("\n")
    assert lines[0] == "#chr,pos,alleles,freq,phenotype,statistic,pvalue" and len(lines) > 100
    dev = pb.mle_iterate(ctx, counts, c1["phen"], fs, c1["codes"])
    expect = pb.format_rows(pb.KIND_MLE, dev, pos, chr_names=names, chr_index=c1["chrom_idx"][:L], exact_p_pools=5).decode()
    assert "\n".join(lines[1:]) + "\n" == expect
    rng = np.random.default_rng(5)
    fmt = _gwalpha_fmt(5, rng)
    srcg = pb.FileSyncPhen(str(fsync), [f"p{i}" for i in range(5)], c1["pool_sizes"], fmt, "gwalpha")
    outg = srcg.read_analyse_write(ctx, fs, str(tmp_path / "gw.csv"), 2, pb.gwalpha_ml, block_bytes=16 << 10)
    gl = open(outg).read().strip().split("\n")
    assert len(gl) > 100 and all(l.endswith(",Unknown") for l in gl[1:])
    devg = pb.gwalpha(ctx, counts, fmt, fs, "ML", c1["codes"])
    assert "\n".join(gl[1:]) + "\n" == pb.format_rows(pb.KIND_GWALPHA_ML, devg, pos, chr_names=names, chr_index=c1["chrom_idx"][:L]).decode()


@pytest.mark.parametrize("n,P,m,k", [(40, 300, 0, 2), (25, 200, 1, 1), (60, 150, 3, 2), (300, 70, 2, 1), (2000, 40, 0, 1)])
def test_mle_with_covariate(ctx, n, P, m, k):
    """mle_iter_with_kinship's scan (pg_kin_mle_scan vs the oracle's mle_with_covariate, gwas/mle.rs:307-463): per
    (column, phenotype) the last coefficient of the maximum-likelihood fit of y on [1 | covariates | g].  Both sides get
    the SAME covariate columns -- unlike the OLS scan the simplex search depends on the basis, not only on the span.
    Up to four covariates the reference's 1,000 iterations converge and the declared tolerance of this file applies;
    beyond that its own result is the end of a capped, unconverged path (test_mle_with_covariate_capped_path)."""
    rng = np.random.default_rng(n * 7 + m)
    G = np.clip(0.45 + 0.2 * rng.standard_normal((P, n)), 0.0, 1.0)
    G[3] = 0.25                                             # a constant column: X'X has no inverse -> NaN
    cov = rng.standard_normal((n, m)) / np.sqrt(n)          # the scale of unit eigenvectors
    phen = rng.standard_normal((n, k)) + 3.0 * G[5][:, None]
    kin = pb.Kinship(ctx, n, P)
    kin.append_columns(G)
    kin.set_covariates(cov)
    b_d, v_d, p_d = kin.mle_scan(phen)
    kin.close()
    _, b_o, v_o, p_o = pgo.mle_with_covariate(G, phen, 0.5, covariates=cov)
    b_o, v_o, p_o = b_o.T, v_o.T, p_o.T
    assert np.isnan(b_d[:, 3]).all() and np.isnan(b_o[:, 3]).all() and np.isnan(p_d[:, 3]).all()
    ok = ~np.isnan(b_o)
    assert (ok == ~np.isnan(b_d)).all() and ok.sum() == k * (P - 1)
    # v_b = sigma2 [(X'X)^-1]_gg is the squared standard error up to (n - p) / n
    eb = np.abs(b_d[ok] - b_o[ok]) / np.maximum(np.abs(b_o[ok]), np.sqrt(v_o[ok]))
    ev = np.abs(v_d[ok] - v_o[ok]) / v_o[ok]
    ep = np.abs(p_d[ok] - p_o[ok]) / np.maximum(p_o[ok], 1e-12)
    print(f"mle_with_covariate n={n} m={m} k={k}: beta err median {np.median(eb):.2e} max {eb.max():.2e}; "
          f"v_b median {np.median(ev):.2e} max {ev.max():.2e}; p median {np.median(ep):.2e} max {ep.max():.2e}")
    assert np.median(eb) < 5e-6 and eb.max() < 1e-3
    assert np.median(ev) < 1e-6 and ev.max() < 1e-3
    assert np.median(ep) < 5e-6 and ep.max() < 1e-3


def test_mle_with_covariate_capped_path(ctx):
    """Six covariates = nine parameters: the reference's 1,000 simplex iterations end far from the optimum (the oracle's
    coefficients are tens of standard errors from the least-squares ones), so the records are whatever the capped path
    reaches -- parity unpinned.  What holds on both sides: the search runs, every record is finite, and v_b follows
    sigma2 [(X'X)^-1]_gg with the sigma2 the path ended at.  More than 13 covariates are refused."""
    n, P, m = 50, 64, 6
    rng = np.random.default_rng(11)
    G = np.clip(0.45 + 0.2 * rng.standard_normal((P, n)), 0.0, 1.0)
    cov = rng.standard_normal((n, m)) / np.sqrt(n)
    phen = rng.standard_normal((n, 1))
    kin = pb.Kinship(ctx, n, P)
    kin.append_columns(G)
    kin.set_covariates(cov)
    b_d, v_d, p_d = kin.mle_scan(phen)
    assert np.isfinite(b_d).all() and (v_d > 0).all() and ((p_d >= 0) & (p_d <= 1)).all()
    _, b_o, v_o, p_o = pgo.mle_with_covariate(G, phen, 0.5, covariates=cov, columns=range(8))
    assert np.isfinite(b_o[:8]).all() and (v_o[:8] > 0).all()
    kin.set_covariates(rng.standard_normal((n, 14)))
    with pytest.raises(pb.PgError):
        kin.mle_scan(phen)
    kin.close()
