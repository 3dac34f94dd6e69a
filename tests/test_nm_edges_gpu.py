"""GPU tests of the Nelder-Mead kernels (pg_nm.cu) at the shapes test_nm_gpu.py does not reach: more phenotypes than one
pass of mle_kernel holds, batches past the first sweep of each grid-stride loop, the size limits (2 .. 64 gwalpha
pools, 13 covariates and 16 phenotypes of mle_iter_with_kinship, fewer pools than coefficients) and mle_iter designs
built count by count (collinear minor alleles, a minor allele whose frequency is the same in every pool).

Two references:
  * the device against itself, bit for bit, where a record must not depend on where it was computed: every locus and
    every (column, phenotype) is computed on its own (moments by warp_sum_fixed, each search in one lane), so the
    records of a phenotype, a locus or a column do not depend on the other phenotypes, on the lane or on the sweep;
  * the oracle at the declared tolerance of test_nm_gpu.py (medians 5e-6, every value within 1e-3; gwalpha 1e-6 /
    1e-4), and for well-conditioned loci the 50-digit closed form of the optimum, which does not depend on the simplex
    path: beta is the least-squares solution and sigma2 = 2 RSS / n (the reference's cost has no 1/2 on RSS / sigma2).
"""
import numpy as np
import pytest

import poolgen_b200 as pb
from oracle import pgo
from tests import helpers as H

pytestmark = pytest.mark.gpu

COND_FAILED = 1e12          # helpers.compare_regression: past this f64 solves legitimately disagree on invertibility
KEPS = 2.220446049250313e-16


def _fs(n):
    return pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))


def _same_records(a, b, label):
    """bit-identical records (NaN == NaN)"""
    for f in ("status", "n_out", "alleles", "freq_mean", "stats"):
        x, y = getattr(a, f), getattr(b, f)
        eq = np.array_equal(x, y, equal_nan=True) if x.dtype.kind == "f" else np.array_equal(x, y)
        if not eq:
            bad = np.nonzero(~((x == y) | (np.isnan(x) & np.isnan(y))).reshape(x.shape[0], -1).all(axis=1))[0] \
                if x.dtype.kind == "f" else np.nonzero((x != y).reshape(x.shape[0], -1).any(axis=1))[0]
            raise AssertionError(f"{label}: {f} differs at {bad.size} loci, first {bad[:8]}")


def _window(rec, lo, hi):
    return pb.ScanResults(rec.status[lo:hi], rec.n_out[lo:hi], rec.alleles[lo:hi], rec.freq_mean[lo:hi], rec.stats[lo:hi])


def _counts6(rng, L, n, depth=(40, 200)):
    """[L, 6, n] counts over A T C G N D with five alleles in play (odd loci: four, without T): per locus a Dirichlet
    allele spectrum, per pool a Dirichlet draw around it, multinomial counts; N (column 4) stays rare so the filter
    keeps most loci"""
    out = np.zeros((L, 6, n), dtype=np.uint32)
    for l in range(L):
        p = rng.dirichlet([3.0, 2.0, 1.5, 1.0, 0.05, 0.8])
        for i in range(n):
            q = rng.dirichlet(40.0 * p + 1e-3)
            if l % 2:
                q[1] = 0.0          # odd loci without T: four kept alleles, three allele columns
                q /= q.sum()
            out[l, :, i] = rng.multinomial(int(rng.integers(*depth)), q)
    return out


def _gwalpha_fmt(n, rng):
    """a gwalpha_fmt matrix for n pools: bins sum to 1, increasing quantiles, sig / MIN / MAX in column 2"""
    bins = rng.dirichlet(np.full(n, 8.0))
    q = np.concatenate([[0.0], np.sort(rng.uniform(0.05, 0.95, size=n - 1))])
    fmt = np.full((max(n, 3), 3), -np.inf)
    fmt[:n, 0], fmt[:n, 1] = bins, q
    fmt[:3, 2] = (0.15, 0.0, 1.0)
    return fmt


def _oracle_design(counts_locus, codes, ofs):
    """the X of mle_iterate after remove_collinearities_in_x (mle.rs:56-83), statement for statement with the oracle's
    own Pearson r; None where the reference's `i -= 1` would underflow"""
    X = H._design(counts_locus, codes, ofs)
    cols = list(range(X.shape[1]))
    if len(cols) == 2:
        return X
    i = 1
    while i < len(cols):
        j = i + 1
        while j < len(cols):
            if i < 0:
                return None
            r, _ = pgo.pearsons_correlation(X[:, cols[i]], X[:, cols[j]])
            if abs(r) >= 0.99:
                del cols[j]
                i -= 1
                j -= 1
            j += 1
        i += 1
    return X[:, cols]


def _cond(X):
    with np.errstate(all="ignore"):
        return float(np.linalg.cond(X.T @ X))


def check_mle_status(counts, codes, fs, dev, orc, label):
    """the statuses of mle_iter against the oracle: the keep-mask exactly; LOCUS_UNSUPPORTED exactly where the
    oracle's design after collinearity removal has fewer pools than columns (the X X' form the device does not
    implement); OK against FAILED only where X'X is numerically singular (cond > 1e12); nothing else.
    Returns (both OK mask, {reason: count})"""
    ofs = H.oracle_fs(fs)
    n = counts.shape[2]
    assert ((orc.status == pgo.FILTERED) == (dev.status == pb.LOCUS_FILTERED)).all(), f"{label}: keep-mask differs"
    assert not (orc.status == pgo.PANIC).any() and not (dev.status == pb.LOCUS_PANIC).any(), f"{label}: panic"
    why = {"unsupported": 0, "singular": 0}
    for l in np.nonzero(orc.status != pgo.FILTERED)[0]:
        o, d = int(orc.status[l]), int(dev.status[l])
        if o == pgo.OK and d == pb.LOCUS_OK and n > 6:
            continue            # X has at most 6 columns: nothing to classify
        X = _oracle_design(counts[l], codes, ofs)
        assert X is not None, f"{label}: locus {l}: the reference would panic"
        pw = X.shape[1]
        assert (d == pb.LOCUS_UNSUPPORTED) == (n < pw), f"{label}: locus {l}: device status {d} with {n} pools, {pw} columns"
        if d == pb.LOCUS_UNSUPPORTED:
            why["unsupported"] += 1
        elif (o == pgo.OK) != (d == pb.LOCUS_OK):
            c = _cond(X)
            assert o == pgo.FAILED or d == pb.LOCUS_FAILED, (label, l, o, d)
            assert c > COND_FAILED, f"{label}: locus {l}: oracle {o} device {d} at cond(X'X) {c:.3g}"
            why["singular"] += 1
        else:
            assert o == pgo.OK or d == pb.LOCUS_FAILED, (label, l, o, d)
    return (orc.status == pgo.OK) & (dev.status == pb.LOCUS_OK), why


def zero_rows(stat, var, t, p):
    """the rows the reference leaves at Array2::zeros (removed collinear columns): beta 0, v_b 0, t NaN, p 0"""
    return (stat == 0.0) & (var == 0.0) & np.isnan(t) & (p == 0.0)


def compare_mle(dev, orc, both, n, label, median_tol=5e-6, max_tol=1e-3):
    """mle_iter records against the oracle at loci both solved: allele order and the zero-row pattern exactly, the
    filled rows at the declared tolerance.  Returns the relative errors of beta, v_b and p."""
    k = dev.stats.shape[2]
    S = dev.stats.shape[1]
    assert (orc.n_out[both] == dev.n_out[both]).all() and (orc.allele[both] == dev.alleles[both]).all(), f"{label}: alleles"
    slot = np.broadcast_to((np.arange(S)[None, :] < orc.n_out[both][:, None])[:, :, None], (both.sum(), S, k))
    o = [a[both][:, :S] for a in (orc.stat, orc.var, orc.t, orc.pval)]
    d = [dev.stats[both][..., e] for e in range(4)]
    zo, zd = zero_rows(*o), zero_rows(*d)
    assert np.array_equal(zo & slot, zd & slot), f"{label}: rows of removed columns differ at {np.nonzero((zo != zd) & slot)[0][:8]}"
    fill = slot & ~zo
    b_o, b_d, v_o, v_d, p_o, p_d = o[0][fill], d[0][fill], o[1][fill], d[1][fill], o[3][fill], d[3][fill]
    pw = np.broadcast_to(orc.n_out[both][:, None, None] + 1.0 - (zo & slot).sum(axis=1, keepdims=True), zo.shape)[fill]
    se = np.sqrt(np.abs(v_o) * n / (2.0 * np.maximum(n - pw, 1.0)))
    eb = np.abs(b_d - b_o) / np.maximum(np.abs(b_o), se)
    ev = np.abs(v_d - v_o) / np.abs(v_o)
    ep = np.abs(p_d - p_o) / np.maximum(p_o, 1e-12)
    if fill.sum():
        print(f"{label}: {fill.sum()} coefficients vs oracle: beta err median {np.median(eb):.2e} max {eb.max():.2e}; "
              f"v_b median {np.median(ev):.2e} max {ev.max():.2e}; p median {np.median(ep):.2e} max {ep.max():.2e}")
        for name, e in (("beta", eb), ("v_b", ev), ("p", ep)):
            assert np.median(e) < median_tol and e.max() < max_tol, (label, name, np.median(e), e.max())
    return eb, ev, ep


def _hp_closed_form(X, y):
    """the optimum of the reference's cost at 50 digits: beta = (X'X)^-1 X'y, sigma2 = 2 RSS / n, v_b = sigma2 diag"""
    import mpmath as mp
    mp.mp.dps = 50
    n = X.shape[0]
    Xm, ym = mp.matrix(X.tolist()), mp.matrix([[v] for v in y.tolist()])
    inv = (Xm.T * Xm) ** -1
    b = inv * (Xm.T * ym)
    e = ym - Xm * b
    s2 = 2 * (e.T * e)[0] / n
    return [float(b[i]) for i in range(X.shape[1])], [float(s2 * inv[i, i]) for i in range(X.shape[1])]


def compare_closed_form(counts, codes, phen, fs, dev, both, label, n_loci=12, max_cond=1e6):
    """a sample of well-conditioned loci (cond(X'X) < 1e6, at least 3 residual degrees of freedom) that kept every
    column against the 50-digit optimum (median 5e-6, max 1e-3)"""
    ofs = H.oracle_fs(fs)
    n, k = counts.shape[2], phen.shape[1]
    eb, ev, used = [], [], 0
    for l in np.nonzero(both)[0]:
        if used == n_loci:
            break
        X = _oracle_design(counts[l], codes, ofs)
        if X.shape[1] != int(dev.n_out[l]) + 1 or n < X.shape[1] + 3 or _cond(X) > max_cond:
            continue
        used += 1
        for j in range(k):
            b, vb = _hp_closed_form(X, phen[:, j])
            for s in range(int(dev.n_out[l])):
                se = np.sqrt(vb[s + 1] * n / (2.0 * (n - X.shape[1])))
                eb.append(abs(dev.stats[l, s, j, 0] - b[s + 1]) / max(abs(b[s + 1]), se))
                ev.append(abs(dev.stats[l, s, j, 1] - vb[s + 1]) / vb[s + 1])
    assert used >= min(n_loci, 3), f"{label}: only {used} well-conditioned loci"
    eb, ev = np.array(eb), np.array(ev)
    print(f"{label}: {used} loci vs the 50-digit closed form: beta err median {np.median(eb):.2e} max {eb.max():.2e}; "
          f"v_b median {np.median(ev):.2e} max {ev.max():.2e}")
    assert np.median(eb) < 5e-6 and eb.max() < 1e-3
    assert np.median(ev) < 5e-6 and ev.max() < 1e-3


# ---- 1. phenotype passes ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,n,A", [(4, 30, 4), (5, 100, 6), (8, 30, 6), (9, 100, 4)])
def test_mle_iter_phenotype_passes(ctx, k, n, A):
    """mle_kernel takes the phenotypes four at a time (kMlePhen): k = 4 is one full pass, 5 a second pass of one
    phenotype, 8 two full passes, 9 a third pass.  Phenotype j must not depend on the others: its records are those of a
    one-phenotype scan of column j, bit for bit."""
    L = 160
    seed = 0xE0 + 16 * k + n
    counts = pb.synth_counts_host(seed, 0, L, n, 4) if A == 4 else _counts6(np.random.default_rng(seed), L, n)
    phen = pb.synth_phen_host(seed, n, k)
    fs, codes = _fs(n), np.arange(A, dtype=np.uint8)
    dev = pb.mle_iterate(ctx, counts, phen, fs, codes)
    assert dev.stats.shape[2] == k
    # loci without a solution carry NaN records for every phenotype, not only the first
    assert np.isnan(dev.stats[dev.status != pb.LOCUS_OK]).all()
    for j in range(k):
        one = pb.mle_iterate(ctx, counts, phen[:, j:j + 1].copy(), fs, codes)
        for f in ("status", "n_out", "alleles"):
            assert np.array_equal(getattr(one, f), getattr(dev, f)), (j, f)
        assert np.array_equal(one.freq_mean, dev.freq_mean, equal_nan=True), j
        assert np.array_equal(one.stats[:, :, 0], dev.stats[:, :, j], equal_nan=True), f"phenotype {j} of {k} differs from its own scan"
    orc = pgo.scan_batch(pgo.SCAN_MLE, counts, codes, phen, H.oracle_fs(fs), 8)
    both, why = check_mle_status(counts, codes, fs, dev, orc, f"k={k} n={n} A={A}")
    assert both.sum() > 0.8 * L and (dev.n_out[both] == A - 1 - (A == 6)).sum() > 0.3 * both.sum()
    # four allele columns (five coefficients and sigma2) are past what 1,000 iterations reach from the all-ones
    # simplex: both searches end short of the optimum, where the path turns on near ties and the device's and the
    # oracle's paths part (measured: beta up to 0.29 apart) -- those loci are held bit for bit above, not to the oracle
    held = both & (orc.n_out <= 3)
    assert held.sum() > 0.3 * L
    compare_mle(dev, orc, held, n, f"mle_iter k={k} n={n} A={A}")
    if A == 4:
        # five coefficients and sigma2 (A = 6) are past what 1,000 iterations reach from the all-ones simplex: the
        # oracle's own search ends up to 1e-2 from the optimum there, so the path-free anchor is checked at A = 4
        compare_closed_form(counts, codes, phen, fs, dev, both, f"mle_iter k={k} n={n} A={A}")


@pytest.mark.parametrize("k", [5, 16])
def test_kin_mle_scan_phenotypes(ctx, k):
    """pg_kin_mle_scan keeps a row of 2 + m + k moments per column: phenotype j of a k-phenotype call is the
    one-phenotype call of column j, bit for bit.  More than 16 phenotypes are refused."""
    n, P, m = 40, 100, 2
    rng = np.random.default_rng(50 + k)
    G = np.clip(0.45 + 0.2 * rng.standard_normal((P, n)), 0.0, 1.0)
    cov = rng.standard_normal((n, m)) / np.sqrt(n)
    phen = rng.standard_normal((n, k)) + 2.0 * G[3][:, None]
    kin = pb.Kinship(ctx, n, P)
    try:
        kin.append_columns(G)
        kin.set_covariates(cov)
        b, v, p = kin.mle_scan(phen)
        assert np.isfinite(b).all() and (v > 0).all()
        for j in range(k):
            bj, vj, pj = kin.mle_scan(phen[:, j:j + 1].copy())
            for x, y in ((b, bj), (v, vj), (p, pj)):
                assert np.array_equal(x[j], y[0], equal_nan=True), f"phenotype {j} of {k}"
        with pytest.raises(pb.PgError):
            kin.mle_scan(rng.standard_normal((n, 17)))
    finally:
        kin.close()


# ---- 2. grid sweeps and ragged tails ---------------------------------------------------------------------------------
def _windows(L, W):
    """(start, length) of the windows: the first loci, the middle of the batch (past the first sweep whatever the
    occupancy), the last loci; no start a multiple of 32, so every locus of a window sits on another lane than in the
    batch"""
    last = L - W - ((L - W) % 32 == 0)
    out = [(5, W), ((L // 2) // 32 * 32 + 19, W), (last, L - last)]
    assert all(s % 32 for s, _ in out), out
    return out


def test_mle_iter_grid_sweeps(ctx):
    """L past two full sweeps of mle_kernel's grid at the largest occupancy (16 CTAs of 4 warps per SM, 32 loci a
    warp), ending on a partial warp: windows of the batch re-run on their own are bit-identical, and match the oracle"""
    n, A, k = 30, 4, 1
    seed = 0x5EED0031
    sm = ctx.info()["sm_count"]
    sweep = sm * 16 * 4 * 32
    L = 2 * sweep + 13
    print(f"mle_iter grid: L = {L} loci, largest sweep = {sweep} loci ({sm} SMs x 16 CTAs x 128 loci)")
    phen = pb.synth_phen_host(seed, n, k)
    fs, codes = _fs(n), np.arange(A, dtype=np.uint8)
    scan = pb.Scan(ctx, pb.KIND_MLE, fs, n, codes, phen)
    try:
        b = scan.batch(L)
        b.synth(seed, 0, L)
        b.run()
        big = b.fetch()
        b.close()
        assert (big.status == pb.LOCUS_OK).mean() > 0.9
        for s, W in _windows(L, 300):
            c = pb.synth_counts_host(seed, s, W, n, A)
            w = scan.run_counts(c)
            _same_records(_window(big, s, s + W), w, f"mle_iter loci {s}..{s + W}")
            orc = pgo.scan_batch(pgo.SCAN_MLE, c, codes, phen, H.oracle_fs(fs), 8)
            both, _ = check_mle_status(c, codes, fs, w, orc, f"window {s}")
            compare_mle(w, orc, both, n, f"mle_iter window {s}")
    finally:
        scan.close()


@pytest.mark.parametrize("method", ["LS", "ML"])
def test_gwalpha_grid_sweeps(ctx, method):
    """gwalpha_kernel's grid is capped at sm_count x 8 CTAs x 128 (locus, allele) items: L (A - 1) past two such
    sweeps, windows re-run on their own bit-identical to the batch and within tolerance of the oracle"""
    n, A = 5, 4
    seed = 0x6A1 + (method == "ML")
    sm = ctx.info()["sm_count"]
    sweep = sm * 8 * 128
    L = (2 * sweep) // (A - 1) + 37
    print(f"gwalpha {method} grid: L = {L} loci = {L * (A - 1)} items, sweep = {sweep} items ({sm} SMs x 8 x 128)")
    fmt = _gwalpha_fmt(n, np.random.default_rng(seed))
    fs, codes = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.01), np.arange(A, dtype=np.uint8)
    kind = pb.KIND_GWALPHA_LS if method == "LS" else pb.KIND_GWALPHA_ML
    scan = pb.Scan(ctx, kind, fs, n, codes, fmt)
    try:
        b = scan.batch(L)
        b.synth(seed, 0, L)
        b.run()
        big = b.fetch()
        b.close()
        for s, W in _windows(L, 97):
            c = pb.synth_counts_host(seed, s, W, n, A)
            w = scan.run_counts(c)
            _same_records(_window(big, s, s + W), w, f"gwalpha {method} loci {s}..{s + W}")
            check_gwalpha(c, codes, fmt, fs, w, method, f"gwalpha {method} window {s}")
    finally:
        scan.close()


def test_kin_mle_grid_sweeps(ctx):
    """kin_mle_kernel's grid is capped at sm_count x 4 CTAs x 4 warps x 32 columns: P past two such sweeps, made of
    copies of a tile of distinct columns whose length is not a multiple of 32 (each copy starts on another lane) plus a
    partial copy; every copy is bit-identical to a handle holding only the tile, which matches the oracle"""
    n, m, T = 24, 2, 299
    sm = ctx.info()["sm_count"]
    sweep = sm * 4 * 4 * 32
    copies = (2 * sweep) // T + 1
    P = copies * T + 17
    print(f"kin_mle grid: P = {P} columns, sweep = {sweep} columns ({sm} SMs x 4 x 128)")
    rng = np.random.default_rng(24)
    tile = np.clip(0.45 + 0.2 * rng.standard_normal((T, n)), 0.0, 1.0)
    cov = rng.standard_normal((n, m)) / np.sqrt(n)
    phen = rng.standard_normal((n, 1)) + 2.0 * tile[4][:, None]
    G = np.concatenate([np.tile(tile, (copies, 1)), tile[:17]])
    kin = pb.Kinship(ctx, n, P)
    ref = pb.Kinship(ctx, n, T)
    try:
        kin.append_columns(G)
        kin.set_covariates(cov)
        big = kin.mle_scan(phen)
        ref.append_columns(tile)
        ref.set_covariates(cov)
        one = ref.mle_scan(phen)
    finally:
        kin.close()
        ref.close()
    for x, y, name in zip(big, one, ("beta", "v_b", "p")):
        assert x.shape == (1, P)
        for c in range(copies):
            assert np.array_equal(x[:, c * T:(c + 1) * T], y, equal_nan=True), f"{name}: copy {c} (columns {c * T}..)"
        assert np.array_equal(x[:, copies * T:], y[:, :17], equal_nan=True), f"{name}: the partial copy"
    _, b_o, v_o, p_o = pgo.mle_with_covariate(tile, phen, 0.5, covariates=cov)
    b_d, v_d, p_d = (a[0] for a in one)
    ok = ~np.isnan(b_o[:, 0])
    assert (ok == ~np.isnan(b_d)).all() and ok.sum() == T
    eb = np.abs(b_d - b_o[:, 0]) / np.maximum(np.abs(b_o[:, 0]), np.sqrt(v_o[:, 0]))
    ev = np.abs(v_d - v_o[:, 0]) / v_o[:, 0]
    ep = np.abs(p_d - p_o[:, 0]) / np.maximum(p_o[:, 0], 1e-12)
    print(f"kin_mle tile vs oracle: beta err median {np.median(eb):.2e} max {eb.max():.2e}; v_b median {np.median(ev):.2e} "
          f"max {ev.max():.2e}; p median {np.median(ep):.2e} max {ep.max():.2e}")
    assert np.median(eb) < 5e-6 and eb.max() < 1e-3
    assert np.median(ev) < 1e-6 and ev.max() < 1e-3
    assert np.median(ep) < 5e-6 and ep.max() < 1e-3


# ---- 3. limits -------------------------------------------------------------------------------------------------------
def check_gwalpha(counts, codes, fmt, fs, dev, method, label):
    okind = pgo.SCAN_GWALPHA_LS if method == "LS" else pgo.SCAN_GWALPHA_ML
    orc = pgo.scan_batch(okind, counts, codes, fmt, H.oracle_fs(fs), 8)
    assert ((orc.status == pgo.FILTERED) == (dev.status == pb.LOCUS_FILTERED)).all(), f"{label}: keep-mask"
    ok = orc.status == pgo.OK
    assert (dev.status[ok] == pb.LOCUS_OK).all() and ok.sum() > 0
    assert (orc.n_out[ok] == dev.n_out[ok]).all() and (orc.allele[ok] == dev.alleles[ok]).all(), f"{label}: alleles"
    S = dev.stats.shape[1]
    slot = np.arange(S)[None, :] < orc.n_out[ok][:, None]
    assert np.allclose(dev.freq_mean[ok][slot], orc.freq_mean[ok][:, :S][slot], rtol=1e-12, atol=0)
    a_o, a_d = orc.stat[ok][:, :S, 0][slot], dev.stats[ok][:, :, 0, 0][slot]
    err = np.abs(a_d - a_o) / np.maximum(np.abs(a_o), 1.0)
    print(f"{label}: {slot.sum()} alphas vs oracle, median err {np.median(err):.2e}, max {err.max():.2e}")
    assert np.median(err) < 1e-6
    far = np.nonzero(err >= 1e-4)[0]
    if far.size:
        # a path split: the ML cost floors every cdf difference below epsilon, and with tens of bins the search meets
        # exact ties that a last-bit difference of a Beta cdf decides.  Such an alpha is not pinned to better than the
        # oracle's own answer under a one-ulp change of the bins, so the device may differ there, by no more than the
        # oracle moves itself, and at a few alphas only
        moved = np.zeros_like(err)
        for seed in range(4):
            fm = fmt.copy()
            n = counts.shape[2]
            fm[:n, 0] = fmt[:n, 0] * (1.0 + np.random.default_rng(seed).choice([-1.0, 1.0], n) * 2.0 ** -52)
            o2 = pgo.scan_batch(okind, counts, codes, fm, H.oracle_fs(fs), 8)
            a2 = o2.stat[ok][:, :S, 0][slot]
            moved = np.maximum(moved, np.abs(a2 - a_o) / np.maximum(np.abs(a_o), 1.0))
        print(f"{label}: {far.size} alphas at a path split: device err {err[far]}, oracle's own one-ulp spread {moved[far]}")
        assert far.size <= max(2, 0.05 * err.size) and (err[far] <= 4.0 * moved[far]).all()
    return orc


@pytest.mark.parametrize("n", [2, 3, 63, 64])
@pytest.mark.parametrize("method", ["LS", "ML"])
def test_gwalpha_pool_limits(ctx, method, n):
    """gwalpha keeps per-thread arrays of kGwMaxPools = 64 pools.  At 63 pools the biallelic loci take the m == 1
    unrolled dot of ndarray (7 blocks of 8 and a remainder of 7); 65 pools are refused."""
    A = 4
    L = 24 if n > 8 else 120
    seed = 0x6A2 + n
    rng = np.random.default_rng(seed)
    counts = pb.synth_counts_host(seed, 0, L, n, A)
    if n == 63:
        counts[: L // 2, 2:] = 0                       # biallelic: one minor allele kept
    fmt = _gwalpha_fmt(n, rng)
    fs, codes = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.01), np.arange(A, dtype=np.uint8)
    dev = pb.gwalpha(ctx, counts, fmt, fs, method, codes)
    orc = check_gwalpha(counts, codes, fmt, fs, dev, method, f"gwalpha {method} n={n}")
    if n == 63:
        assert ((orc.status == pgo.OK) & (orc.n_out == 1)).sum() >= L // 4
    if n == 64:
        c65 = pb.synth_counts_host(seed, 0, 4, 65, A)
        with pytest.raises(pb.PgError):
            pb.gwalpha(ctx, c65, _gwalpha_fmt(65, rng), pb.FilterStats(pool_sizes=np.full(65, 1.0 / 65)), method, codes)


def _mle_cost_np(par, X, y):
    s2 = KEPS + (1e9 - KEPS) / (1.0 + np.exp(-par[0]))
    r = y - X @ par[1:]
    return (len(y) / 2.0) * np.log(2.0 * np.pi * s2) + (r @ r) / s2


@pytest.mark.parametrize("m,k", [(7, 2), (10, 3), (13, 16)])
def test_kin_mle_many_covariates(ctx, m, k):
    """Up to 13 covariates (a simplex of 16 parameters) and, at 13, 16 phenotypes: the largest row of shared memory,
    2 + m + k doubles a column.  Past about five covariates the capped search ends anywhere (the oracle's path too,
    test_mle_with_covariate_capped_path), so what is asserted is what holds for any end point: finite records, v_b > 0,
    p in [0, 1], v_b = sigma2 [(X'X)^-1]_gg with a sigma2 whose cost is no worse than the best initial vertex (a
    Nelder-Mead search never loses its best cost), and the phenotype split of test_kin_mle_scan_phenotypes.  n = m + 2
    pools are accepted, m + 1 refused."""
    n, P = 48, 40
    rng = np.random.default_rng(100 + m)
    G = np.clip(0.45 + 0.2 * rng.standard_normal((P, n)), 0.0, 1.0)
    cov = rng.standard_normal((n, m)) / np.sqrt(n)
    phen = rng.standard_normal((n, k)) + 2.0 * G[2][:, None]
    kin = pb.Kinship(ctx, n, P)
    try:
        kin.append_columns(G)
        kin.set_covariates(cov)
        b, v, p = kin.mle_scan(phen)
        assert np.isfinite(b).all() and np.isfinite(v).all() and (v > 0).all() and ((p >= 0) & (p <= 1)).all()
        for j in sorted({0, k - 1}):
            one = kin.mle_scan(phen[:, j:j + 1].copy())
            for x, y in zip((b, v, p), one):
                assert np.array_equal(x[j], y[0], equal_nan=True), f"phenotype {j} of {k}"
    finally:
        kin.close()
    d = 3 + m
    for c in range(P):
        X = np.hstack([np.ones((n, 1)), cov, G[c][:, None]])
        inv_gg = np.linalg.inv(X.T @ X)[-1, -1]
        for j in range(k):
            s2 = v[j, c] / inv_gg
            assert KEPS <= s2 <= 1e9, (c, j, s2)
            y = phen[:, j]
            f0 = min(_mle_cost_np(np.where(np.arange(d) == i, 1.5, 1.0), X, y) for i in range(d + 1))
            rss = y @ y - y @ X @ np.linalg.lstsq(X, y, rcond=None)[0]
            lower = (n / 2.0) * np.log(2.0 * np.pi * s2) + max(rss, 0.0) / s2
            assert lower <= f0 * (1 + 1e-9) + 1e-9, f"column {c} phenotype {j}: sigma2 {s2:.6g} costs at least {lower:.6g} > start {f0:.6g}"
    for nn, ok in ((m + 2, True), (m + 1, False)):
        kin = pb.Kinship(ctx, nn, 8)
        try:
            kin.append_columns(np.clip(0.45 + 0.2 * rng.standard_normal((8, nn)), 0.0, 1.0))
            if ok:
                kin.set_covariates(rng.standard_normal((nn, m)) / np.sqrt(nn))
                _, _, pp = kin.mle_scan(rng.standard_normal((nn, 1)))
                assert pp.shape == (1, 8) and (np.isnan(pp) | ((pp >= 0) & (pp <= 1))).all()
            else:
                with pytest.raises(pb.PgError):
                    kin.set_covariates(rng.standard_normal((nn, m)) / np.sqrt(nn))
                    kin.mle_scan(rng.standard_normal((nn, 1)))
        finally:
            kin.close()


def _counts_all_alleles(rng, L, n, A):
    """[L, A, n] counts where every allele (N excepted) is common in every pool: nothing is filtered away"""
    out = np.zeros((L, A, n), dtype=np.uint32)
    live = [a for a in range(A) if not (A == 6 and a == 4)]
    for l in range(L):
        p = rng.dirichlet(np.full(len(live), 6.0))
        for i in range(n):
            out[l, live, i] = rng.multinomial(int(rng.integers(60, 200)), rng.dirichlet(30.0 * p))
    return out


@pytest.mark.parametrize("n", [2, 3, 4])
@pytest.mark.parametrize("A", [4, 5, 6])
def test_mle_iter_fewer_pools_than_coefficients(ctx, n, A):
    """mle_iter with as many or fewer pools than coefficients: LOCUS_UNSUPPORTED exactly where the oracle's design after
    collinearity removal has more columns than pools (the X X' form of mle.rs:130-140, not built on the device), OK
    where it has as many"""
    L = 80
    rng = np.random.default_rng(40 * n + A)
    counts = _counts_all_alleles(rng, L, n, A)
    phen = rng.standard_normal((n, 1))
    fs, codes = _fs(n), np.arange(A, dtype=np.uint8)
    dev = pb.mle_iterate(ctx, counts, phen, fs, codes)
    orc = pgo.scan_batch(pgo.SCAN_MLE, counts, codes, phen, H.oracle_fs(fs), 8)
    both, why = check_mle_status(counts, codes, fs, dev, orc, f"n={n} A={A}")
    ofs = H.oracle_fs(fs)
    assert (orc.status != pgo.FILTERED).all()
    pw = np.array([_oracle_design(counts[l], codes, ofs).shape[1] for l in range(L)])
    assert (dev.status[pw <= n] == pb.LOCUS_OK).all() and (pw == n).any()
    assert (orc.n_out[both] == dev.n_out[both]).all() and (orc.allele[both] == dev.alleles[both]).all()
    print(f"mle_iter n={n} A={A}: pw {np.bincount(pw).tolist()}, unsupported {why['unsupported']}, ok {both.sum()}")


# ---- 4. degenerate mle_iter designs, built count by count ------------------------------------------------------------
DEPTH = 1000


def _locus(minor_counts, depth=DEPTH):
    """one locus over A T C G N D (6 columns, N empty): the major allele first (its frequency is the largest on
    average), then the minor alleles in the order given; every pool has the same depth"""
    mc = np.asarray(minor_counts)
    n = mc.shape[1]
    out = np.zeros((6, n), dtype=np.uint32)
    live = [1, 2, 3, 5][: mc.shape[0]]
    out[live] = mc
    out[0] = depth - mc.sum(axis=0)
    assert (out[0] > 0).all() and out[0].mean() > 0.4 * depth
    return out


def _collinear_locus(rng, n, m, groups):
    """m minor alleles with well separated mean frequencies; the columns of each group in `groups` track the first of
    the group (|r| >= 0.995); every other pair |r| <= 0.985 -- both at least 0.005 from the 0.99 threshold"""
    means = [0.16, 0.10, 0.06, 0.035][:m]
    while True:
        mc = np.zeros((m, n))
        for a in range(m):
            mc[a] = np.round(DEPTH * means[a] * rng.uniform(0.4, 1.6, n))
        for g in groups:
            for a in g[1:]:
                mc[a] = np.round(mc[g[0]] * means[a] / means[g[0]] + rng.integers(-1, 2, n))
        loc = _locus(mc.astype(np.uint32))
        f = loc[[1, 2, 3, 5][:m]] / DEPTH
        same = {frozenset((a, b)) for g in groups for a in g for b in g if a != b}
        r = {(a, b): abs(pgo.pearsons_correlation(f[a], f[b])[0]) for a in range(m) for b in range(a + 1, m)}
        if all((v >= 0.995) if frozenset(ab) in same else (v <= 0.985) for ab, v in r.items()):
            return loc


@pytest.mark.parametrize("m,groups", [(2, [(0, 1)]), (3, [(0, 1)]), (3, [(0, 2)]), (3, [(1, 2)]), (4, [(0, 1)]),
                                      (4, [(1, 2)]), (4, [(2, 3)]), (4, [(0, 3)]), (3, [(0, 1, 2)]), (4, [(1, 2, 3)])],
                         ids=lambda x: str(x).replace(" ", ""))
def test_mle_iter_collinear_alleles(ctx, m, groups):
    """remove_collinearities_in_x (mle.rs:56-83): a minor allele whose frequency tracks another's across the pools is
    dropped from X, and the reference fills only the first pw rows of its zero matrix (rows of removed columns stay beta
    0, v_b 0, t NaN, p 0, whichever column was removed).  Three mutually collinear columns take two removals, the
    second through the reference's `i -= 1` re-scan.  The zero-row pattern equals the oracle's exactly, the filled rows
    are held to the declared tolerance."""
    n, L, k = 40, 24, 2
    rng = np.random.default_rng(1000 * m + 10 * len(groups[0]) + groups[0][-1])
    counts = np.stack([_collinear_locus(rng, n, m, groups) for _ in range(L)])
    phen = rng.standard_normal((n, k))
    fs, codes = _fs(n), np.arange(6, dtype=np.uint8)
    dev = pb.mle_iterate(ctx, counts, phen, fs, codes)
    orc = pgo.scan_batch(pgo.SCAN_MLE, counts, codes, phen, H.oracle_fs(fs), 8)
    both, _ = check_mle_status(counts, codes, fs, dev, orc, f"collinear m={m} {groups}")
    assert both.all() and (dev.n_out == m).all()
    removed = sum(len(g) - 1 for g in groups)
    zo = zero_rows(orc.stat[:, :m], orc.var[:, :m], orc.t[:, :m], orc.pval[:, :m])
    assert (zo.sum(axis=1) == removed).all(), "the constructed design removes a different number of columns"
    assert (zo[:, m - removed:].all()) and not zo[:, :m - removed].any()
    compare_mle(dev, orc, both, n, f"collinear m={m} {groups}")


@pytest.mark.parametrize("values", [(0.25,), (1 / 3,), (0.1,), (1 / 3, 0.1), (0.3, 0.1), (0.25, 0.1)],
                         ids=["0.25", "1/3", "0.1", "1/3+0.1", "0.3+0.1", "0.25+0.1"])
def test_mle_iter_constant_allele(ctx, values):
    """A minor allele whose frequency is the same in every pool is a multiple of the intercept: X'X is singular in exact
    arithmetic.  Pinned on the device (DESIGN.md 11): such a column is recognised exactly (every pool the same double)
    and centred to zero, so it is never removed as collinear, never removes another column, and the locus is
    LOCUS_FAILED ("Non-invertible x_matrix").  The reference's outcome turns on the last bit of its sequential mean (0.25
    centres to 0 exactly, 1/3 and 0.1 to a pool-count dependent residue): it may solve the locus, so OK against FAILED
    is allowed there (cond > 1e12) and nothing else; keep-mask and allele order exact, nothing raises."""
    k = 1
    rng = np.random.default_rng(int(1e6 * sum(values)))
    rows = []
    for n in (12, 13, 18, 19, 24, 25, 30):
        for pos in range(3 - len(values) + 1):
            for _ in range(2):
                depth = 600
                mc = np.zeros((3, n))
                free = [a for a in range(3) if not (pos <= a < pos + len(values))]
                for e, v in enumerate(values):
                    mc[pos + e] = round(v * depth)
                for a, mu in zip(free, (0.12, 0.05)):
                    mc[a] = np.round(depth * mu * rng.uniform(0.3, 1.7, n))
                # the constant columns sort by their mean into the position asked for only if the others allow it:
                # whatever order the filter's sort gives, the column is constant
                rows.append((n, _locus(mc.astype(np.uint32), depth)))
    checked = {"failed_both": 0, "oracle_ok": 0}
    for n in sorted({r[0] for r in rows}):
        counts = np.stack([c for nn, c in rows if nn == n])
        phen = rng.standard_normal((n, k))
        fs, codes = _fs(n), np.arange(6, dtype=np.uint8)
        dev = pb.mle_iterate(ctx, counts, phen, fs, codes)
        orc = pgo.scan_batch(pgo.SCAN_MLE, counts, codes, phen, H.oracle_fs(fs), 8)
        both, why = check_mle_status(counts, codes, fs, dev, orc, f"constant {values} n={n}")
        assert (dev.status == pb.LOCUS_FAILED).all(), f"n={n}: device statuses {dev.status}"
        assert not both.any()
        p = dev.stats[..., 3]
        assert (np.isnan(p) | ((p >= 0) & (p <= 1))).all()
        checked["oracle_ok"] += int((orc.status == pgo.OK).sum())
        checked["failed_both"] += int((orc.status == pgo.FAILED).sum())
    print(f"constant allele {values}: {checked}")
