"""Every Student-t p-value the device writes, held to the reference's p of the recorded t over the whole range of t.

A record's p is a function of its t and the analysis's degrees of freedom alone, so the expected p is
2 (1 - StudentsT::cdf(|t|)) of the device's own t (the oracle, whose tail test_student_t_tails.py pins to mpmath), with
the records' metric |d - o| <= PTOL |o| + P_FLOOR.  The data are planted so that t lands in every region where the
table lookup (pg_ptable.h, student_batch / student_two_sided_tab) or its edges can go wrong: the |t| <= epsilon gate,
statrs' two cut-offs (p exactly 1 up to t_one, exactly 0 from t_zero on), every 2^-12 step of w = 1 + |t| / sqrt(df)
in every octave up to where p is 0, the quantised-to-0 tail past the table's last interval, inf and NaN.  Each test
asserts that the recorded t populate those regions.  A |t| within 4 ulps of a cut-off is skipped: a last-bit
difference of t legitimately flips p between the cut-off's value and the tail there."""
from __future__ import annotations

import math
import os
import subprocess
import sys

import numpy as np
import pytest

import poolgen_b200 as pb
from tests import helpers as H

pytestmark = pytest.mark.gpu

EPS = 2.220446049250313e-16
T_REACH = 1e8  # planted t beyond this are not steered finely enough (f64 columns / 2^30 read depths) to hit one interval


def _near_cutoff(t, df):
    t_one, t_zero = H.student_t_cutoffs(df)
    a = np.abs(t)
    return (np.abs(a - t_one) <= 4 * np.spacing(t_one)) | (np.abs(a - t_zero) <= 4 * np.spacing(t_zero))


def _expected_p(t, df):
    """the reference's p of each recorded t; NaN t has p forced to 1 (ols.rs:150-151), |t| <= epsilon is t = 0"""
    e = np.where(np.isnan(t), 1.0, 0.0)
    fin = ~np.isnan(t)
    e[fin] = H.student_t_p(t[fin], df)
    return e


def _regions(t, df):
    """which of the regions of the tail the recorded t reach"""
    t_one, t_zero = H.student_t_cutoffs(df)
    a = np.abs(t)
    with np.errstate(invalid="ignore"):
        exp = _expected_p(t, df)
        return dict(gate=int((a <= EPS).sum()),
                    one=int(((a > EPS) & (a <= t_one)).sum()),
                    just_above_one=int(((a > t_one) & (a <= 4 * t_one)).sum()),
                    tail=int(((a > 4 * t_one) & (exp > 0)).sum()),
                    quantised_zero=int(((a < t_zero) & (exp == 0)).sum()),
                    zero=int(((a >= t_zero) & np.isfinite(a)).sum()),
                    inf=int(np.isinf(a).sum()),
                    nan=int(np.isnan(a).sum()))


def _check(t, p, df, label):
    t = np.asarray(t, dtype=np.float64).ravel()
    p = np.asarray(p, dtype=np.float64).ravel()
    keep = ~_near_cutoff(t, df)
    e = _expected_p(t[keep], df)
    d = p[keep]
    bad = ~(np.abs(d - e) <= H.PTOL * np.abs(e) + H.P_FLOOR)
    if bad.any():
        i = np.nonzero(bad)[0][:6]
        pytest.fail(f"{label} df={df}: {int(bad.sum())} p differ, e.g. |t| {np.abs(t[keep][i])!r} device {d[i]!r} "
                    f"reference {e[i]!r}")
    return _regions(t, df)


def _w_keys(t, df):
    """(octave, multiple of 2^-12) of w = 1 + |t| / sqrt(df)"""
    w = 1.0 + np.abs(t) / math.sqrt(df)
    m, e = np.frexp(w)  # w = m 2^e, m in [0.5, 1)
    return set(zip((e - 1).tolist(), np.floor((2.0 * m - 1.0) * 4096).astype(np.int64).tolist()))


def _sweep_targets(df):
    """|t| at the middle of every 2^-12 step of w in every octave, up to where the reference's p is 0 (or T_REACH)"""
    ts = []
    for e in range(0, 64):
        w = np.ldexp(1.0 + (np.arange(4096) + 0.5) / 4096.0, e)
        t = (w - 1.0) * math.sqrt(df)
        t = t[t <= T_REACH]
        if t.size == 0:
            break
        p_end = H.student_t_p(t[-1:], df)[0]
        ts.append(t)
        if p_end == 0.0:
            break
    return np.concatenate(ts)


def _edge_targets(df):
    t_one, t_zero = H.student_t_cutoffs(df)
    out = [t_one * f for f in (0.25, 0.5, 0.9, 0.999, 1.001, 1.1, 1.5, 2.0, 3.0)]
    out += [t_zero * f for f in (0.5, 0.9, 0.999, 1.001, 1.1, 2.0, 10.0)]
    out += [1e-12, 1e-9, 1e-6, 1e-3]
    return np.array([t for t in out if t <= T_REACH])


# ---- the covariate scan (ols_iter_with_kinship): one planted t per column ---------------------------------------------
def _plant_columns(y, cov, targets, rng):
    """columns g = alpha y~ + e with e centred and orthogonal to [1 | cov | y]: the last coefficient of y on
    [1 | cov | g] has t = alpha sqrt(dfe Y / E) (Y = y~'y~, E = e'e), so alpha is solved for each target"""
    n = y.shape[0]
    B = np.hstack([np.ones((n, 1)), cov])
    Qb, _ = np.linalg.qr(B)
    yt = y - Qb @ (Qb.T @ y)
    Q2, _ = np.linalg.qr(np.hstack([B, yt[:, None]]))
    dfe = n - 2 - cov.shape[1]
    P = targets.size
    E = rng.standard_normal((P, n))
    E -= (E @ Q2) @ Q2.T
    E -= (E @ Q2) @ Q2.T
    Y = yt @ yt
    EE = np.einsum("ij,ij->i", E, E)
    alpha = targets * np.sqrt(EE / (dfe * Y))
    return alpha[:, None] * yt[None, :] + E


@pytest.mark.parametrize("n,m", [(3, 0), (4, 0), (5, 0), (100, 0), (2000, 0), (2901, 0), (3500, 0), (4000, 0),
                                 (100, 4), (2000, 4), (2901, 4)])
def test_covariate_scan_p_over_the_whole_tail(ctx, n, m):
    """covar_kernel (m = 0), covar_mma_kernel (m = 4, k = 1: five vectors) and the explicit-residual list kernel
    (nearly constant columns, near-perfect fits); df = n - 1 for every column"""
    df = n - 1
    rng = np.random.default_rng(7000 + 10 * n + m)
    y = np.arange(n, dtype=np.float64)  # integers: y~ and the exact-fit column's sums are exact (t = inf)
    cov = rng.standard_normal((n, m))
    targets = np.concatenate([_sweep_targets(df), _edge_targets(df)])
    G = _plant_columns(y, cov, targets, rng)
    P0 = targets.size
    nan_col, const_col, fit_col = P0, P0 + 1, P0 + 2
    extra = [np.full(n, np.nan),                      # NaN frequencies: p forced to 1
             np.full(n, 0.25),                        # a constant column: singular, NaN records
             y.copy()]                                # an exact fit: rss 0 or rounding noise, t = inf or beyond t_zero
    # nearly constant columns (a rare allele) take the explicit-residual list kernel
    near = 0.999 + 1e-7 * _plant_columns(y, cov, np.array([1e-7, 1e-3, 1.0, 30.0, 1e3, 1e5]), rng)
    # orthogonal to y: b within rounding of 0, the |b| <= epsilon gate
    orth = _plant_columns(y, cov, np.zeros(4), rng)
    G = np.vstack([G, np.array(extra), near, orth])
    kin = pb.Kinship(ctx, n, G.shape[0])
    try:
        kin.append_columns(G)
        kin.set_covariates(cov)
        beta, var, pval = kin.covar_scan(y[:, None])
    finally:
        kin.close()
    beta, var, pval = beta[0], var[0], pval[0]
    assert np.isnan(beta[const_col]) and np.isnan(beta[nan_col]) and pval[nan_col] == 1.0
    with np.errstate(invalid="ignore", divide="ignore"):
        t = np.where(np.abs(beta) <= EPS, 0.0, beta / np.sqrt(var))  # the kernels' b / sqrt(var)
    sel = np.ones(G.shape[0], dtype=bool)
    sel[const_col] = False
    t_one, t_zero = H.student_t_cutoffs(df)
    assert abs(t[fit_col]) >= t_zero and pval[fit_col] == 0.0, (t[fit_col], pval[fit_col])
    reg = _check(t[sel], pval[sel], df, f"covar n={n} m={m}")
    print(f"covar n={n} m={m}: {G.shape[0]} columns, regions {reg}")
    # (b is exactly 0 only by luck: y~ is formed on the host, so the orthogonal columns land in the gate or below t_one)
    assert reg["gate"] + reg["one"] > 0, f"covar n={n} m={m}: no t below t_one: {reg}"
    for r in ("just_above_one", "tail", "zero", "nan"):
        assert reg[r] > 0, f"covar n={n} m={m}: no t in region {r}: {reg}"
    assert reg["quantised_zero"] > 0 or df <= 3, reg
    want = _w_keys(targets[(targets > 0) & (H.student_t_p(targets, df) > 0)], df)
    got = _w_keys(t[np.isfinite(t)], df)
    assert want <= got, f"covar n={n} m={m}: {len(want - got)} steps of w not reached, e.g. {sorted(want - got)[:5]}"


# ---- the kinship MLE scan (mle_iter_with_kinship): t = beta / var -----------------------------------------------------
@pytest.mark.parametrize("n", [3, 4, 2901])
def test_kin_mle_scan_p_large_t(ctx, n):
    df = n - 1
    rng = np.random.default_rng(8100 + n)
    y = np.arange(n, dtype=np.float64) / n
    targets = np.concatenate([10.0 ** np.linspace(-8, 8, 161), _edge_targets(df)])
    G = 0.5 + 0.1 * _plant_columns(y, np.zeros((n, 0)), targets, rng) / np.maximum(1.0, targets[:, None])
    kin = pb.Kinship(ctx, n, G.shape[0])
    try:
        kin.append_columns(G)
        kin.set_covariates(np.zeros((n, 0)))
        beta, var, pval = kin.mle_scan(y[:, None])
    finally:
        kin.close()
    with np.errstate(invalid="ignore", divide="ignore"):
        t = beta[0] / var[0]  # mle.rs:176: the variance, not its root
    reg = _check(t, pval[0], df, f"kin mle n={n}")
    print(f"{'kin mle'} n={n}: regions {reg}")
    assert reg["tail"] > 0 and (reg["zero"] + reg["quantised_zero"]) > 0, reg
    if df <= 3:
        assert reg["zero"] > 0, f"kin mle n={n}: no t beyond t_zero: {reg}"


# ---- ols_iter / pearson_corr scan: u32 count slabs, the records carry t ----------------------------------------------
D = 1 << 29  # reads per allele column of a pool: frequencies steered to 2^-30


def _counts_from_minor(f_minor, rare_reads=False):
    """[L, A, n] u32 counts of two alleles with these minor-allele frequencies (+ a third allele of one read below
    the MAF threshold in some pools of every other locus: a removed allele that carries reads)"""
    L, n = f_minor.shape
    tot = 2 * D
    c0 = np.rint(f_minor * tot).astype(np.int64)
    out = np.zeros((L, 3, n), dtype=np.uint32)
    out[:, 0] = tot - c0
    out[:, 1] = c0
    if rare_reads:
        out[::2, 2, ::3] = 1
    return out


def _few_pool_loci(n, y, rng):
    """near-collinear frequency vectors: minor frequency 0.3 + 0.1 (y~ + delta e) / |y~|, delta on a log grid"""
    yt = y - y.mean()
    yt /= np.abs(yt).max()
    deltas = np.concatenate([10.0 ** np.linspace(-10, 1, 300), [0.0]])
    E = rng.standard_normal((deltas.size, n))
    E -= E.mean(axis=1, keepdims=True)
    E -= np.outer(E @ yt / (yt @ yt), yt)
    E /= np.abs(E).max(axis=1, keepdims=True)
    return 0.3 + 0.1 * (yt[None, :] + deltas[:, None] * E) / (1.0 + deltas[:, None])


def _many_pool_loci(n, rng):
    """pools in pairs of opposite centred phenotype and equal frequency (t = 0), then k reads moved in pool 0: t grows
    with k through 1e-7 .. 3e-6 (statrs' t_one is 1.26e-6 .. 1.78e-6 at 2,899 .. 6,143 degrees of freedom)"""
    half = rng.uniform(0.5, 1.5, n // 2)
    y = np.empty(n)
    y[0::2][: n // 2], y[1::2][: n // 2] = half, -half
    if n % 2:
        y[-1] = 0.0
    fpair = rng.uniform(0.2, 0.4, (n + 1) // 2)
    f = np.repeat(fpair, 2)[:n]
    counts = _counts_from_minor(f[None, :])[0]
    # t per moved read, measured with the oracle's ols on one locus
    return y, counts


def _scan_records(ctx, kind, counts, phen, n, stream):
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    codes = np.array([0, 1, 2], dtype=np.uint8)
    scan = pb.Scan(ctx, kind, fs, n, codes, phen)
    try:
        if not stream:
            return scan.run_counts(counts)
        scan.stream_begin(512)
        parts = [scan.collect(scan.submit_counts(np.ascontiguousarray(counts[l0:l0 + 512])))
                 for l0 in range(0, counts.shape[0], 512)]
        return pb.ScanResults(np.concatenate([p.status for p in parts]), np.concatenate([p.n_out for p in parts]),
                              np.concatenate([p.alleles for p in parts]), np.concatenate([p.freq_mean for p in parts]),
                              np.concatenate([p.stats for p in parts]))
    finally:
        scan.close()


def _scan_check(res, kind, n, label):
    ok = res.status == pb.LOCUS_OK
    assert ok.sum() > 0.9 * res.status.size, f"{label}: only {ok.sum()} of {res.status.size} loci kept"
    st = res.stats[ok][:, 0]  # slot 0: [loci, k, 4]
    df = n - 1 if kind == pb.KIND_OLS else n - 2
    t, p = st[..., 2], st[..., 3]
    if kind == pb.KIND_CORR:
        perfect = np.isnan(t) & ~np.isnan(st[..., 1])   # |r| >= 1: p = epsilon (correlation_test.rs:57-66)
        assert np.all(p[perfect] == EPS), f"{label}: |r| >= 1 records must carry p = epsilon"
        has_r = ~np.isnan(st[..., 1])
        t, p = t[~perfect & has_r], p[~perfect & has_r]
    reg = _check(t, p, df, label)
    print(f"{label}: regions {reg}")
    return reg, df


@pytest.mark.parametrize("stream", [False, True])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("kind,n", [(pb.KIND_OLS, 3), (pb.KIND_OLS, 4), (pb.KIND_OLS, 5),
                                    (pb.KIND_CORR, 3), (pb.KIND_CORR, 4), (pb.KIND_CORR, 5)])
def test_scan_p_few_pools(ctx, kind, n, k, stream):
    """near-perfect fits at 3-5 pools: t up to ~1e8, through statrs' t_zero (1.0e5 .. 1.7e5 at 1 .. 3 degrees of
    freedom), where the table used to print p up to 6e-6 for a reference 0"""
    rng = np.random.default_rng(9000 + 10 * n + kind)
    y = rng.standard_normal(n)
    f = _few_pool_loci(n, y, rng)
    counts = _counts_from_minor(f, rare_reads=True)
    phen = np.stack([y, -2.0 * y + 1.0, rng.standard_normal(n)][:k], axis=1)
    res = _scan_records(ctx, kind, counts, phen, n, stream)
    reg, df = _scan_check(res, kind, n, f"kind={kind} n={n} k={k} stream={stream}")
    assert reg["tail"] > 0, reg
    if df <= 3:
        assert reg["zero"] > 0, f"kind={kind} n={n}: no t beyond t_zero: {reg}"


@pytest.mark.parametrize("stream", [False, True])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("n", [2900, 4097, 6144])
def test_ols_scan_p_near_t_one(ctx, n, k, stream):
    """|t| in 1e-7 .. 3e-6 at 2,899 .. 6,143 degrees of freedom: the reference's p is exactly 1 up to t_one, where the
    table used to print 1 - 1.4e-6"""
    rng = np.random.default_rng(9500 + n)
    y, base = _many_pool_loci(n, rng)
    from oracle import pgo
    x1 = np.ones((n, 2))
    f0 = base[1].astype(np.float64) / (2 * D)
    x1[:, 1] = f0
    x1[0, 1] = (float(base[1, 0]) + 1000.0) / (2 * D)
    _, _, _, _, t1000 = pgo.ols(x1, y)
    per_read = abs(float(t1000[1, 0])) / 1000.0
    t_one, _ = H.student_t_cutoffs(n - 1)
    targets = np.concatenate([10.0 ** np.linspace(-7, math.log10(3e-6), 120), t_one * np.array([0.9, 0.99, 1.01, 1.1])])
    moves = np.unique(np.rint(targets / per_read).astype(np.int64))
    counts = np.repeat(base[None], moves.size + 1, axis=0)
    counts[1:, 1, 0] += moves.astype(np.uint32)
    counts[1:, 0, 0] -= moves.astype(np.uint32)
    phen = np.stack([y, -2.0 * y, np.roll(y, 2)][:k], axis=1)
    res = _scan_records(ctx, pb.KIND_OLS, counts, phen, n, stream)
    reg, _ = _scan_check(res, pb.KIND_OLS, n, f"ols n={n} k={k} stream={stream}")
    assert reg["one"] > 0 and reg["just_above_one"] > 0, f"ols n={n}: t did not straddle t_one: {reg}"


# ---- mle_iter: t = beta / v_b ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3, 4, 2901])
def test_mle_iter_p_large_t(ctx, n):
    rng = np.random.default_rng(9900 + n)
    y = rng.standard_normal(n)
    f = _few_pool_loci(n, y, rng)
    counts = _counts_from_minor(f)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    res = pb.mle_iterate(ctx, counts, y[:, None], fs, allele_codes=np.array([0, 1, 2], dtype=np.uint8))
    ok = res.status == pb.LOCUS_OK
    assert ok.sum() > 0.9 * ok.size
    st = res.stats[ok][:, 0, 0]
    reg = _check(st[:, 2], st[:, 3], n - 1, f"mle_iter n={n}")
    print(f"{'mle_iter'} n={n}: regions {reg}")
    assert reg["tail"] > 0 and (reg["zero"] + reg["quantised_zero"]) > 0, reg


# ---- the same scans through the continued fraction and through the fix-up kernel -------------------------------------
def test_continued_fraction_fallback(ctx, monkeypatch):
    """PG_PVALUE=cf (read at every pg_scan_open): the device's continued fraction is statrs' own arithmetic, so it
    agrees with the oracle to 1e-12 relative plus one quantum, inside the cut-offs too"""
    monkeypatch.setenv("PG_PVALUE", "cf")
    for kind, n, k in ((pb.KIND_OLS, 3, 3), (pb.KIND_CORR, 4, 1), (pb.KIND_OLS, 2900, 1)):
        rng = np.random.default_rng(9000 + 10 * n + kind)
        if n < 10:
            y = rng.standard_normal(n)
            counts = _counts_from_minor(_few_pool_loci(n, y, rng))
            phen = np.stack([y, -2.0 * y + 1.0, rng.standard_normal(n)][:k], axis=1)
        else:
            y, base = _many_pool_loci(n, rng)
            counts = np.repeat(base[None], 200, axis=0)
            mv = np.unique(np.rint(10.0 ** np.linspace(3, 6, 199)).astype(np.uint32))
            counts[1:1 + mv.size, 1, 0] += mv
            counts[1:1 + mv.size, 0, 0] -= mv
            phen = y[:, None]
        res = _scan_records(ctx, kind, counts, phen, n, False)
        ok = res.status == pb.LOCUS_OK
        st = res.stats[ok][:, 0]
        t, p = st[..., 2].ravel(), st[..., 3].ravel()
        df = n - 1 if kind == pb.KIND_OLS else n - 2
        keep = ~np.isnan(t) & ~_near_cutoff(t, df)
        e = _expected_p(t[keep], df)
        err = np.abs(p[keep] - e)
        assert np.all(err <= 1e-12 * e + H.P_FLOOR), f"cf kind={kind} n={n}: max {err.max()}"
        reg = _regions(t, df)
        assert reg["one"] + reg["zero"] > 0, reg


def test_fixup_path_without_ingest_hints():
    """PG_NOHINT=1 (read once per process) sends the loci whose removed allele carries reads through the fix-up
    kernel's renormalising path: the few-pool scan cases must hold there too"""
    if os.environ.get("PG_NOHINT"):
        pytest.skip("already inside the no-hint run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PG_NOHINT="1")
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_student_t_tails_gpu.py"),
                          "-m", "gpu", "-q", "-x", "-k", "test_scan_p_few_pools and not True"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=root, env=env, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:]
    assert " passed" in out.stdout
