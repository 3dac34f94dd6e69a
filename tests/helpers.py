"""Shared parity helpers: run the CPU oracle and the CUDA path on the same loci and compare.

Tolerances (BASELINE.json north_star): keep-mask, kept-allele set and allele order bit-exact;
beta / SE / t within RTOL = 1e-9 relative; p-values within PTOL = 1e-6 relative with the absolute
floor 2.3e-16 that the reference's own `2 * (1 - cdf)` cancellation imposes (SURVEY.md H4).
beta is compared relative to max(|beta|, SE): a coefficient that is zero within its own standard
error has no meaningful relative error below SE * 1e-9.  Loci whose design matrix is so
ill-conditioned that two correct f64 algorithms legitimately differ (SURVEY.md H5) are arbitrated by a
50-digit mpmath solve: the device passes if it is at least as close to the exact answer as 4x the
oracle's own error (or within RTOL of it).
"""
from __future__ import annotations

import json
import os

import numpy as np

from oracle import pgo

HERE = os.path.dirname(os.path.abspath(__file__))
RTOL = 1e-9
PTOL = 1e-6
P_FLOOR = 2.3e-16


def load_c1():
    """config C1: the reference's tests/test.sync + tests/test.csv (committed fixture)."""
    z = np.load(os.path.join(HERE, "golden", "c1_sync.npz"))
    counts = np.ascontiguousarray(z["counts"].astype(np.uint32).transpose(0, 2, 1))  # [L, 6, n]
    with open(os.path.join(HERE, "golden", "c1_phen.json")) as fh:
        ph = json.load(fh)
    raw = ph["pool_sizes_raw"]
    tot = 0.0
    for v in raw:  # phen.rs:82-84 pool sizes normalised by their sequential sum
        tot = tot + v
    pool_sizes = np.array([v / tot for v in raw])
    phen = np.array(ph["phen"], dtype=np.float64)
    return dict(counts=counts, codes=np.arange(6, dtype=np.uint8), phen=phen, pool_sizes=pool_sizes,
                chrom_names=z["chrom_names"], chrom_idx=z["chrom_idx"], pos=z["pos"])


def student_t_cutoffs(df):
    """statrs' two cut-offs of the Student-t tail as (t_one, t_zero): checked_beta_reg sets bt = 0 when
    x = df / (df + t^2) is within 4 ulps of 1 (x >= 1 - 4 * 2^-53) or below 1e-10, so the reference's two-sided p is
    exactly 1 for |t| <= t_one and exactly 0 for |t| >= t_zero.  x is formed in f64 without contraction (Python
    floats), and is non-increasing in t, so each edge is found by bisection on the bit patterns of non-negative doubles
    (the restatement of pg_ptable.h's student_t_cutoffs)."""
    import struct

    def dbl(u):
        return struct.unpack("<d", struct.pack("<Q", u))[0]

    def x_of(t):
        return df / (df + t * t)

    lo, hi = 0, 0x7FF0000000000000
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if x_of(dbl(mid)) >= 1.0 - 4.0 * 2.0 ** -53:
            lo = mid
        else:
            hi = mid
    t_one = dbl(lo)
    lo, hi = 0, 0x7FF0000000000000
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if abs(x_of(dbl(mid))) < 1e-10:
            hi = mid
        else:
            lo = mid
    return t_one, dbl(hi)


def student_t_p(t, df):
    """the reference's two-sided p of each |t| (src/gwas/ols.rs:153): 2 * (1 - StudentsT(0, 1, df).cdf(|t|))"""
    t = np.abs(np.asarray(t, dtype=np.float64))
    return np.array([2.0 * (1.0 - pgo.students_t_cdf(float(v), float(df))) for v in t.ravel()]).reshape(t.shape)


def oracle_fs(fs):
    return pgo.FilterStats(pool_sizes=np.asarray(fs.pool_sizes, dtype=np.float64), remove_ns=fs.remove_ns,
                           min_coverage_depth=fs.min_coverage_depth,
                           min_allele_frequency=fs.min_allele_frequency,
                           max_missingness_rate=fs.max_missingness_rate)


def _design(counts_locus, codes, ofs):
    """X = [1 | sorted kept freqs without the major allele] exactly as ols_iterate builds it."""
    c = counts_locus.T.astype(np.uint64)  # n x A
    st, ck, ak = pgo.filter_locus(c, codes, ofs)
    assert st == pgo.OK
    f = pgo.to_frequencies(ck)
    f, ak = pgo.sort_by_allele_freq(f, ak, True)
    f = f[:, 1:]
    return np.hstack([np.ones((f.shape[0], 1)), f])


def _hp_solve_square(X, y):
    """the coefficients of a design with as many pools as coefficients (X b = y) or fewer (the minimum-norm solution
    X'(XX')^-1 y of src/gwas/ols.rs:67-75) at 50 digits; y [n, k] -> b[i][j] floats, or None"""
    import mpmath as mp
    mp.mp.dps = 50
    Xm = mp.matrix(X.tolist())
    try:
        b = (Xm ** -1) * mp.matrix(y.tolist()) if X.shape[0] == X.shape[1] else Xm.T * ((Xm * Xm.T) ** -1) * mp.matrix(y.tolist())
    except ZeroDivisionError:
        return None
    return [[float(b[i, j]) for j in range(y.shape[1])] for i in range(X.shape[1])]


def _hp_ols(X, y):
    import mpmath as mp
    mp.mp.dps = 50
    n, p = X.shape
    Xm = mp.matrix(X.tolist())
    ym = mp.matrix([[v] for v in y.tolist()])
    XtX = Xm.T * Xm
    try:
        inv = XtX ** -1
    except ZeroDivisionError:
        return None
    b = inv * (Xm.T * ym)
    e = ym - Xm * b
    ee = (e.T * e)[0]
    dfe = n - p
    if dfe <= 0:
        return None
    ve = ee / dfe
    ybar = sum(ym) / n
    syy = sum((v - ybar) ** 2 for v in ym)
    out = []
    for i in range(p):
        vb = ve * inv[i, i]
        se = mp.sqrt(vb)
        out.append((float(b[i]), float(se), float(b[i] / se) if se != 0 else float("nan")))
    return out, float(ee / syy) if syy != 0 else 0.0


def compare_regression(kind, counts, codes, phen, fs, dev, n_threads=8, label=""):
    """Returns a dict of statistics; raises AssertionError on any parity violation."""
    import poolgen_b200 as pb
    ofs = oracle_fs(fs)
    y = np.asarray(phen, dtype=np.float64)
    if y.ndim == 1:
        y = y[:, None]
    k = y.shape[1]
    n = counts.shape[2]
    orc = pgo.scan_batch(pgo.SCAN_OLS if kind == pb.KIND_OLS else pgo.SCAN_CORR, counts, codes, y, ofs, n_threads)
    L = counts.shape[0]
    assert dev.status.shape[0] == L
    # 1. keep-mask, bit-exact
    o_filtered = orc.status == pgo.FILTERED
    d_filtered = dev.status == pb.LOCUS_FILTERED
    bad = np.nonzero(o_filtered != d_filtered)[0]
    assert bad.size == 0, f"{label}: keep-mask differs at loci {bad[:10]} (oracle {orc.status[bad[:10]]}, device {dev.status[bad[:10]]})"
    assert not (orc.status == pgo.PANIC).any(), "oracle reported a reference panic"
    o_ok = orc.status == pgo.OK
    d_ok = dev.status == pb.LOCUS_OK
    both = o_ok & d_ok
    S = dev.stats.shape[1]
    # 2. kept-allele set and order, bit-exact (also for loci whose solve disagrees)
    cand = np.nonzero(o_ok & (dev.status != pb.LOCUS_UNSUPPORTED))[0]
    cand_ok = cand[d_ok[cand]]
    assert (orc.n_out[cand_ok] == dev.n_out[cand_ok]).all(), f"{label}: number of output rows differs"
    assert (orc.allele[cand_ok] == dev.alleles[cand_ok]).all(), f"{label}: allele order differs"
    stats = dict(loci=L, kept=int((~o_filtered).sum()), ok=int(both.sum()), arbitrated=0, unpinnable=0,
                 max_rel_beta=0.0, max_rel_se=0.0, max_rel_t=0.0, max_rel_p=0.0)
    idx = np.nonzero(both)[0]
    if idx.size == 0:
        return stats
    slot = np.arange(S)[None, :] < orc.n_out[idx][:, None]  # [m, S]
    o_stat = orc.stat[idx][:, :S, :]
    o_p = orc.pval[idx][:, :S, :]
    d_stat = dev.stats[idx][..., 0]
    d_p = dev.stats[idx][..., 3]
    fm_o = orc.freq_mean[idx][:, :S]
    fm_d = dev.freq_mean[idx]
    m3 = np.broadcast_to(slot[:, :, None], o_stat.shape)
    with np.errstate(invalid="ignore", divide="ignore"):
        fm_err = np.abs(fm_d - fm_o) / np.maximum(np.abs(fm_o), 1e-300)
    fm_err = np.where(np.isnan(fm_o) & np.isnan(fm_d), 0.0, fm_err)
    assert (fm_err[slot] <= RTOL).all(), f"{label}: mean frequency differs (max rel {np.nanmax(fm_err[slot])})"
    if kind == pb.KIND_OLS:
        o_se = np.sqrt(orc.var[idx][:, :S, :])
        o_t = orc.t[idx][:, :S, :]
        d_se = dev.stats[idx][..., 1]
        d_t = dev.stats[idx][..., 2]
        with np.errstate(invalid="ignore", divide="ignore"):
            # (fewer pools than coefficients: the reference's variance is rounding noise, often negative -> NaN root)
            e_b = np.abs(d_stat - o_stat) / np.maximum(np.abs(o_stat), np.nan_to_num(np.abs(o_se), nan=0.0, posinf=0.0))
            e_se = np.abs(d_se - o_se) / np.abs(o_se)
            e_t = np.abs(d_t - o_t) / np.maximum(np.abs(o_t), 1.0)
            e_p = np.abs(d_p - o_p) / (np.abs(o_p) + P_FLOOR / PTOL)
        # a pool without coverage (only reachable with --min-coverage-depth 0) puts NaN into X: beta, SE and t are
        # NaN on both sides and p is forced to 1 (src/gwas/ols.rs:150-151)
        nanrow = np.isnan(o_stat) & np.isnan(d_stat)
        e_b = np.where(nanrow, 0.0, e_b)
        e_se = np.where(nanrow & np.isnan(d_se), 0.0, e_se)
        e_t = np.where(nanrow & np.isnan(d_t) & np.isnan(o_t), 0.0, e_t)
        o_se = np.where(nanrow, 0.0, o_se)
        o_t = np.where(nanrow, 0.0, o_t)
        d_se = np.where(nanrow, 0.0, d_se)
        d_t = np.where(nanrow, 0.0, d_t)
        # saturated models (n == number of coefficients): the residual is rounding noise in the reference
        saturated = (orc.n_out[idx].astype(int) + 1 >= n)
        fail = m3 & ~((e_b <= RTOL) & ((e_se <= RTOL) | saturated[:, None, None]) &
                      ((e_t <= RTOL) | saturated[:, None, None]) & (e_p <= PTOL))
        fail |= m3 & ~np.isfinite(np.where(saturated[:, None, None], 0.0, d_se + d_t)) & np.isfinite(o_se + o_t)
        bad_loci = np.unique(np.nonzero(fail)[0])
        for bl in bad_loci:
            l = idx[bl]
            X = _design(counts[l], codes, ofs)
            cond = np.linalg.cond(X.T @ X) if X.shape[0] >= X.shape[1] else np.linalg.cond(X @ X.T)
            if saturated[bl]:
                # only beta and p are pinned (p = 1 in the reference through t = 0 / NaN).  The reference inverts X'X
                # (condition number squared) by LU, so with as many coefficients as pools its own beta is off by
                # cond * epsilon: the arbiter is the 50-digit solution, and the device may be as far from it as the
                # oracle is (times 4), or within the conditioning bound
                okb = bool((np.nan_to_num(e_b[bl][m3[bl]], nan=np.inf) <= max(RTOL, cond * 1e-15)).all())
                if not okb and np.isfinite(cond) and cond < 1e13:
                    hp = _hp_solve_square(X, y)
                    if hp is not None:
                        okb = True
                        for j in range(k):
                            bnorm = max(abs(hp[i][j]) for i in range(len(hp)))   # the conditioning bound is norm-wise
                            for s_ in range(int(orc.n_out[l])):
                                hv, dv, ov = hp[s_ + 1][j], d_stat[bl, s_, j], o_stat[bl, s_, j]
                                if not (abs(dv - hv) <= max(RTOL * abs(hv), 4.0 * abs(ov - hv), cond * 4e-16 * bnorm)):
                                    okb = False
                assert okb or not (cond < 1e13), \
                    f"{label}: saturated locus {l} beta differs (cond {cond:.3g}): device {d_stat[bl][m3[bl]]} oracle {o_stat[bl][m3[bl]]}"
                stats["unpinnable"] += 1
                continue
            arb_ok = True
            for j in range(k):
                hp = _hp_ols(X, y[:, j])
                if hp is None:
                    stats["unpinnable"] += 1
                    continue
                hp, resid_ratio = hp
                # an exact fit (residual below f64 resolution): SE, t and p are rounding noise in the reference
                perfect = resid_ratio < 1e-24
                if perfect:
                    stats["unpinnable"] += 1
                for s in range(int(orc.n_out[l])):
                    hb, hse, ht = hp[s + 1]
                    if perfect:
                        hse = max(abs(float(o_se[bl, s, j])), abs(hb) * 1e-9)
                    for name, dv, ov, hv in (("beta", d_stat[bl, s, j], o_stat[bl, s, j], hb),
                                             ("se", d_se[bl, s, j], o_se[bl, s, j], hse),
                                             ("t", d_t[bl, s, j], o_t[bl, s, j], ht))[:1 if perfect else 3]:
                        scale = max(abs(hv), abs(hse) if name == "beta" else (1.0 if name == "t" else 0.0), 1e-300)
                        de, oe = abs(dv - hv) / scale, abs(ov - hv) / scale
                        if not (de <= max(RTOL, 4.0 * oe, cond * 4e-16)):
                            arb_ok = False
                            msg = f"{label}: locus {l} slot {s} phen {j} {name}: device {dv!r} oracle {ov!r} exact {hv!r} cond {cond:.3g}"
            assert arb_ok, msg
            stats["arbitrated"] += 1
        good = m3 & ~fail
        for key, e in (("max_rel_beta", e_b), ("max_rel_se", e_se), ("max_rel_t", e_t), ("max_rel_p", e_p)):
            v = e[good & np.isfinite(e)]
            stats[key] = float(v.max()) if v.size else 0.0
    else:
        d_raw = dev.stats[idx][..., 1]
        with np.errstate(invalid="ignore", divide="ignore"):
            e_r = np.abs(d_stat - o_stat)
            e_p = np.abs(d_p - o_p) / (np.abs(o_p) + P_FLOOR / PTOL)
        nan_both = np.isnan(o_stat) & np.isnan(d_stat)
        # r is rounded to 7 digits (correlation_test.rs:70): a last-bit difference of the raw r may move the rounded
        # value by one unit of 1e-7 at a rounding boundary
        okr = nan_both | (e_r <= 1.0000001e-7)
        assert (okr | ~m3).all(), f"{label}: r differs (max {np.nanmax(e_r[m3])})"
        # a perfect correlation (always the case with two pools): s2 = (1 - r^2) / (n - 2) is 0, a negative rounding
        # residue or 0 / 0, and correlation_test.rs:57-66 returns the unrounded r with p = epsilon, or NaN, depending
        # on the last bit of r -- nothing beyond |r| = 1 to 1e-7 can be pinned there
        perfect = np.abs(o_stat) >= 0.9999999 - 1e-12     # the rounded r is 1 or 0.9999999: 1 - r^2 below 3e-7
        m3 = m3 & ~perfect
        exact = (e_r == 0) | nan_both
        stats["r_exact_fraction"] = float(exact[m3].mean()) if m3.any() else 1.0
        assert stats["r_exact_fraction"] > 0.999, f"{label}: too many rounded r differ: {stats['r_exact_fraction']}"
        rounded_again = np.round(d_raw * 1e7) / 1e7
        assert ((np.abs(rounded_again - d_stat) <= 1e-15) | ~m3 | np.isnan(d_raw) | (np.abs(d_raw) >= 1.0)).all()
        okp = (np.isnan(o_p) & np.isnan(d_p)) | (e_p <= PTOL)
        badp = m3 & ~okp
        assert not badp.any(), f"{label}: p differs: device {d_p[badp][:5]} oracle {o_p[badp][:5]}"
        v = e_p[m3 & np.isfinite(e_p)]
        stats["max_rel_p"] = float(v.max()) if v.size else 0.0
    # loci the oracle solved but the device flagged as failed must be rank deficient
    for l in np.nonzero(o_ok & (dev.status == pb.LOCUS_FAILED))[0]:
        X = _design(counts[l], codes, ofs)
        assert np.linalg.cond(X.T @ X) > 1e12, f"{label}: device failed a well-conditioned locus {l}"
        stats["unpinnable"] += 1
    for l in np.nonzero((orc.status == pgo.FAILED) & d_ok)[0]:
        X = _design(counts[l], codes, ofs)
        assert np.linalg.cond(X.T @ X) > 1e12, f"{label}: oracle failed a well-conditioned locus {l}"
        stats["unpinnable"] += 1
    return stats


def compare_tables(kind, counts, codes, fs, dev, n_threads=8, label=""):
    import poolgen_b200 as pb
    ofs = oracle_fs(fs)
    orc = pgo.scan_batch(pgo.SCAN_CHISQ if kind == pb.KIND_CHISQ else pgo.SCAN_FISHER, counts, codes, None, ofs, n_threads)
    o_filtered = orc.status == pgo.FILTERED
    d_filtered = dev.status == pb.LOCUS_FILTERED
    bad = np.nonzero(o_filtered != d_filtered)[0]
    assert bad.size == 0, f"{label}: keep-mask differs at loci {bad[:10]}"
    o_ok = orc.status == pgo.OK
    assert ((dev.status == pb.LOCUS_OK) == o_ok).all(), f"{label}: status differs"
    assert ((dev.status == pb.LOCUS_PANIC) == (orc.status == pgo.PANIC)).all()
    idx = np.nonzero(o_ok)[0]
    assert (orc.n_out[idx] == dev.n_out[idx]).all()
    assert (orc.allele[idx] == dev.alleles[idx]).all()
    o_s, o_p = orc.stat[idx, 0, 0], orc.pval[idx, 0, 0]
    d_s, d_p = dev.stats[idx, 0, 0, 0], dev.stats[idx, 0, 0, 3]
    with np.errstate(invalid="ignore", divide="ignore"):
        e_s = np.abs(d_s - o_s) / np.maximum(np.abs(o_s), 1e-300)
        e_p = np.abs(d_p - o_p) / (np.abs(o_p) + P_FLOOR / PTOL)
    both_nan_s = np.isnan(o_s) & np.isnan(d_s)
    both_nan_p = np.isnan(o_p) & np.isnan(d_p)
    # a chi-square of identical rows is 0 in exact arithmetic and rounding noise (~1e-32) in any f64 evaluation: the
    # one-thread kernels reproduce the reference's noise, the one-warp-per-locus kernels have their own
    floor = 1e-24 if kind == pb.KIND_CHISQ else 0.0
    assert ((e_s <= RTOL) | both_nan_s | ((o_s == 0) & (np.abs(d_s) < 1e-300)) |
            (np.abs(d_s - o_s) <= floor)).all(), f"{label}: statistic differs, max rel {np.nanmax(e_s)}"
    assert ((e_p <= PTOL) | both_nan_p).all(), f"{label}: p differs, max rel {np.nanmax(e_p)}"
    return dict(loci=counts.shape[0], ok=int(o_ok.sum()),
                max_rel_stat=float(np.nanmax(e_s)) if idx.size else 0.0,
                max_rel_p=float(np.nanmax(e_p)) if idx.size else 0.0)
