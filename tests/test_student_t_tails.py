"""The expectation side of every Student-t p-value the device writes: the oracle's StudentsT::cdf (statrs 0.16,
oracle/poolgen_oracle.c) against a 50-digit mpmath tail over the whole range of t, and statrs' two cut-offs.

checked_beta_reg sets bt = 0 when x = df / (df + t^2) is below 1e-10 or within 4 ulps of 1, so the reference's p is
exactly 0 from t_zero on and exactly 1 up to t_one, whatever the tail is there.  Between them, 2 (1 - cdf) is the
regularised incomplete beta I_x(df/2, 1/2) of the f64 x the reference forms, to 1e-12 relative plus one quantum of the
final 2 (1 - (1 - ib)) (2.3e-16), plus the offset d of statrs' own ln_gamma in ln B(df/2, 1/2): up to 6e-12 at a few
thousand degrees of freedom, a relative error d of the prefactor bt, which the symmetric branch p = 1 - bt h / b turns
into d (1 - p) / p.  The exception is where statrs' continued fraction stops at its 140-term cap before it has
converged (t near sqrt(3), the switch to the symmetric branch, at hundreds of degrees of freedom and more).  There the
reference departs from the exact tail by up to ~5e-8 relative, still 20x inside the 1e-6 tolerance of the records.
The GPU tests (test_student_t_tails_gpu.py) hold the device to these values."""
from __future__ import annotations

import math

import numpy as np
import pytest

from oracle import pgo
from tests import helpers as H

DFS = [1, 2, 3, 4, 9, 99, 999, 1999, 2899, 4999, 6143]
QUANTUM = 2.3e-16
MPMATH_RTOL = 1e-12
UNCONVERGED_RTOL = 1e-7


def _exact_tail(df, x):
    """I_x(df/2, 1/2) at 50 digits for the f64 x the reference forms"""
    import mpmath as mp
    mp.mp.dps = 50
    return mp.betainc(mp.mpf(df) / 2, mp.mpf(1) / 2, 0, mp.mpf(x), regularized=True)


def _ln_beta_offset(df):
    """|ln B(df/2, 1/2)| of statrs' Lanczos ln_gamma minus the exact value: a relative offset of every p"""
    import mpmath as mp
    mp.mp.dps = 50
    a = df / 2.0
    lnb = pgo.ln_gamma(a + 0.5) - pgo.ln_gamma(a) - pgo.ln_gamma(0.5)
    return abs(float(lnb - (mp.loggamma(mp.mpf(a) + 0.5) - mp.loggamma(mp.mpf(a)) - mp.loggamma(mp.mpf(0.5)))))


def _cf_converges(df, x):
    """whether statrs' Lentz continued fraction (checked_beta_reg) meets its stopping rule within its 140 terms"""
    a, b = df / 2.0, 0.5
    if x >= (a + 1.0) / (a + b + 2.0):
        a, b, x = b, a, 1.0 - x
    eps, fpmin = 1.1102230246251565e-16, 2.2250738585072014e-308 / 1.1102230246251565e-16
    qab, qap, qam = a + b, a + 1.0, a - 1.0
    c, d = 1.0, 1.0 - qab * x / qap
    d = 1.0 / (fpmin if abs(d) < fpmin else d)
    for mi in range(1, 141):
        m = float(mi)
        m2 = m * 2.0
        for aa in (m * (b - m) * x / ((qam + m2) * (a + m2)), -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2))):
            d = 1.0 + aa * d
            d = fpmin if abs(d) < fpmin else d
            c = 1.0 + aa / c
            c = fpmin if abs(c) < fpmin else c
            d = 1.0 / d
        if abs(d * c - 1.0) <= eps:
            return True
    return False


def _grid(df):
    """|t| on a log grid from 1e-12 to 1e16 (6 points per decade), a finer sweep of 0.01 .. 100 x sqrt(df) where the
    tail moves, and each cut-off double with its neighbours"""
    t_one, t_zero = H.student_t_cutoffs(df)
    ts = list(10.0 ** np.linspace(-12, 16, 169)) + list(math.sqrt(df) * 10.0 ** np.linspace(-2, 2, 121))
    for c in (t_one, t_zero):
        ts += [c, math.nextafter(c, 0.0), math.nextafter(c, math.inf)]
    return np.array(sorted(set(float(t) for t in ts))), t_one, t_zero


@pytest.mark.parametrize("df", DFS)
def test_oracle_tail_against_mpmath(df):
    ts, t_one, t_zero = _grid(df)
    n_inside, n_tail, n_unconverged = 0, 0, 0
    offset = _ln_beta_offset(df)
    for t in ts:
        p = 2.0 * (1.0 - pgo.students_t_cdf(t, float(df)))
        if t <= t_one:
            assert p == 1.0, f"df={df} |t|={t!r} <= t_one: p={p!r}"
            n_inside += 1
            continue
        if t >= t_zero:
            assert p == 0.0, f"df={df} |t|={t!r} >= t_zero: p={p!r}"
            n_inside += 1
            continue
        x = df / (df + t * t)
        ref = _exact_tail(df, x)
        err = float(abs(p - ref))
        if _cf_converges(df, x):
            symm = x >= (df / 2.0 + 1.0) / (df / 2.0 + 2.5)
            rtol = MPMATH_RTOL + offset * (max(1.0, (1.0 - float(ref)) / float(ref)) if symm else 1.0)
            assert err <= rtol * float(ref) + QUANTUM, f"df={df} |t|={t!r}: oracle {p!r} exact {float(ref)!r}"
            n_tail += 1
        else:
            assert err <= UNCONVERGED_RTOL * float(ref), f"df={df} |t|={t!r} (140-term cap): oracle {p!r} exact {float(ref)!r}"
            n_unconverged += 1
    assert n_inside >= 6 and n_tail > 100, (n_inside, n_tail)
    # the 140-term cap is only ever short near the symmetric switch at hundreds of degrees of freedom and more
    assert n_unconverged == 0 or df >= 99, (df, n_unconverged)


@pytest.mark.parametrize("df", DFS)
def test_cutoffs_are_the_edges(df):
    """t_one / t_zero are the exact edges: p is 1 (0) on them and not one double beyond; NaN stays NaN, 0 and inf give
    1 and 0.  At df <= 3 the exact tail just inside t_zero is more than a quantum (the band the table used to print
    a non-zero p in), at larger df the quantisation has already made it 0."""
    t_one, t_zero = H.student_t_cutoffs(df)
    p = lambda t: 2.0 * (1.0 - pgo.students_t_cdf(t, float(df)))
    assert 0.0 < t_one < t_zero < math.inf
    assert p(t_one) == 1.0 and p(0.0) == 1.0
    assert p(math.nextafter(t_one, math.inf)) < 1.0
    assert p(t_zero) == 0.0 and p(math.inf) == 0.0 and p(1e300) == 0.0
    assert math.isnan(pgo.students_t_cdf(math.nan, float(df)))
    below = math.nextafter(t_zero, 0.0)
    if df <= 3:
        assert p(below) > QUANTUM
        assert abs(p(below) - float(_exact_tail(df, df / (df + below * below)))) <= 1e-12 * p(below) + QUANTUM
    # the edges in closed form: t_one^2 / df is a few units of 2^-53 (df + t^2 moves in steps of ulp(df)), and
    # t_zero^2 = df (1e10 - 1) to the rounding of x
    assert 2.0 <= t_one ** 2 / df / 2.0 ** -53 <= 6.0
    assert t_zero == pytest.approx(math.sqrt(df * (1e10 - 1.0)), rel=1e-9)
