"""The OLS / Pearson scan on every kernel instantiation and launch plan it can pick (tests/scan_plan.py lists the cases
and tests/test_scan_plan.py checks, without a GPU, that they reach every (A, K, W, P, kind) scan_kernel, every planner
branch, multi-pass reductions and the phenotype-pass rules).

- test_instantiation: each of the 204 scan_kernel instantiations against the oracle, on inputs that take every
  decision path of the scan (see make_inputs).
- test_planner_shapes: larger shapes on each planner branch, on unequal phenotype passes and the 96 KB cap.
- test_position_independence: a locus gets the same record bits wherever it lands (device against device).
- test_every_fixup_kernel_gets_work: every fixup_kernel<A, K, W> receives deferred loci from these inputs.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import poolgen_b200 as pb
from tests import helpers as H
from tests import scan_plan as SP

pytestmark = pytest.mark.gpu

MAF = 0.02
# the share of loci the oracle keeps and solves is 0.76 to 0.95 over these cases (A = 2 loses the loci with stray reads
# and the threshold loci that land under it)
MIN_OK = 0.7


def _pool_sizes(n, W):
    ps = (10.0 + (np.arange(n) % 7)) if W else np.ones(n)
    tot = 0.0
    for v in ps:  # phen.rs:82-84: normalised by their sequential sum
        tot = tot + v
    return np.array([v / tot for v in ps])


def make_inputs(c, seed, L=None):
    """counts [L, len(codes), n], phenotypes [n, k] and FilterStats of a case.  Besides the generator's loci (about 5 %
    monomorphic, 2 % with a pool without coverage) the slab holds, by locus index l:
      l % 20 == 3   stray reads on an allele the MAF filter removes (the ingest hint renormalises them in the scan)
      l % 20 == 7   a minor allele whose pooled frequency sits on the MAF threshold (exact re-evaluation, deferral)
      l % 20 == 11  one or two pools without coverage (NaN frequencies under --min-coverage-depth 0)
      l % 20 == 15  monomorphic
      l % 20 == 18  reads on the N column when it is dropped, on D otherwise
    Pearson cases with an odd A + K get a NaN phenotype value (pairs dropped per phenotype)."""
    L = c.L if L is None else L
    n, A_in = c.n, len(c.codes)
    rng = np.random.default_rng(seed)
    counts = pb.synth_counts_host(seed, 0, L, n, A_in)
    if A_in > 4:                             # the generator leaves columns 4 and 5 empty
        extra = rng.random((L, A_in - 4, n)) < 0.3
        counts[:, 4:] = extra * rng.integers(1, 20, (L, A_in - 4, n))
    dev_cols = [j for j, code in enumerate(c.codes) if not (c.remove_ns and code == 4)]
    last = dev_cols[-1]
    l = np.arange(L)
    # stray reads: the last device column carries one read in a few pools
    s = l[l % 20 == 3]
    counts[s, last] = (rng.random((s.size, n)) < 0.15).astype(np.uint32)
    counts[s, last, 0] = 1                   # at least one read
    # threshold: depth 100 in every pool, the last device column at 1, 2 or 3 reads with a weighted mean of exactly 2
    # (pools i and i + 7 have the same size and get 2 - s and 2 + s), so the pooled frequency is 0.02 up to rounding,
    # on either side of it depending on the locus
    t = l[l % 20 == 7]
    counts[t] = 0
    minor = np.full((t.size, n), 2)
    for b in range(0, n - 13, 14):
        sh = rng.integers(-1, 2, (t.size, 7))
        minor[:, b:b + 7] -= sh
        minor[:, b + 7:b + 14] += sh
    major = rng.integers(10, 60, (t.size, n))
    counts[t, last] = minor
    if last == dev_cols[1]:                  # two device columns: the minor allele itself sits on the threshold
        counts[t, dev_cols[0]] = 100 - minor
    else:
        counts[t, dev_cols[0]] = 100 - minor - major
        counts[t, dev_cols[1]] = major
    # pools without coverage
    z = l[l % 20 == 11]
    counts[z, :, (z * 7) % n] = 0
    two = z[z % 40 == 11]
    counts[two, :, (two * 3 + 1) % n] = 0
    # monomorphic
    m = l[l % 20 == 15]
    counts[m] = 0
    counts[m, dev_cols[0]] = rng.integers(5, 80, (m.size, n))
    # reads on N (dropped) or D
    d = l[l % 20 == 18]
    col = c.codes.index(4) if 4 in c.codes else (c.codes.index(5) if 5 in c.codes else None)
    if col is not None:
        counts[d, col] += rng.integers(0, 30, (d.size, n)).astype(np.uint32)
    phen = pb.synth_phen_host(seed, n, c.k)
    if c.kind == SP.KIND_CORR and (c.A + c.k) % 2 == 1:
        phen[(seed % n), c.k - 1] = np.nan
    fs = pb.FilterStats(pool_sizes=_pool_sizes(n, c.W), remove_ns=c.remove_ns, min_coverage_depth=0,
                        min_allele_frequency=MAF, max_missingness_rate=0.2)
    return np.ascontiguousarray(counts), phen, fs


def _seed(c):
    return 0x5CA9 + 1009 * c.n + 101 * c.A + 11 * c.k + 3 * c.W + c.kind


def _run(ctx, c, counts, phen, fs):
    scan = pb.Scan(ctx, c.kind, fs, c.n, np.array(c.codes, dtype=np.uint8), phen)
    try:
        return scan.run_counts(counts)
    finally:
        scan.close()


def _compare(ctx, c, min_ok):
    counts, phen, fs = make_inputs(c, _seed(c))
    dev = _run(ctx, c, counts, phen, fs)
    codes = np.array(c.codes, dtype=np.uint8)
    st = H.compare_regression(c.kind, counts, codes, phen, fs, dev, label=c.id)
    assert st["ok"] >= min_ok * c.L, (c.id, st)
    print(c.id, st)


@pytest.mark.parametrize("c", SP.MATRIX, ids=[c.id for c in SP.MATRIX])
def test_instantiation(ctx, c):
    _compare(ctx, c, MIN_OK)


@pytest.mark.parametrize("c", SP.PLANNER, ids=[c.id for c in SP.PLANNER])
def test_planner_shapes(ctx, c):
    """branches of the G / nbuf / warps fit, multi-pass reductions, the 96 KB phenotype cap and passes of unequal K"""
    _compare(ctx, c, MIN_OK)


@pytest.mark.parametrize("n", [3, 6, 7, 12, 31, 100, 300])
@pytest.mark.parametrize("nan_phen", [False, True])
def test_correlation_of_a_constant_column(ctx, n, nan_phen):
    """pearson_corr on loci whose allele frequencies are the same in every pool (or in every pool with coverage).  The
    reference's mean is a sequential sum of n copies over n: where it is not exactly the value, the centred column is
    that rounding residue and r rounds to 0 with p = 1; where it is, r = 0 / 0 = NaN.  Found by test_instantiation
    (A = 2, 7 pools, a NaN phenotype): the fix-up kernel's pairwise and two-pass paths took the mean from a warp's tree
    sum, which can land on the value where the sequential sum does not, and wrote NaN where the reference writes 0."""
    rng = np.random.default_rng(n)
    L = 240
    minor = rng.integers(1, 40, L)
    depth = minor + rng.integers(1, 60, L)
    counts = np.zeros((L, 2, n), dtype=np.uint32)
    counts[:, 0] = (depth - minor)[:, None]
    counts[:, 1] = minor[:, None]
    counts[1::3, :, n // 2] = 0                     # a pool without coverage: NaN frequencies, dropped pairwise
    phen = pb.synth_phen_host(n, n, 2)
    if nan_phen:
        phen[n - 1, 1] = np.nan
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_coverage_depth=0, min_allele_frequency=0.0,
                        max_missingness_rate=0.5)
    codes = np.array([0, 1], dtype=np.uint8)
    scan = pb.Scan(ctx, pb.KIND_CORR, fs, n, codes, phen)
    dev = scan.run_counts(counts)
    scan.close()
    st = H.compare_regression(pb.KIND_CORR, counts, codes, phen, fs, dev, label=f"constant column n={n}")
    assert st["ok"] == L, st
    print(st)


# ---- position independence -------------------------------------------------------------------------------------
def _assert_same(got, want, what):
    """records bit for bit (any NaN equals any NaN)"""
    assert (got.status == want.status).all(), f"{what}: status differs at {np.nonzero(got.status != want.status)[0][:8]}"
    assert (got.n_out == want.n_out).all(), f"{what}: n_out differs"
    assert (got.alleles == want.alleles).all(), f"{what}: alleles differ"
    for name in ("freq_mean", "stats"):
        a, b = getattr(got, name), getattr(want, name)
        same = (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))
        bad = np.nonzero(~same.reshape(same.shape[0], -1).all(axis=1))[0]
        assert bad.size == 0, f"{what}: {name} differs at loci {bad[:8]}"


def _take(r, idx):
    return pb.ScanResults(r.status[idx], r.n_out[idx], r.alleles[idx], r.freq_mean[idx], r.stats[idx])


@pytest.mark.parametrize("c", SP.POSITION, ids=[c.id for c in SP.POSITION])
def test_position_independence(ctx, c):
    """the records of a slab's loci are the same bits alone, rotated, behind other loci, streamed in odd-sized slabs,
    repeated through batches the plan says fill one grid round and more than two (each ending in a partial block),
    and one locus at a time"""
    seed = _seed(c)
    counts, phen, fs = make_inputs(c, seed)
    other, _, _ = make_inputs(c, seed + 1, L=33)
    L = c.L
    scan = pb.Scan(ctx, c.kind, fs, c.n, np.array(c.codes, dtype=np.uint8), phen)
    try:
        base = scan.run_counts(counts)
        assert (base.status == pb.LOCUS_OK).sum() > L // 2
        r = scan.run_counts(np.ascontiguousarray(np.roll(counts, 7, axis=0)))
        _assert_same(r, _take(base, (np.arange(L) - 7) % L), "rotated by 7")
        for p in (1, 5, 33):
            r = scan.run_counts(np.concatenate([other[:p], counts]))
            _assert_same(_take(r, np.arange(p, p + L)), base, f"behind {p} loci")
        one, many = SP.grid_lengths(c, ctx.info()["sm_count"])
        for Lg in (one, many):
            idx = (np.arange(Lg) + 3) % L
            r = scan.run_counts(counts[idx])
            _assert_same(r, _take(base, idx), f"inside {Lg} loci")
        for l in (0, 3, 7, 11, 15):
            _assert_same(scan.run_counts(counts[l:l + 1]), _take(base, [l]), f"locus {l} alone")
        sizes = [1, 7, 33, 97, 161]
        sizes.append(L - sum(sizes))
        scan.stream_begin(max(sizes))
        pend, parts, l0 = [], [], 0
        for sz in sizes:
            slab = np.ascontiguousarray(counts[l0:l0 + sz])
            pend.append((scan.submit_counts(slab), slab))
            l0 += sz
            if len(pend) == 3:
                parts.append(scan.collect(pend.pop(0)[0]))
        for t, _ in pend:
            parts.append(scan.collect(t))
        cat = pb.ScanResults(*(np.concatenate([getattr(p, f) for p in parts])
                               for f in ("status", "n_out", "alleles", "freq_mean", "stats")))
        _assert_same(cat, base, "streamed in odd-sized slabs")
    finally:
        scan.close()


# ---- every fix-up instantiation gets work ----------------------------------------------------------------------
_DEFER = re.compile(r"\[pg\] deferred (\d+) of (\d+) loci \(last phenotype pass\): threshold (\d+), "
                    r"removed-with-reads (\d+), no coverage (\d+), NaN under hint (\d+), redo ols (\d+), "
                    r"redo corr (\d+), corr NaN (\d+), tie (\d+)")
REASONS = ("threshold", "removed-with-reads", "no coverage", "NaN under hint", "redo ols", "redo corr", "corr NaN", "tie")


def defer_report(which):
    """run in a subprocess with PG_REPORT_DEFER=1 (read once per process): one timed run per matrix case, a marker line
    before each so that the library's report can be attributed; also checks the launches of the run against the plan"""
    ctx = pb.Context(0)
    cases = [c for c in SP.MATRIX if which == "all" or SP.lanes(c.n, c.A) == int(which)]
    for c in cases:
        counts, phen, fs = make_inputs(c, _seed(c))
        scan = pb.Scan(ctx, c.kind, fs, c.n, np.array(c.codes, dtype=np.uint8), phen)
        b = scan.batch(c.L)
        b.upload_counts(counts)
        print(f"@case {c.A} {c.k} {int(c.W)} {SP.lanes(c.n, c.A)} {c.kind}", file=sys.stderr, flush=True)
        _, launches = b.time_runs(1)
        sys.stderr.flush()
        assert launches == 2 * len(SP.plan(c.n, c.A, c.k, c.W)), (c.id, launches)
        b.close()
        scan.close()
    ctx.close()


def _defer_counts(env_extra, which):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PG_REPORT_DEFER="1", **env_extra)
    out = subprocess.run([sys.executable, "-c", f"from tests import test_scan_matrix_gpu as M; M.defer_report({which!r})"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=root, env=env, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:]
    per_case, case = {}, None
    for line in out.stdout.splitlines():
        if line.startswith("@case "):
            case = tuple(int(v) for v in line.split()[1:])
            continue
        m = _DEFER.search(line)
        if m:
            assert case is not None and case not in per_case, line
            per_case[case] = [int(v) for v in m.groups()]
            case = None
    return per_case


def test_every_fixup_kernel_gets_work():
    """every fixup_kernel<A, K, W> receives loci from these inputs, at every lane count and both kinds.  With the
    ingest hints (the default) loci whose removed alleles carry reads are renormalised in the streaming kernel; with
    PG_NOHINT=1 they take the fix-up kernel's own renormalising path, the "removed-with-reads" reason"""
    if os.environ.get("PG_REPORT_DEFER") or os.environ.get("PG_NOHINT"):
        pytest.skip("inside a diagnostic run")
    want = {(c.A, c.k, int(c.W), SP.lanes(c.n, c.A), c.kind) for c in SP.MATRIX}
    totals = {}
    for env_extra, which in (({}, "all"), ({"PG_NOHINT": "1"}, "16")):
        per_case = _defer_counts(env_extra, which)
        expect = want if which == "all" else {w for w in want if w[3] == int(which)}
        assert set(per_case) == expect, sorted(expect - set(per_case))
        empty = sorted(k for k, v in per_case.items() if v[0] == 0)
        assert not empty, f"no deferred loci at (A, K, W, P, kind) {empty}"
        fix = {(A, K, W) for A, K, W, _, _ in per_case}
        assert len(fix) == 34
        tot = np.array(list(per_case.values())).sum(axis=0)
        totals["hints" if not env_extra else "no hints"] = tot
        print(f"{'PG_NOHINT=1' if env_extra else 'default'}: {len(per_case)} runs, deferred {tot[0]} of {tot[1]} loci: " +
              ", ".join(f"{name} {v}" for name, v in zip(REASONS, tot[2:])))
    assert totals["hints"][2] > 0 and totals["hints"][4] > 0           # threshold, no coverage
    assert totals["no hints"][3] > 0                                   # removed-with-reads
