"""The OLS / Pearson / mle_iter scans past 6,144 pools: scan_kernel_wide reads the phenotype rows and pool weights from
L2 where scan_kernel holds them in shared memory (pg_scan.cuh, pg::scan_wide in pg_internal.h).

- test_wide_kernel_records_equal_resident: PG_SCAN_WIDE=1 (read once per process, so in a subprocess) puts every
  32-lane scan on the wide kernel; its records equal the resident kernel's bit for bit on all 68 (A, K, W, kind)
  instantiations, deferred loci included.
- test_oracle_past_the_old_limit: OLS and Pearson at 6,145 to 20,000 pools against the oracle.
- test_position_independence_8192: a locus's records alone, rotated and inside a batch of three grid rounds.
- test_mle_iter_past_the_old_limit, test_p_over_the_whole_range_of_t, test_file_level_8192_pools.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import poolgen_b200 as pb
from oracle import pgo
from tests import helpers as H
from tests import scan_plan as SP
from tests import test_scan_matrix_gpu as M
from tests import test_student_t_tails_gpu as T

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _wide_passes(A, k):
    kp = SP.MAX_K[A]
    return [min(kp, k - b) for b in range(0, k, kp)]


def make_inputs(c, seed, L=None):
    """the scan matrix's inputs (threshold loci, stray reads, pools without coverage, monomorphic loci, a NaN
    phenotype for Pearson at odd A + k) plus, at l % 20 == 5, two allele columns with the same counts in every pool
    (a rank-deficient design) where there are three device columns or more"""
    counts, phen, fs = M.make_inputs(c, seed, L)
    dev_cols = [j for j, code in enumerate(c.codes) if not (c.remove_ns and code == 4)]
    if len(dev_cols) >= 3:
        r = np.arange(counts.shape[0])
        r = r[r % 20 == 5]
        counts[r, dev_cols[-1]] = counts[r, dev_cols[1]]
    return counts, phen, fs


# ---- bit identity with the resident kernel ----------------------------------------------------------------------
# the matrix's 32-lane cases reach all 34 (A, K, W) x 2 kinds; the larger shapes are ones where the resident plan's
# phenotype passes equal the wide plan's (the wide kernel takes no 96 KB cut), so the two run the same launches
IDENTITY = [c for c in SP.MATRIX if SP.lanes(c.n, c.A) == 32] + [
    SP.Case(2000, 5, 5, True, SP.KIND_CORR, (0, 1, 2, 3, 4, 5), True, 300),
    SP.Case(4000, 4, 3, False, SP.KIND_CORR, (0, 1, 2, 3), True, 200),
    SP.Case(6144, 2, 2, False, SP.KIND_OLS, (1, 3), True, 200),
    SP.Case(6144, 3, 1, True, SP.KIND_OLS, (0, 2, 5), True, 200),
]


def _seed(c):
    return 0x71DE + 1009 * c.n + 101 * c.A + 11 * c.k + 3 * c.W + c.kind


def _records(out_path):
    """every IDENTITY case's records, with the library's deferral report before each (run with PG_REPORT_DEFER)"""
    ctx = pb.Context(0)
    arrays = {}
    for i, c in enumerate(IDENTITY):
        counts, phen, fs = make_inputs(c, _seed(c))
        scan = pb.Scan(ctx, c.kind, fs, c.n, np.array(c.codes, dtype=np.uint8), phen)
        b = scan.batch(c.L)
        b.upload_counts(counts)
        print(f"@case {i}", file=sys.stderr, flush=True)
        b.time_runs(1)
        sys.stderr.flush()
        r = b.fetch()
        for f in ("status", "n_out", "alleles", "freq_mean", "stats"):
            arrays[f"{i}_{f}"] = getattr(r, f)
        b.close()
        scan.close()
    ctx.close()
    np.savez(out_path, **arrays)


def _run_records(tmp_path, env_extra):
    out = tmp_path / ("wide.npz" if env_extra else "resident.npz")
    env = dict(os.environ, PG_REPORT_DEFER="1")
    env.pop("PG_SCAN_WIDE", None)
    env.update(env_extra)
    res = subprocess.run([sys.executable, "-c", f"from tests import test_wide_pools_gpu as W; W._records({str(out)!r})"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=ROOT, env=env, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    deferred, case = {}, None
    for line in res.stdout.splitlines():
        if line.startswith("@case "):
            case = int(line.split()[1])
        m = M._DEFER.search(line)
        if m and case is not None:
            deferred[case] = int(m.group(1))
    return np.load(out), deferred


def test_wide_kernel_records_equal_resident(tmp_path):
    if os.environ.get("PG_SCAN_WIDE"):
        pytest.skip("inside a PG_SCAN_WIDE run")
    assert all(SP.lanes(c.n, c.A) == 32 for c in IDENTITY)
    assert {(c.A, K, c.W, c.kind) for c in IDENTITY for K in _wide_passes(c.A, c.k)} == \
        {(A, K, W, kind) for A in range(2, 7) for K in range(1, SP.MAX_K[A] + 1) for W in (False, True)
         for kind in (SP.KIND_OLS, SP.KIND_CORR)}
    for c in IDENTITY:
        assert SP.phen_passes(c.n, c.A, c.k, c.W)[0] == _wide_passes(c.A, c.k), c.id
    res, _ = _run_records(tmp_path, {})
    wide, deferred = _run_records(tmp_path, {"PG_SCAN_WIDE": "1"})
    assert len(deferred) == len(IDENTITY)
    assert not [IDENTITY[i].id for i, v in deferred.items() if v == 0], "cases without deferred loci"
    for i, c in enumerate(IDENTITY):
        got = pb.ScanResults(*(wide[f"{i}_{f}"] for f in ("status", "n_out", "alleles", "freq_mean", "stats")))
        want = pb.ScanResults(*(res[f"{i}_{f}"] for f in ("status", "n_out", "alleles", "freq_mean", "stats")))
        assert (got.status == pb.LOCUS_OK).sum() > c.L // 2, c.id
        M._assert_same(got, want, c.id)


# ---- past the old limit, against the oracle ---------------------------------------------------------------------
def _case(n, A, k, W, kind, L=160):
    codes, rn = SP._codes(A, (n + A) % 2 == 1)
    return SP.Case(n, A, k, W, kind, codes, rn, L)


ORACLE = [
    _case(6145, 2, 1, False, SP.KIND_OLS), _case(6145, 3, 2, True, SP.KIND_CORR),
    _case(8192, 4, 4, True, SP.KIND_OLS), _case(8192, 5, 5, False, SP.KIND_CORR),
    _case(12289, 6, 3, True, SP.KIND_OLS), _case(12289, 2, 5, False, SP.KIND_CORR),
    _case(20000, 3, 3, False, SP.KIND_OLS), _case(20000, 6, 5, True, SP.KIND_CORR),
]


@pytest.mark.parametrize("c", ORACLE, ids=[c.id for c in ORACLE])
def test_oracle_past_the_old_limit(ctx, c):
    counts, phen, fs = make_inputs(c, _seed(c))
    dev = M._run(ctx, c, counts, phen, fs)
    st = H.compare_regression(c.kind, counts, np.array(c.codes, dtype=np.uint8), phen, fs, dev, label=c.id)
    assert st["ok"] >= M.MIN_OK * c.L, (c.id, st)
    print(c.id, st)


# ---- position independence at 8,192 pools ----------------------------------------------------------------------
def _wide_rounds(n, A, K, W, L, sm_count):
    """grid rounds of a wide-kernel launch: the fit of launch_scan_p without the phenotypes' shared memory"""
    n_pad, rc, _, _ = SP.make_layout(n, A)
    N = SP.acc_n(A, K, W)
    stage = SP._up128(A * rc * 8)

    def fit(g, nb):
        return min(SP.SCAN_WARPS, SP.SMEM_AVAIL // (64 + nb * stage + SP._up128(g * (N | 1) * 8)))
    G, nbuf = next(((g, nb) for g, nb in ((32, 3), (32, 2), (16, 2)) if fit(g, nb) >= SP.SCAN_WARPS), (32, 2))
    warps = fit(G, nbuf)
    gw = sm_count * warps
    r = (L + gw * G - 1) // (gw * G)
    g = min(G, (L + gw * r - 1) // (gw * r))
    nb = (L + g - 1) // g
    ctas = max(1, min(sm_count, (nb + warps - 1) // warps))
    return (nb + ctas * warps - 1) // (ctas * warps), gw * G


def test_position_independence_8192(ctx):
    c = _case(8192, 2, 1, False, SP.KIND_OLS, L=300)
    counts, phen, fs = make_inputs(c, _seed(c))
    dt = np.uint8 if counts.max() < 256 else np.uint16
    counts = counts.astype(dt)
    scan = pb.Scan(ctx, c.kind, fs, c.n, np.array(c.codes, dtype=np.uint8), phen)
    try:
        base = scan.run_counts(counts)
        assert (base.status == pb.LOCUS_OK).sum() > c.L // 2
        r = scan.run_counts(np.ascontiguousarray(np.roll(counts, 7, axis=0)))
        M._assert_same(r, M._take(base, (np.arange(c.L) - 7) % c.L), "rotated by 7")
        for l in (0, 5, 7, 11, 15):
            M._assert_same(scan.run_counts(counts[l:l + 1]), M._take(base, [l]), f"locus {l} alone")
        sm = ctx.info()["sm_count"]
        _, per_round = _wide_rounds(c.n, c.A, c.k, c.W, 1, sm)
        Lg = 2 * per_round + 37
        rounds, _ = _wide_rounds(c.n, c.A, c.k, c.W, Lg, sm)
        assert rounds >= 3, rounds
        idx = (np.arange(Lg) + 3) % c.L
        big = counts[idx]
        r = scan.run_counts(big)
        del big
        M._assert_same(r, M._take(base, idx), f"inside {Lg} loci ({rounds} grid rounds)")
    finally:
        scan.close()


# ---- mle_iter ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,A,k,L", [(6145, 4, 2, 40), (8192, 3, 1, 40)])
def test_mle_iter_past_the_old_limit(ctx, n, A, k, L):
    """the bar of tests/test_nm_gpu.py::test_mle_iter_synthetic"""
    from tests.test_nm_edges_gpu import check_mle_status
    counts = pb.synth_counts_host(0x31E + n, 0, L, n, min(A, 4))
    full = np.zeros((L, A, n), dtype=np.uint32)
    full[:, :min(A, 4)] = counts
    phen = pb.synth_phen_host(0x31E + n, n, k)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    codes = np.arange(A, dtype=np.uint8)
    dev = pb.mle_iterate(ctx, full, phen, fs, codes)
    orc = pgo.scan_batch(pgo.SCAN_MLE, full, codes, phen, H.oracle_fs(fs), 8)
    both, why = check_mle_status(full, codes, fs, dev, orc, f"mle_iter n={n} k={k}")
    assert both.sum() > 0.5 * L, why
    assert (orc.n_out[both] == dev.n_out[both]).all() and (orc.allele[both] == dev.alleles[both]).all()
    S = dev.stats.shape[1]
    slot = np.broadcast_to((np.arange(S)[None, :] < orc.n_out[both][:, None])[:, :, None], (both.sum(), S, k))
    b_o, b_d = orc.stat[both][:, :S][slot], dev.stats[both][..., 0][slot]
    v_o, v_d = orc.var[both][:, :S][slot], dev.stats[both][..., 1][slot]
    p_o, p_d = orc.pval[both][:, :S][slot], dev.stats[both][..., 3][slot]
    se = np.sqrt(np.abs(v_o) * n / (2.0 * np.maximum(n - (orc.n_out[both].astype(float)[:, None, None] + 1.0), 1.0) * np.ones((1, S, k)))[slot])
    eb = np.abs(b_d - b_o) / np.maximum(np.abs(b_o), se)
    ev = np.abs(v_d - v_o) / np.abs(v_o)
    ep = np.abs(p_d - p_o) / np.maximum(p_o, 1e-12)
    print(f"mle_iter n={n} k={k}: {slot.sum()} coefficients, beta err median {np.median(eb):.2e} max {eb.max():.2e}; "
          f"v_b err median {np.median(ev):.2e} max {ev.max():.2e}; p err median {np.median(ep):.2e} max {ep.max():.2e}")
    assert np.median(eb) < 5e-6 and eb.max() < 1e-3
    assert np.median(ev) < 1e-6 and ev.max() < 1e-3
    assert np.median(ep) < 5e-6 and ep.max() < 1e-3


# ---- p-values at df = n - 1 and n - 2 ----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [pb.KIND_OLS, pb.KIND_CORR])
@pytest.mark.parametrize("n", [6145, 16384, 65536])
def test_p_over_the_whole_range_of_t(ctx, n, kind):
    """near-collinear loci (t up to where p is 0) and loci whose t straddles statrs' t_one, held to the reference's p
    of the recorded t (tests/test_student_t_tails_gpu.py); whichever form build_ptable leaves at this df"""
    rng = np.random.default_rng(9700 + n + kind)
    y, base = T._many_pool_loci(n, rng)
    x1 = np.ones((n, 2))
    x1[:, 1] = base[1].astype(np.float64) / (2 * T.D)
    x1[0, 1] = (float(base[1, 0]) + 1000.0) / (2 * T.D)
    _, _, _, _, t1000 = pgo.ols(x1, y)
    per_read = abs(float(t1000[1, 0])) / 1000.0
    t_one, _ = H.student_t_cutoffs(n - 1)
    targets = np.concatenate([10.0 ** np.linspace(-8, -4, 60), t_one * np.array([0.9, 0.99, 1.01, 1.1])])
    moves = np.unique(np.rint(targets / per_read).astype(np.int64))
    near = np.repeat(base[None], moves.size + 1, axis=0)
    near[1:, 1, 0] += moves.astype(np.uint32)
    near[1:, 0, 0] -= moves.astype(np.uint32)
    far = T._counts_from_minor(T._few_pool_loci(n, y, rng), rare_reads=True)
    counts = np.concatenate([near, far])
    res = T._scan_records(ctx, kind, counts, y[:, None], n, False)
    reg, df = T._scan_check(res, kind, n, f"kind={kind} n={n}")
    assert reg["tail"] > 0 and reg["zero"] + reg["quantised_zero"] > 0, reg
    if kind == pb.KIND_OLS:
        assert reg["one"] > 0 and reg["just_above_one"] > 0, f"n={n}: t did not straddle t_one: {reg}"


# ---- file level ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("analysis", ["ols_iter", "pearson_corr", "mle_iter"])
def test_file_level_8192_pools(ctx, tmp_path, analysis):
    """FileSyncPhen.read_analyse_write on an 8,192-pool sync file, three reader threads over blocks that end inside
    lines: the file equals the header and the rows of the same records computed in one batch"""
    from tests.test_text_gpu import _sync_text
    n, L = 8192, 48 if analysis == "mle_iter" else 120
    counts = np.zeros((L, 6, n), dtype=np.uint32)
    counts[:, :4] = pb.synth_counts_host(0xF11E, 0, L, n, 4)
    pos = list(range(101, 101 + 7 * L, 7))
    fsync = tmp_path / "wide.sync"
    fsync.write_bytes(_sync_text(counts, ["chr2"] * L, pos))
    phen = pb.synth_phen_host(0xF11E, n, 2)
    sizes = np.full(n, 1.0 / n)
    fs = pb.FilterStats(pool_sizes=sizes, min_coverage_depth=1, min_allele_frequency=0.01)
    fn, kind = {"ols_iter": (pb.ols_iterate, pb.KIND_OLS), "pearson_corr": (pb.correlation, pb.KIND_CORR),
                "mle_iter": (pb.mle_iterate, pb.KIND_MLE)}[analysis]
    src = pb.FileSyncPhen(str(fsync), [f"p{i}" for i in range(n)], sizes, phen, analysis)
    out = src.read_analyse_write(ctx, fs, str(tmp_path / "out.csv"), 3, fn, block_bytes=1 << 20)
    whole = fn(ctx, counts, phen, fs)
    assert (whole.status == pb.LOCUS_OK).sum() > L // 2
    expect = pb.format_header(kind) + pb.format_rows(kind, whole, np.array(pos), chr_names=["chr2"],
                                                     chr_index=np.zeros(L, np.uint32), exact_p_pools=n)
    got = open(out, "rb").read()
    assert got == expect and got.count(b"\n") > L
