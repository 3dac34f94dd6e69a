"""The cases of tests/test_scan_matrix_gpu.py against the Python restatement of the scan's launch plan
(tests/scan_plan.py): together they must reach every scan_kernel instantiation, every planner branch at each lane
count where it exists, a multi-pass reduction for every allele count, a phenotype pass cut by the 96 KB rule, passes
of unequal K, and for A <= 3 a last row chunk of 4 rows and a middle chunk.  Runs without a GPU."""
import collections

from tests import scan_plan as SP

BRANCHES = {8: {"32x3", "32x2", "few"}, 16: {"32x3", "32x2", "few"}, 32: {"32x3", "32x2", "16x2", "few"}}


def _launches(cases):
    for c in cases:
        for lp in SP.plan(c.n, c.A, c.k, c.W):
            yield c, lp


def test_layout_and_passes_restate_the_host_rules():
    assert SP.make_layout(1, 2) == (4, 4, 1, 4)
    assert SP.make_layout(256, 2) == (256, 256, 1, 256)
    assert SP.make_layout(257, 2) == (260, 256, 2, 4)
    assert SP.make_layout(385, 3) == (388, 192, 3, 4)
    assert SP.make_layout(1000, 4) == (1000, 128, 8, 104)
    assert [SP.lanes(n, 4) for n in (2, 64, 65, 128, 129)] == [8, 8, 16, 16, 32]
    assert SP.phen_passes(300, 5, 5, False) == ([3, 2], False)
    assert SP.phen_passes(4000, 4, 3, True) == ([2, 1], True)     # 96 KB / 32,000 B = 3 vectors, one is the weights
    assert SP.phen_passes(4000, 4, 3, False) == ([3], True)
    assert SP.phen_passes(13000, 2, 1, True) == ([1], True)        # never below one phenotype per pass
    # the tiny stage of test_tiny_stage: two alleles over four pools is a 256-byte stage, raised to one reduction row
    lp = SP.launch_plan(4, 2, 1, False)
    assert (lp.P, lp.red_rows, lp.multi_pass) == (8, 1, True)
    # the full-size C2 shape: 100 pools, 16 lanes; three 6,400-byte stages leave room for 9 warps, two for 12
    lp = SP.launch_plan(100, 4, 1, False, L=1_000_000)
    assert (lp.P, lp.branch, lp.warps, lp.multi_pass) == (16, "32x2", 12, False)
    assert lp.rounds == 18 and lp.block == 32 and lp.ctas == SP.B200_SMS


def test_case_inputs_are_consistent():
    for c in SP.MATRIX + SP.PLANNER + SP.POSITION:
        assert SP.device_columns(c.codes, c.remove_ns) == c.A, c
        assert all(a < b for a, b in zip(c.codes, c.codes[1:]))   # sync column order
    for c in SP.MATRIX:
        assert 600 <= c.L <= 1500
        P = SP.lanes(c.n, c.A)
        cr = SP.chunk_rows(c.A)
        if P == 8:
            assert c.n % 2 == 1 and c.n <= 64
        elif P == 16:
            assert 64 < c.n <= cr
        else:
            assert c.n in (cr + 1, 2 * cr + 1)
    assert any(c.codes == (2, 4, 5) for c in SP.MATRIX)   # two device columns from three with N dropped
    # the top edge of the one-chunk layout at 16 lanes, for every A
    for A in SP.MAX_K:
        assert any(c.A == A and c.n == SP.chunk_rows(A) for c in SP.MATRIX)


def test_matrix_reaches_every_instantiation():
    want = {(A, K, W, P, kind) for A in SP.MAX_K for K in range(1, SP.MAX_K[A] + 1) for W in (False, True)
            for P in (8, 16, 32) for kind in (SP.KIND_OLS, SP.KIND_CORR)}
    assert len(want) == 204
    got = {(c.A, lp.K, c.W, lp.P, c.kind) for c, lp in _launches(SP.MATRIX)}
    assert got == want, sorted(want - got)
    fix = {(A, K, W) for A, K, W, _, _ in got}
    print(f"\nscan_kernel instantiations reached: {len(got)} of {len(want)}; fixup_kernel: {len(fix)} of 34")
    assert len(fix) == 34


def test_cases_reach_every_planner_branch():
    table = collections.defaultdict(set)
    multi = set()
    cut, unequal = [], []
    for c, lp in _launches(SP.MATRIX + SP.PLANNER):
        table[lp.P].add(lp.branch)
        if lp.multi_pass:
            multi.add(c.A)
    for c in SP.MATRIX + SP.PLANNER:
        passes, was_cut = SP.phen_passes(c.n, c.A, c.k, c.W)
        if was_cut and c.k > passes[0]:
            cut.append(c.id)
        if len(set(passes)) > 1:
            unequal.append(c.id)
    print()
    print("lanes  branches reached")
    for P in (8, 16, 32):
        print(f"{P:5d}  {', '.join(sorted(table[P]))}  (of {', '.join(sorted(BRANCHES[P]))})")
    print(f"multi-pass reduction at A = {sorted(multi)}")
    print(f"K cut by the 96 KB rule: {cut}")
    print(f"phenotype passes of unequal K: {unequal}")
    for P in (8, 16, 32):
        assert table[P] == BRANCHES[P], (P, table[P])
    assert multi == {2, 3, 4, 5, 6}
    assert cut and unequal


def test_last_chunk_of_four_rows_and_a_middle_chunk():
    for A in (2, 3):
        lays = [SP.make_layout(c.n, A) for c in SP.MATRIX if c.A == A and SP.lanes(c.n, A) == 32]
        assert any(rc_last == 4 for _, _, _, rc_last in lays), A
        assert any(n_chunks >= 3 for _, _, n_chunks, _ in lays), A


def test_position_cases_cover_every_grid():
    """each position case is run inside batches the plan says end in a partial block, take exactly one grid round and
    more than two rounds"""
    seen = set()
    for c in SP.POSITION:
        seen.add((c.A, SP.lanes(c.n, c.A), c.W))
        assert c.k == SP.MAX_K[c.A]
        one, many = SP.grid_lengths(c)
        lo = SP.launch_plan(c.n, c.A, c.k, c.W, L=one)
        hi = SP.launch_plan(c.n, c.A, c.k, c.W, L=many)
        assert lo.rounds == 1 and lo.partial, (c.id, lo)
        assert hi.rounds > 2 and hi.partial, (c.id, hi)
    assert len(seen) == 30
