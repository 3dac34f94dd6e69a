"""The launch plan of the OLS / Pearson scan, restated in Python, and the cases that put the scan on each of its
kernel instantiations and planner branches.

`plan(n, A, k, W, L)` follows the host code that chooses a launch:
  make_layout, chunk_rows                    poolgen_b200/csrc/pg_internal.h:27-62
  max_phen_per_pass, the 96 KB phenotype cap poolgen_b200/csrc/pg_internal.h:66, pg_api.cu:586-590
  P (lanes per locus)                        poolgen_b200/csrc/pg_scan.cuh:1731-1740
  G / nbuf / warps fit                       poolgen_b200/csrc/pg_scan.cuh:1656-1690
  block size and grid                        poolgen_b200/csrc/pg_scan.cuh:1691-1716
  red_rows (reduction passes)                poolgen_b200/csrc/pg_scan.cuh:1462
No tuning knob (PG_NBUF, PG_G, PG_WARPS, PG_P) is modelled: the cases reach every branch with real shapes.

The case lists (MATRIX, PLANNER, POSITION) are shared by tests/test_scan_plan.py, which checks without a GPU
that they cover every instantiation and branch, and tests/test_scan_matrix_gpu.py, which runs them.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

KIND_OLS, KIND_CORR = 0, 1          # PG_KIND_OLS / PG_KIND_CORR (include/poolgen_cuda.h)
B200_SMS = 148
SCAN_WARPS = 12                      # kScanWarps
RED_PITCH = 33                       # kRedPitch
SMEM_AVAIL = 227 * 1024 - 512        # dynamic shared memory of a scan CTA
PHEN_SMEM = 96 * 1024                # resident phenotype vectors of one pass
MAX_K = {2: 4, 3: 4, 4: 4, 5: 3, 6: 2}  # max_phen_per_pass(A)


def chunk_rows(A):
    return 256 if A <= 2 else (192 if A == 3 else 128)


def make_layout(n, A):
    """(n_pad, rc, n_chunks, rc_last)"""
    n_pad = (n + 3) & ~3
    cr = chunk_rows(A)
    if n_pad <= cr:
        return n_pad, n_pad, 1, n_pad
    n_chunks = (n_pad + cr - 1) // cr
    return n_pad, cr, n_chunks, n_pad - (n_chunks - 1) * cr


def acc_n(A, K, W):
    """accumulators per lane: column sums, products, cross products, weighted column sums (Acc<A, K, W>::N)"""
    return A + A * (A + 1) // 2 + A * K + (A if W else 0)


def phen_passes(n, A, k, W):
    """K of each phenotype pass (run_once in pg_api.cu)"""
    n_pad = make_layout(n, A)[0]
    kpass = MAX_K[A]
    fit = PHEN_SMEM // (n_pad * 8) - (1 if W else 0)
    if kpass > fit:
        kpass = max(fit, 1)
    return [min(kpass, k - b) for b in range(0, k, kpass)], kpass < MAX_K[A]


def lanes(n, A):
    n_pad, _, n_chunks, _ = make_layout(n, A)
    if n_chunks == 1:
        return 16 if n_pad > 64 else 8
    return 32


def _up128(x):
    return (x + 127) // 128 * 128


@dataclass
class Launch:
    K: int
    P: int
    branch: str        # "32x3", "32x2", "16x2" (P = 32 only) or "few" (fewer than 12 warps)
    G: int             # loci per block before the block-size rule
    nbuf: int
    warps: int
    red_rows: int
    N: int
    multi_pass: bool   # the reduction takes several passes through the scratch (red_rows < N)
    block: int = 0     # loci per block after the block-size rule (L given)
    ctas: int = 0
    rounds: int = 0    # blocks per warp of the grid, rounded up
    partial: bool = False  # the last block holds fewer loci than the others


def launch_plan(n, A, K, W, L=None, sm_count=B200_SMS):
    n_pad, rc, _, _ = make_layout(n, A)
    P = lanes(n, A)
    N = acc_n(A, K, W)
    NP = N | 1
    common = _up128((K + (1 if W else 0)) * n_pad * 8)
    stage = _up128(A * rc * 8 if P == 32 else (32 // P) * A * n_pad * 8)
    if stage < RED_PITCH * 8:
        stage = _up128(RED_PITCH * 8)

    def fit(g, nb):
        wbytes = 64 + nb * stage + _up128(g * NP * 8)
        return min(SCAN_WARPS, (SMEM_AVAIL - common) // wbytes if common + wbytes <= SMEM_AVAIL else 0)

    g_min = 16 if P == 32 else 32
    if fit(32, 3) >= SCAN_WARPS:
        br, G, nbuf = "32x3", 32, 3
    elif fit(32, 2) >= SCAN_WARPS:
        br, G, nbuf = "32x2", 32, 2
    elif fit(g_min, 2) >= SCAN_WARPS:
        br, G, nbuf = f"{g_min}x2", g_min, 2
    else:
        br, G, nbuf = "few", 32, 2
    warps = fit(G, nbuf)
    assert warps >= 1, (n, A, K, W)
    red_rows = max(1, min(stage // (RED_PITCH * 8), N))
    lp = Launch(K, P, br, G, nbuf, warps, red_rows, N, red_rows < N)
    if L:
        gw = sm_count * warps
        step = 1 if P == 32 else 32 // P
        r = (L + gw * G - 1) // (gw * G)
        g = (L + gw * r - 1) // (gw * r)
        g = max(step, (g + step - 1) // step * step)
        lp.block = min(G, g)
        nb = (L + lp.block - 1) // lp.block
        lp.ctas = max(1, min(sm_count, (nb + warps - 1) // warps))
        lp.rounds = (nb + lp.ctas * warps - 1) // (lp.ctas * warps)
        lp.partial = L % lp.block != 0
    return lp


def plan(n, A, k, W, L=None, sm_count=B200_SMS):
    """the launches of one run: one per phenotype pass"""
    passes, _ = phen_passes(n, A, k, W)
    return [launch_plan(n, A, K, W, L, sm_count) for K in passes]


# ---- the cases ---------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    n: int
    A: int          # allele columns on the device
    k: int
    W: bool
    kind: int
    codes: tuple    # allele codes of the input columns
    remove_ns: bool
    L: int

    @property
    def id(self):
        return (f"A{self.A}-k{self.k}-{'W' if self.W else 'u'}-P{lanes(self.n, self.A)}-"
                f"{'ols' if self.kind == KIND_OLS else 'corr'}-n{self.n}")


def device_columns(codes, remove_ns):
    return sum(1 for c in codes if not (remove_ns and c == 4))


def _codes(A, variant):
    """input allele codes and remove_ns giving A device columns; `variant` alternates between a plain set and one
    whose N column (code 4) is dropped on the device"""
    if A == 6:
        return (0, 1, 2, 3, 4, 5), False
    if A == 5:
        return ((0, 1, 2, 3, 4, 5), True) if variant else ((0, 1, 2, 3, 5), True)
    plain = {2: (1, 3), 3: (0, 2, 5), 4: (0, 1, 2, 3)}[A]
    with_n = {2: (2, 4, 5), 3: (0, 1, 4, 5), 4: (0, 1, 2, 4, 5)}[A]
    return (with_n, True) if variant else (plain, True)


def _pools(A, P, i):
    """pool count of the i-th case of a P class: P = 8 odd n <= 64 (padding rows), P = 16 n in (64, chunk_rows],
    the top edge included, P = 32 one row past a chunk (a last chunk of 4 rows) or past two chunks (a middle chunk)"""
    cr = chunk_rows(A)
    if P == 8:
        return (13, 29, 45, 61, 63, 7)[i % 6]
    if P == 16:
        return (cr, 65, 2 * cr // 3 + 1, cr - 3)[i % 4]
    return (cr + 1, 2 * cr + 1)[i % 2]


def _matrix():
    out = []
    seen = {8: 0, 16: 0, 32: 0}     # (A, K, W) triples so far in each P class: pool counts and codes rotate
    for A in (2, 3, 4, 5, 6):
        for K in range(1, MAX_K[A] + 1):
            for W in (False, True):
                for P in (8, 16, 32):
                    j = seen[P]
                    seen[P] += 1
                    n = _pools(A, P, j)
                    codes, rn = _codes(A, (j + A) % 2 == 1)
                    L = 600 if P == 32 and n > 2 * chunk_rows(A) else 1000
                    for kind in (KIND_OLS, KIND_CORR):        # both kinds of a (A, K, W, P) share the input
                        out.append(Case(n, A, K, W, kind, codes, rn, L))
    return out


MATRIX = _matrix()

# larger shapes: every planner branch at each P where it exists, multi-pass reductions, the 96 KB phenotype cap and
# phenotype passes of unequal K
PLANNER = [
    Case(2000, 3, 4, False, KIND_OLS, (0, 1, 2), True, 300),
    Case(2000, 3, 4, True, KIND_CORR, (0, 1, 2), True, 300),
    Case(4000, 4, 3, True, KIND_OLS, (0, 1, 2, 3), True, 200),
    Case(4000, 4, 3, True, KIND_CORR, (0, 1, 2, 3), True, 200),
    Case(300, 5, 5, False, KIND_OLS, (0, 1, 2, 3, 4, 5), True, 400),
    Case(300, 5, 5, True, KIND_CORR, (0, 1, 2, 3, 4, 5), True, 400),
    Case(64, 4, 4, True, KIND_OLS, (0, 1, 2, 3), True, 600),
    Case(2000, 4, 4, True, KIND_OLS, (0, 1, 2, 3), True, 300),
    Case(700, 6, 3, True, KIND_OLS, (0, 1, 2, 3, 4, 5), False, 300),
    Case(1000, 2, 5, True, KIND_CORR, (0, 1), True, 300),
    Case(128, 6, 2, True, KIND_OLS, (0, 1, 2, 3, 4, 5), False, 600),
    Case(60, 6, 2, True, KIND_CORR, (0, 1, 2, 3, 4, 5), False, 600),
]


def _position():
    """every A and P class at the largest K of one pass, both W"""
    out = []
    for A in (2, 3, 4, 5, 6):
        for P in (8, 16, 32):
            for W in (False, True):
                n = {8: 29, 16: 65 if W else chunk_rows(A), 32: chunk_rows(A) + 1}[P]
                codes, rn = _codes(A, W)
                out.append(Case(n, A, MAX_K[A], W, KIND_CORR if W else KIND_OLS, codes, rn, 500))
    return out


POSITION = _position()


def grid_lengths(c, sm_count=B200_SMS):
    """two batch sizes for a case: one whose blocks fill exactly one round of the grid, and one that takes more than
    two rounds; both end in a partial block"""
    def first(L):
        while True:
            lp = launch_plan(c.n, c.A, c.k, c.W, L=L, sm_count=sm_count)
            yield L, lp
            L += 1

    gw = sm_count * launch_plan(c.n, c.A, c.k, c.W).warps
    one = next(L for L, lp in first(3 * gw + 1) if lp.rounds == 1 and lp.partial)
    many = next(L for L, lp in first(2 * gw * 32 + 1) if lp.rounds > 2 and lp.partial)
    return one, many
