#!/usr/bin/env python
"""Times the OLS scan past the resident-phenotype limit (scan_kernel_wide, DESIGN 3.5) on device-synthesised batches.

For each shape: loci/s of one run (streaming kernel + fix-up kernel) and the algorithmic bytes per locus
8 n A + 32 (A - 1) k over the run time, as a fraction of the device-to-device copy rate measured in the same process.
Shapes: n = 8,192 and 16,384 at A = 4, k = 1 and 3 (the wide kernel), and n = 6,144 at A = 4, k = 1 and 3 on the
resident kernel and on the wide kernel (PG_SCAN_WIDE=1, read once per process: a second process).  Each batch holds
about 8 GB of frequencies, far above the 126 MB of L2.

usage: wide_scan_time.py [--out FILE] [--iters N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

A = 4
SHAPES = [(8192, 1), (8192, 3), (16384, 1), (16384, 3)]
EDGE = [(6144, 1), (6144, 3)]
BATCH_BYTES = 8e9


def gpu_name_and_power():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout.strip().splitlines()
    name, power = out[0].rsplit(",", 1)
    return name.strip(), power.strip()


def copy_rate_gbs():
    """device-to-device copy of 4 GiB: bytes read + written over the time, best of 5"""
    import torch
    src = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * src.numel() * 8 / (e0.elapsed_time(e1) * 1e6))
    del src, dst
    torch.cuda.empty_cache()
    return best


def time_shapes(shapes, iters):
    import poolgen_b200 as pb
    ctx = pb.Context(0)
    out = []
    for n, k in shapes:
        L = int(BATCH_BYTES // (8 * n * A))
        phen = pb.synth_phen_host(0x5EED0003, n, k)
        fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
        scan = pb.Scan(ctx, pb.KIND_OLS, fs, n, np.arange(A, dtype=np.uint8), phen)
        b = scan.batch(L)
        b.synth(0x5EED0003, 0, L)
        b.time_runs(2)
        ms, _ = b.time_runs(iters)
        per = ms / iters
        alg = 8 * n * A + 32 * (A - 1) * k
        out.append(dict(n=n, A=A, k=k, loci=L, ms_per_run=per, loci_per_s=L / (per * 1e-3),
                        alg_gbs=alg * L / (per * 1e6), kernel="wide" if os.environ.get("PG_SCAN_WIDE") or n > 6144
                        else "resident"))
        b.close()
        scan.close()
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--edge-only", action="store_true", help=argparse.SUPPRESS)  # the PG_SCAN_WIDE=1 process
    a = ap.parse_args()
    if a.edge_only:
        print(json.dumps(time_shapes(EDGE, a.iters)))
        return
    name, power = gpu_name_and_power()
    hbm = copy_rate_gbs()
    rows = time_shapes(SHAPES + EDGE, a.iters)
    env = dict(os.environ, PG_SCAN_WIDE="1")
    sub = subprocess.run([sys.executable, os.path.abspath(__file__), "--edge-only", "--iters", str(a.iters)],
                         stdout=subprocess.PIPE, text=True, env=env, check=True)
    rows += json.loads(sub.stdout.strip().splitlines()[-1])
    for r in rows:
        r["frac_of_copy_rate"] = r["alg_gbs"] / hbm
        print(f"n={r['n']:6d} A={r['A']} k={r['k']} {r['kernel']:8s}: {r['loci_per_s'] / 1e6:8.3f} M loci/s  "
              f"{r['alg_gbs']:7.0f} GB/s alg  {r['frac_of_copy_rate']:.3f} of the copy rate")
    res = dict(gpu=name, power_limit=power, copy_rate_gbs=hbm, alg_bytes="8 n A + 32 (A - 1) k per locus", rows=rows)
    print(f"{name}, power limit {power}, device copy {hbm:.0f} GB/s")
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
