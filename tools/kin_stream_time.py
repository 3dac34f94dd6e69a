#!/usr/bin/env python
"""Kinship analyses beyond one GPU's memory, timed on one GPU; prints one JSON document (and writes it to --out).

1. The whole C4 job (2,000 pools x 5 M biallelic loci = 10 M allele columns, 160 GB of f64) from synthetic columns
   through a 1.25 M-column handle (20 GB): pass 1 synthesises each of 8 blocks and adds its G G' to K (pg_kin_gram,
   then pg_kin_gram_accumulate); the eigen step runs once with P_total = 10 M; pass 2 re-synthesises each block and
   runs the covariate scan (k = 1), the records gathered on the host.  The accumulated K is checked against the fp64
   host sum of the blocks' own Gram matrices; the Gram rate is compared with the one-shot rate of pg_kin_gram_time.
2. File level: a synthetic 2,000-pool sync file through ols_iter_with_kinship, once with the default device budget
   (one device block) and once with a budget that forces about 4 blocks; per-phase wall times and the two outputs
   compared.

usage: kin_stream_time.py [--out FILE] [--file-gb 4] [--skip-file]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import poolgen_b200 as pb  # noqa: E402
from poolgen_b200 import sync_io  # noqa: E402

SEED = 0x5EED0004
N = 2000


def gpu_name_and_power():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    name, power = out[0].rsplit(",", 1)
    return name.strip(), power.strip()


def hw_flops(n, P):
    """what bench.py counts: the upper triangle of 128 x 128 tiles that the Gram kernel computes"""
    nt = (n + 127) // 128
    return 2.0 * (nt * (nt + 1) // 2) * 128 * 128 * P


def c4_job(ctx):
    blocks, per = 8, 625_000                       # loci per block: 1.25 M columns, 20 GB of G
    P_block, P_total = 2 * per, 2 * per * blocks
    kin = pb.Kinship(ctx, N, P_block)
    sync = kin.partial_device_ptr                   # returns after the handle's stream has drained
    # the one-shot rate at 1.25 M columns (and every module loaded)
    kin.synth(SEED, 0, per)
    kin.gram_time(1)
    one_shot_ms = kin.gram_time(3) / 3
    # pass 1
    synth_s, gram_s = [], []
    t_pass1 = time.perf_counter()
    for b in range(blocks):
        t0 = time.perf_counter()
        kin.reset()
        kin.synth(SEED, b * per, per)
        sync()
        t1 = time.perf_counter()
        kin.gram(accumulate=b > 0)
        sync()
        synth_s.append(t1 - t0)
        gram_s.append(time.perf_counter() - t1)
    pass1_s = time.perf_counter() - t_pass1
    K = kin.partial_get()
    # the check: the fp64 host sum of the blocks' own Gram matrices (not timed)
    S = np.zeros((N, N))
    for b in range(blocks):
        kin.reset()
        kin.synth(SEED, b * per, per)
        kin.gram()
        S += kin.partial_get()
    rel = float(np.abs(K - S).max() / np.abs(S).max())
    symmetric = bool(np.array_equal(K, K.T))
    kin.partial_set(K)
    # eigen step over the 10 M columns
    t0 = time.perf_counter()
    m = kin.eig_select(P_total, 0.75)
    eig_s = time.perf_counter() - t0
    # pass 2: re-synthesise, scan, gather
    phen = pb.synth_phen_host(SEED, N, 1)
    beta, pval = np.empty((1, P_total)), np.empty((1, P_total))
    load2_s, scan_s = [], []
    t_pass2 = time.perf_counter()
    for b in range(blocks):
        t0 = time.perf_counter()
        kin.reset()
        kin.synth(SEED, b * per, per)
        sync()
        t1 = time.perf_counter()
        bb, _v, pv = kin.covar_scan(phen)
        beta[:, b * P_block:(b + 1) * P_block] = bb
        pval[:, b * P_block:(b + 1) * P_block] = pv
        load2_s.append(t1 - t0)
        scan_s.append(time.perf_counter() - t1)
    pass2_s = time.perf_counter() - t_pass2
    kin.close()
    acc_ms = 1e3 * np.array(gram_s[1:])
    return {
        "pools": N, "columns": P_total, "device_blocks": blocks, "columns_per_block": P_block,
        "handle_gb": P_block * ((N + 3) & ~3) * 8 / 1e9,
        "pass1_s": pass1_s, "pass1_synth_s": float(sum(synth_s)), "pass1_gram_s": float(sum(gram_s)),
        "gram_first_ms": 1e3 * gram_s[0], "gram_accumulate_ms_median": float(np.median(acc_ms)),
        "gram_accumulate_ms_max": float(acc_ms.max()), "gram_one_shot_ms": one_shot_ms,
        "gram_hardware_tflops_one_shot": hw_flops(N, P_block) / one_shot_ms / 1e9,
        "gram_hardware_tflops_accumulated": hw_flops(N, P_total) / (1e3 * sum(gram_s)) / 1e9,
        "gram_accumulated_rate_over_one_shot": one_shot_ms * blocks / (1e3 * sum(gram_s)),
        "gram_timing": "host clock around each call, stream synchronised after it (one-shot: CUDA events, 3 launches)",
        "K_vs_host_sum_of_block_grams_max_rel": rel, "K_symmetric": symmetric, "K_check_rtol": 1e-13,
        "K_check_passed": bool(rel <= 1e-13 and symmetric),
        "eig_select_s": eig_s, "n_eigenvecs": m,
        "pass2_s": pass2_s, "pass2_synth_s": float(sum(load2_s)), "pass2_scan_s": float(sum(scan_s)),
        "total_s": pass1_s + eig_s + pass2_s,
        "records_finite_fraction": float(np.isfinite(beta).mean()),
    }


def write_sync_file(path, target_bytes):
    """a 2,000-pool synthetic sync file of about target_bytes bytes (the integer-hash workload, four alleles)"""
    per_line = 16 + N * 24
    chunk = max(1, (64 << 20) // per_line)
    n_chunks = max(1, int(target_bytes // (chunk * 28_900)))

    def gen(i):
        buf = np.empty(chunk * per_line, dtype=np.uint8)
        nb = pb.synth_sync_text_host(SEED, i * chunk, chunk, N, 4, buf)
        return buf[:nb]

    with open(path, "wb") as fh, ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        for i in range(0, n_chunks, 16):
            for part in ex.map(gen, range(i, min(n_chunks, i + 16))):
                fh.write(memoryview(part))
    return n_chunks * chunk


def file_level(ctx, gb):
    tmp = tempfile.mkdtemp(prefix="kin_stream_")
    try:
        free = shutil.disk_usage(tmp).free
        target = int(min(gb * 1e9, free / 4))
        fsync = os.path.join(tmp, "c4.sync")
        t0 = time.perf_counter()
        loci = write_sync_file(fsync, target)
        gen_s = time.perf_counter() - t0
        size = os.path.getsize(fsync)
        names = [f"p{i}" for i in range(N)]
        fs = pb.FilterStats(pool_sizes=np.full(N, 1.0 / N), min_allele_frequency=0.01)
        phen = pb.synth_phen_host(SEED, N, 1)
        src = pb.FileSyncPhen(fsync, names, fs.pool_sizes, phen, "ols_iter_with_kinship")
        bb = 32 << 20
        runs = {}
        tm = {}
        t0 = time.perf_counter()
        one = sync_io._iter_with_kinship(src, ctx, fs, True, 0.75, os.path.join(tmp, "one.csv"), 8, bb, "ols",
                                         timings=tm)
        tm["wall_s"] = time.perf_counter() - t0
        runs["unlimited"] = tm
        P = tm["columns"]
        cap = -(-P // 4) + sync_io.text_block_columns(bb, N)
        budget = sync_io.kin_device_bytes(N, cap, 1, bb, ctx.info()["sm_count"])
        tm = {}
        t0 = time.perf_counter()
        many = sync_io._iter_with_kinship(src, ctx, fs, True, 0.75, os.path.join(tmp, "many.csv"), 8, bb, "ols",
                                          device_bytes=budget, timings=tm)
        tm["wall_s"] = time.perf_counter() - t0
        tm["device_bytes"] = budget
        runs["forced"] = tm
        same = open(one, "rb").read() == open(many, "rb").read()
        for r in runs.values():
            # the rest of the wall time: reading the file on the host (the column bound's count and pass 1), the labels,
            # the sort and the rows
            r["host_rest_s"] = r["wall_s"] - sum(r[p] for p in ("pass1_load_s", "pass1_gram_s", "eig_s", "pass2_load_s",
                                                                 "scan_s", "write_s"))
            r["pass1_ns_per_column_load"] = 1e9 * r["pass1_load_s"] / r["columns"]
            r["pass1_ns_per_column_gram"] = 1e9 * r["pass1_gram_s"] / r["columns"]
        return {"file_bytes": size, "loci": loci, "disk_free_bytes": free, "generate_s": gen_s, "block_bytes": bb,
                "runs": runs, "outputs_byte_identical": same,
                "timing": "host clock per phase; the stream is synchronised after every Gram"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--file-gb", type=float, default=4.0)
    ap.add_argument("--skip-file", action="store_true")
    a = ap.parse_args()
    name, power = gpu_name_and_power()
    ctx = pb.Context(0)
    res = {"gpu": name, "power_limit": power, "c4_job": c4_job(ctx)}
    if not a.skip_file:
        res["file_level"] = file_level(ctx, a.file_gb)
    ctx.close()
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(doc + "\n")


if __name__ == "__main__":
    main()
