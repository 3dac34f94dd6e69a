#!/usr/bin/env python
"""sync2csv timed on one GPU; prints one JSON document (and writes it to --out).

1. Formatter alone, at 5, 100 and 2,000 pools, over the columns of one 32 MB block of synthetic sync text loaded with
   pg_kin_append_sync_text: (a) the device kernels with the text left in device memory, kernel times from
   torch.profiler's CUDA activity records (fmt_length_kernel, the cub scan, fmt_fit_kernel, fmt_write_kernel) in a run
   of their own; (b) the whole pg_kin_format_frequency_rows call, i.e. the kernels plus the copy of the rows to a pinned
   host buffer, host wall clock (the call ends in a stream synchronise); (c) the host's pg_format_frequency_rows on all
   host threads over the same columns (copied to the host first, not timed).  Rows/s and GB/s of row text.
2. Whole file: synthetic sync text of --file-gb GB at 2,000 and 100 pools (pg_synth_sync_text_host) through
   FileSyncPhen.write_csv: wall seconds per phase, once into a file on the local disk next to the input and once into
   /dev/null (the sink taken out).  The parent commit's write_csv -- every column in one handle, copied to the host,
   rows formatted by host threads -- runs on the same file, alternating with the new one; the sha256 of all outputs
   must be equal.

usage: sync2csv_time.py [--out FILE] [--file-gb 3] [--skip-file]
"""
import argparse
import builtins
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import poolgen_b200 as pb  # noqa: E402
from poolgen_b200 import capi, sync_io  # noqa: E402

SEED = 0x5EED0005
BLOCK = 32 << 20


def gpu_name_and_power():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    name, power = out[0].rsplit(",", 1)
    return name.strip(), power.strip()


def synth_text(n, n_loci, first=0):
    buf = np.empty(n_loci * (n * 20 + 64), np.uint8)  # synthetic depths stay below 100
    nb = pb.synth_sync_text_host(SEED, first, n_loci, n, 2, buf)
    return bytes(buf[:nb])


def formatter_alone(ctx, n):
    import torch
    text = synth_text(n, BLOCK // (n * 12 + 20))
    text = text[:text.rfind(b"\n", 0, BLOCK) + 1]
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.001)
    kin = pb.Kinship(ctx, n, sync_io.text_block_columns(len(text), n))
    L, off, pos, loc, alle = kin.append_sync_text(text, fs, sync_io._max_loci(len(text), n))
    P = kin.columns
    G = kin.get_columns(0, P)
    host_rows = pb.format_frequency_rows(G, loc, alle, pos, text=text, line_offsets=off)
    out, h = ctx.pinned_empty((len(host_rows) + 4096,), np.uint8)
    try:
        nb, nr = kin.format_frequency_rows(0, P, out)  # warm-up: modules, buffers
        assert (nb, nr) == (len(host_rows), P) and bytes(out[:nb]) == host_rows
        iters = 20
        t0 = time.perf_counter()
        for _ in range(iters):
            kin.format_frequency_rows(0, P, out)
        call_s = (time.perf_counter() - t0) / iters
        # kernel and copy times from the CUDA activity records
        acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
        with torch.profiler.profile(activities=acts) as prof:
            for _ in range(5):
                kin.format_frequency_rows(0, P, out)
            torch.cuda.synchronize()
        dev = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                key = ev.name
                if "fmt_" in key:
                    key = key.split("(")[0].split("::")[-1].replace("void ", "")
                elif "Scan" in key or "scan" in key:
                    key = "cub_scan"
                elif "Memcpy DtoH" in key:
                    key = "memcpy_dtoh"
                else:
                    continue
                dev[key] = dev.get(key, 0.0) + ev.time_range.elapsed_us() / 1e6 / 5  # us -> s per call
        kernels_s = sum(v for k, v in dev.items() if k != "memcpy_dtoh")
        threads = os.cpu_count() or 1
        pb.format_frequency_rows(G, loc, alle, pos, text=text, line_offsets=off, n_threads=threads)
        t0 = time.perf_counter()
        for _ in range(3):
            pb.format_frequency_rows(G, loc, alle, pos, text=text, line_offsets=off, n_threads=threads)
        host_s = (time.perf_counter() - t0) / 3

        def rate(s):
            if not s:
                return None  # no activity records
            return {"s": s, "rows_per_s": P / s, "GB_per_s": nb / s / 1e9}
        return {"n_pools": n, "loci": L, "rows": P, "row_bytes": nb, "text_block_bytes": len(text),
                "device_kernels": rate(kernels_s), "device_kernel_breakdown_s": dev,
                "device_call_with_copy": rate(call_s), "host_threads": threads, "host_formatter": rate(host_s)}
    finally:
        ctx.pinned_free(h)
        kin.close()


def parent_write_csv(src, ctx, fs, keep_p_minus_1, out, n_threads, block_bytes=BLOCK):
    """the parent commit's write_csv: every column of the file in one handle, copied to the host, rows formatted by
    host threads"""
    n = len(src.pool_names)
    kin = capi.Kinship(ctx, n, sync_io._count_columns_bound(src.filename_sync))
    max_loci = sync_io._max_loci(block_bytes, n)
    lab = sync_io._Labels()
    fname = src.filename_sync
    try:
        for _, block in sync_io._line_blocks(fname, 0, os.path.getsize(fname), block_bytes,
                                             [np.empty(block_bytes, np.uint8)]):
            lab.add(block, *kin.append_sync_text(block, fs, max_loci, keep_p_minus_1))
        ld = lab.finish()
        G = kin.get_columns(0, kin.columns)
    finally:
        kin.close()
    order = capi.sort_loci(ld.positions, chr_names=ld.chr_names, chr_index=ld.chr_index)
    rows = capi.format_frequency_rows(G, ld.col_locus, ld.col_allele, ld.positions, locus_order=order,
                                      n_threads=max(1, n_threads), chr_names=ld.chr_names, chr_index=ld.chr_index)
    with open(out, "xb") as fo:
        fo.write(capi.format_frequency_header(src.pool_names))
        fo.write(rows)
    return out


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as fh:
        for chunk in iter(lambda: fh.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def whole_file(ctx, n, gb, work):
    per_locus = len(synth_text(n, 100)) / 100
    n_loci = int(gb * 1e9 / per_locus)
    path = os.path.join(work, f"synth_{n}.sync")
    t0 = time.perf_counter()
    with open(path, "wb") as fh:
        step = max(1, (64 << 20) // int(per_locus))
        for a in range(0, n_loci, step):
            fh.write(synth_text(n, min(step, n_loci - a), a))
    gen_s = time.perf_counter() - t0
    names = [f"pool{i}" for i in range(n)]
    src = pb.FileSyncPhen(path, names, np.full(n, 1.0 / n), np.zeros((n, 1)), "sync2csv")
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.001)
    threads = os.cpu_count() or 1
    res = {"n_pools": n, "file_bytes": os.path.getsize(path), "loci": n_loci, "generate_s": gen_s, "runs": []}
    null_name = os.path.join(work, "to_dev_null.csv")
    real_open = builtins.open

    def open_null(f, mode="r", *a, **kw):  # write_csv's output file, redirected to /dev/null
        return real_open(os.devnull, "wb") if f == null_name else real_open(f, mode, *a, **kw)

    for rep in range(2):
        for arm in ("parent", "new_file", "new_null"):
            out = os.path.join(work, f"{arm}_{n}_{rep}.csv")
            tm = {}
            t0 = time.perf_counter()
            if arm == "parent":
                parent_write_csv(src, ctx, fs, False, out, threads)
            elif arm == "new_file":
                src.write_csv(ctx, fs, False, out, threads, timings=tm)
            else:
                sync_io.open = open_null
                try:
                    src.write_csv(ctx, fs, False, null_name, threads, timings=tm)
                finally:
                    del sync_io.open
            wall = time.perf_counter() - t0
            run = {"arm": arm, "rep": rep, "wall_s": wall, **tm}
            if arm != "new_null":
                run["out_bytes"] = os.path.getsize(out)
                run["sha256"] = sha256(out)
                os.remove(out)
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
    shas = {r["sha256"] for r in res["runs"] if "sha256" in r}
    res["outputs_equal"] = len(shas) == 1
    os.remove(path)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--file-gb", type=float, default=3.0)
    ap.add_argument("--skip-file", action="store_true")
    args = ap.parse_args()
    name, power = gpu_name_and_power()
    ctx = pb.Context(0)
    doc = {"gpu": name, "power_limit": power, "host_threads": os.cpu_count(), "formatter": []}
    for n in (5, 100, 2000):
        r = formatter_alone(ctx, n)
        doc["formatter"].append(r)
        print(json.dumps(r), flush=True)
    if not args.skip_file:
        work = tempfile.mkdtemp(prefix="sync2csv_")
        try:
            doc["whole_file"] = [whole_file(ctx, n, args.file_gb, work) for n in (2000, 100)]
        finally:
            shutil.rmtree(work, ignore_errors=True)
    ctx.close()
    txt = json.dumps(doc, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
