#!/usr/bin/env python
"""The file-level entries of poolgen_b200/sync_io.py timed against another commit's Python code on one GPU; prints one
JSON document (and writes it to --out).

A synthetic sync file of --file-gb GB (pg_synth_sync_text_host, --pools pools, four alleles, ends in a newline) goes
through read_analyse_write (ols_iter and chisq, 4 reader threads), write_csv, and ols_iter_with_kinship with the free
device memory and with a budget that forces three device blocks.  --parent names a directory that holds the other
commit's poolgen_b200 package; it loads this tree's libraries, so only the Python code differs.  The two arms alternate
run by run, --reps times, after one untimed pass over a small file.  Per run: wall seconds and the sha256 of the output;
per entry, whether all outputs are identical.

usage: file_entries_time.py --parent DIR [--out FILE] [--file-gb 2] [--pools 100] [--reps 3]
"""
import argparse
import hashlib
import importlib.util
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

SEED = 0x5EED0006
BLOCK = 32 << 20


def gpu_name_and_power():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    name, power = out[0].rsplit(",", 1)
    return name.strip(), power.strip()


def load_parent(path):
    """the poolgen_b200 package under `path`, imported as parent_poolgen_b200 and bound to this tree's libraries"""
    pkg = os.path.join(os.path.abspath(path), "poolgen_b200")
    spec = importlib.util.spec_from_file_location("parent_poolgen_b200", os.path.join(pkg, "__init__.py"),
                                                  submodule_search_locations=[pkg])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    mod.capi.LIB_PATH, mod.capi.SYNTH_LIB_PATH = pb.capi.LIB_PATH, pb.capi.SYNTH_LIB_PATH
    return mod


def write_sync_file(path, n, target_bytes):
    per_line = 16 + n * 24
    chunk = max(1, (64 << 20) // per_line)

    def gen(first):
        buf = np.empty(chunk * per_line, dtype=np.uint8)
        return buf[:pb.synth_sync_text_host(SEED, first, chunk, n, 4, buf)]

    written, first, batch = 0, 0, 4 * chunk
    with open(path, "wb") as fh, ThreadPoolExecutor(max_workers=4) as ex:
        while written < target_bytes:
            for part in ex.map(gen, range(first, first + batch, chunk)):
                fh.write(memoryview(part))
                written += part.size
            first += batch
    return first


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as fh:
        for chunk in iter(lambda: fh.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def run_entry(mod, ctx, entry, path, n, phen, out, budget, timings):
    names = [f"p{i}" for i in range(n)]
    fs = mod.FilterStats(pool_sizes=np.full(n, 1.0 / n), min_allele_frequency=0.01)
    src = mod.FileSyncPhen(path, names, fs.pool_sizes, phen, entry)
    if entry == "ols_iter":
        src.read_analyse_write(ctx, fs, out, 4, mod.KIND_OLS)
    elif entry == "chisq":
        mod.FileSync(path, "chisq_test").read_analyse_write(ctx, fs, out, 4, mod.KIND_CHISQ)
    elif entry == "sync2csv":
        src.write_csv(ctx, fs, False, out, 8)
    else:
        mod.sync_io._iter_with_kinship(src, ctx, fs, True, 0.75, out, 8, BLOCK, "ols",
                                       device_bytes=budget if entry == "kinship_3_blocks" else None, timings=timings)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True)
    ap.add_argument("--out", default="")
    ap.add_argument("--file-gb", type=float, default=2.0)
    ap.add_argument("--pools", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    name, power = gpu_name_and_power()
    arms = {"parent": load_parent(a.parent), "new": pb}
    ctxs = {arm: mod.Context(0) for arm, mod in arms.items()}
    n = a.pools
    phen = pb.synth_phen_host(SEED, n, 1)
    entries = ["ols_iter", "chisq", "sync2csv", "kinship_1_block", "kinship_3_blocks"]
    work = tempfile.mkdtemp(prefix="file_entries_")
    res = {"gpu": name, "power_limit": power, "host_threads": os.cpu_count(), "pools": n, "block_bytes": BLOCK,
           "runs": []}
    try:
        path = os.path.join(work, "synth.sync")
        t0 = time.perf_counter()
        res["loci"] = write_sync_file(path, n, a.file_gb * 1e9)
        res["generate_s"] = time.perf_counter() - t0
        res["file_bytes"] = os.path.getsize(path)
        # the budget of three device blocks, from the column count of a run with the whole device
        tm = {}
        run_entry(pb, ctxs["new"], "kinship_1_block", path, n, phen, os.path.join(work, "probe.csv"), None, tm)
        os.remove(os.path.join(work, "probe.csv"))
        cap = -(-tm["columns"] // 3) + pb.sync_io.text_block_columns(BLOCK, n)
        budget = pb.sync_io.kin_device_bytes(n, cap, 1, BLOCK, ctxs["new"].info()["sm_count"])
        res["kinship_3_blocks_device_bytes"] = budget
        small = os.path.join(work, "small.sync")
        write_sync_file(small, n, 20e6)
        for arm, mod in arms.items():  # modules, buffers, first-call costs
            for entry in entries:
                out = os.path.join(work, f"warm_{arm}_{entry}.csv")
                run_entry(mod, ctxs[arm], entry, small, n, phen, out, budget, {})
                os.remove(out)
        for rep in range(a.reps):
            for entry in entries:
                for arm in (("parent", "new") if rep % 2 == 0 else ("new", "parent")):
                    out = os.path.join(work, f"{arm}_{entry}_{rep}.csv")
                    tm = {}
                    t0 = time.perf_counter()
                    run_entry(arms[arm], ctxs[arm], entry, path, n, phen, out, budget, tm)
                    run = {"entry": entry, "arm": arm, "rep": rep, "wall_s": time.perf_counter() - t0,
                           "out_bytes": os.path.getsize(out), "sha256": sha256(out)}
                    if "device_blocks" in tm:
                        run["device_blocks"] = tm["device_blocks"]
                    os.remove(out)
                    res["runs"].append(run)
                    print(json.dumps(run), flush=True)
    finally:
        shutil.rmtree(work, ignore_errors=True)
        for ctx in ctxs.values():
            ctx.close()
    summary = {}
    for entry in entries:
        rs = [r for r in res["runs"] if r["entry"] == entry]
        walls = {arm: [r["wall_s"] for r in rs if r["arm"] == arm] for arm in arms}
        summary[entry] = {"outputs_identical": len({r["sha256"] for r in rs}) == 1,
                          **{f"{arm}_wall_s": {"min": min(w), "median": float(np.median(w)), "max": max(w)}
                             for arm, w in walls.items()}}
    res["summary"] = summary
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(doc + "\n")


if __name__ == "__main__":
    main()
