#!/usr/bin/env python
"""bench.py -- loci/s of the `ols_iter` per-locus scan (f64) on 1..8 B200, with its HBM roofline.

Workload (BASELINE.json configs[2], "C3"): synthetic sync counts, 1,000 pools x 10,000,000 loci x 4 alleles,
3 phenotypes, sharded over 8 GPUs = 1,250,000 loci per GPU.  The full matrix (323 GB of f64) does not fit one GPU,
so the bench is WEAK-scaled: every rank holds one 1.25M-locus shard (40 GB resident in HBM, generated on the
device by the integer-hash generator the CPU oracle can replay); at --gpus 8 the job is exactly C3.
A step = one pass of the scan kernel over the rank's resident shard (inputs 40 GB >> 126 MB L2, so no flush).
The other BASELINE configs are reported in the same JSON line under the top-level keys "c2", "c4", "c5" and "text".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--loci-per-gpu L] [--dump-outputs DIR]

--dump-outputs DIR writes the records of the last timed step (a fixed, seeded sample of the shard's loci, the output
rows of each) as DIR/<name>.npy in f64, so that two builds can be compared output for output on the same synthetic
inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POOLS, N_ALLELES, N_PHEN = 1000, 4, 3
LOCI_PER_GPU = 1_250_000
SEED = 0x5EED0003
ALG_BYTES_PER_LOCUS = 8 * N_POOLS * N_ALLELES + 32 * (N_ALLELES - 1) * N_PHEN  # SURVEY.md 8(d): 32,288 B
METRIC = "loci/sec for ols_iter (f64)"
DUMP_BYTES = 60_000_000  # all ranks' --dump-outputs files together, below 64 MB with room for the .npy headers
DUMP_SEED = 0x5EED00D


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profile(n_pools: int, n_alleles: int, n_phen: int):
    """DRAM bytes per locus of one step (dram__bytes_read.sum + dram__bytes_write.sum of the streaming kernel and the
    fix-up kernel) read from the committed `ncu --set full` capture of this shape: profiles/ncu_raw_r<N>.csv with its
    sidecar profiles/ncu_raw_r<N>.json ({"shape": [pools, alleles, phenotypes], "loci": L, "kernels": [...]}).
    Returns (bytes per locus, file) or (None, None) when no capture of this shape is committed."""
    import csv
    import glob
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for meta_path in sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_raw_r*.json")), reverse=True):
        try:
            with open(meta_path) as fh:
                meta = json.load(fh)
            if list(meta.get("shape", [])) != [n_pools, n_alleles, n_phen]:
                continue
            with open(meta_path[:-5] + ".csv", newline="") as fh:
                rows = list(csv.reader(fh))
            hdr, units = rows[0], rows[1]
            kcol = hdr.index("Kernel Name")
            total = 0.0
            seen = set()
            for r in rows[2:]:
                name = r[kcol]
                key = next((k for k in meta["kernels"] if k in name), None)
                if key is None or key in seen:
                    continue  # one launch of each kernel
                seen.add(key)
                for col in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    i = hdr.index(col)
                    total += float(r[i].replace(",", "")) * unit[units[i]]
            if seen:
                return total / float(meta["loci"]), os.path.relpath(meta_path[:-5] + ".csv", ROOT)
        except (OSError, ValueError, KeyError, IndexError):
            continue
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.stamps = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 9:
                self.rows.append(f)
                self.stamps.append(time.time())

    def samples_since(self, t0: float) -> int:
        return sum(1 for t in self.stamps if t >= t0)

    def keep_since(self, t0: float):
        """only the samples taken while the GPU was under load count"""
        keep = [i for i, t in enumerate(self.stamps) if t >= t0]
        self.rows = [self.rows[i] for i in keep]
        self.stamps = [self.stamps[i] for i in keep]

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for f in self.rows:
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def cpu_reference_rate(seconds_target: float, n_threads: int, tight: bool = False):
    """The reference's CPU path restated (oracle/poolgen_oracle.c, one OS thread per contiguous locus range like
    src/base/sync.rs:917-939) timed on a bounded sample of the SAME workload.  tight=False is the faithful structure
    (per-locus allocations, the pool-size total re-summed per pool and allele as src/base/sync.rs:262-270 does, X'X
    refactored per phenotype as src/gwas/ols.rs:180); tight=True the same arithmetic without that avoidable work
    (bit-identical records, tests/test_oracle_golden.py) -- the upper bound of what the CPU path could do.  The inputs
    come from libpoolgen_synth.so: this leg never maps the product library."""
    from oracle import pgo
    from poolgen_b200 import capi
    phen = capi.synth_phen_host(SEED, N_POOLS, N_PHEN)
    fs = pgo.FilterStats(pool_sizes=np.full(N_POOLS, 1.0 / N_POOLS))
    codes = np.arange(N_ALLELES, dtype=np.uint8)
    probe = (2048 if tight else 256) * n_threads
    counts = capi.synth_counts_host(SEED, 0, probe, N_POOLS, N_ALLELES)
    t0 = time.perf_counter()
    pgo.scan_batch(pgo.SCAN_OLS, counts, codes, phen, fs, n_threads, tight=tight)
    dt = time.perf_counter() - t0
    rate = probe / dt
    sample = int(max(probe, min(400_000, rate * seconds_target)))
    sample -= sample % n_threads
    counts = capi.synth_counts_host(SEED, 0, sample, N_POOLS, N_ALLELES)

    def step():
        t0 = time.perf_counter()
        pgo.scan_batch(pgo.SCAN_OLS, counts, codes, phen, fs, n_threads, tight=tight)
        return time.perf_counter() - t0
    return step, sample


def product_library_mapped() -> bool:
    with open("/proc/self/maps") as fh:
        return any("libpoolgen_cuda" in line for line in fh)


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    n_threads = os.cpu_count() or 1
    t_start = time.perf_counter()
    step, sample = cpu_reference_rate(args.cpu_seconds, n_threads)
    print(f"[reference arm] sample of {sample} loci ready after {time.perf_counter() - t_start:.1f} s", file=sys.stderr)
    for _ in range(args.warmup):
        step()
    times = [step() for _ in range(args.steps)]
    print(f"[reference arm] {args.warmup}+{args.steps} steps done after {time.perf_counter() - t_start:.1f} s", file=sys.stderr)
    total = sum(times)
    value = sample * args.steps / total
    # the "tight" variant next to it (BASELINE.md 2): same records without the reference's avoidable work
    tstep, tsample = cpu_reference_rate(args.cpu_seconds, n_threads, tight=True)
    tstep()
    tdt = min(tstep() for _ in range(2))
    print(f"[reference arm] tight variant: {tsample} loci in {tdt:.2f} s", file=sys.stderr)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "loci/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"C3 ols_iter shard: {N_POOLS} pools x {LOCI_PER_GPU} loci/GPU x {N_ALLELES} alleles, "
                               f"{N_PHEN} phenotypes (8 GPUs = the 10M-locus job)",
                   "reference_arm": f"the CPU path times a bounded sample of {sample} loci of that workload per step "
                                    "(in-memory counts, parsing and CSV writing excluded) and scales linearly in loci",
                   "filters": "CLI defaults: min depth 1, MAF 0.001, missingness 0"},
        "cpu_baseline": {"value": value, "unit": "loci/s", "cores": n_threads, "kind": "port",
                         "sample": f"{sample} loci of the C3 shape per step, {n_threads} OS threads over contiguous locus ranges",
                         "variant": "faithful (per-locus allocations, pool-size total re-summed per pool and allele, "
                                    "X'X refactored per phenotype -- what the reference does)",
                         "tight": {"value": tsample / tdt, "unit": "loci/s", "cores": n_threads,
                                   "sample": f"{tsample} loci, best of 2",
                                   "variant": "same arithmetic and records, total hoisted, one inversion per locus, "
                                              "no per-locus allocation"}},
        "e2e": {"value": value, "unit": "loci/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "maps_product_library": product_library_mapped(),
    }
    print(json.dumps(line))
    return 0


def sample_records(res, first_locus: int, world: int) -> dict:
    """the ScanResults of a shard reduced to a fixed, seeded sample of its loci (all of them when they fit), every
    array in f64; the samples of all ranks together stay under DUMP_BYTES.  The library leaves the slots of a locus that
    hold no output row NaN (all of them when the locus is filtered or failed): freq_mean [rows] and stats [rows, k, 4]
    keep the output rows only, in locus order, and status / n_out say which locus each row belongs to."""
    L, S = res.freq_mean.shape
    per_locus = 8 * (1 + 1 + 1 + res.alleles.shape[1] + S + res.stats[0].size)
    n = min(L, DUMP_BYTES // (world * per_locus))
    idx = np.arange(L) if n == L else np.sort(np.random.default_rng(DUMP_SEED).choice(L, n, replace=False))
    from poolgen_b200.capi import LOCUS_OK
    status, n_out = res.status[idx], res.n_out[idx]
    rows = (status == LOCUS_OK)[:, None] & (np.arange(S)[None, :] < n_out[:, None])
    return {"locus": (first_locus + idx).astype(np.float64), "status": status.astype(np.float64),
            "n_out": n_out.astype(np.float64), "alleles": res.alleles[idx].astype(np.float64),
            "freq_mean": res.freq_mean[idx][rows], "stats": res.stats[idx][rows]}


def bind_to_gpu_numa_node(gpu_index: int):
    """pin this process to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host memory is allocated:
    with 8 ranks on one box the slabs of the end-to-end leg otherwise sit on one socket and every copy crosses it"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001 -- a missing NVML binding only costs the binding
        return None


def run_cuda(args):
    import torch
    import poolgen_b200 as pb
    rank, local, world = dist_env()
    # rank 0 prints ONE JSON line: everything else a library writes to fd 1 (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    cpus = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist = None
        torch.cuda.set_device(local)
    ctx = pb.Context(local)
    L = args.loci_per_gpu
    phen = pb.synth_phen_host(SEED, N_POOLS, N_PHEN)
    fs = pb.FilterStats(pool_sizes=np.full(N_POOLS, 1.0 / N_POOLS))
    codes = np.arange(N_ALLELES, dtype=np.uint8)
    scan = pb.Scan(ctx, pb.KIND_OLS, fs, N_POOLS, codes, phen)
    batch = scan.batch(L)
    batch.synth(SEED, rank * L, L)  # this rank's contiguous locus range of the 10M-locus job
    batch.sync()
    in_bytes, out_bytes = batch.bytes()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    batch.time_runs(1)
    t_load = time.time()
    batch.time_runs(max(3, args.warmup))  # warm-up (>= 3 passes)
    barrier()
    ms, launches = batch.time_runs(args.steps)  # CUDA events on the stream the kernels are launched on
    barrier()
    # the records of the last timed step, copied out before the batch runs again: the OK fraction (a sanity check, not a
    # parity test: tests/ does that) and the --dump-outputs sample
    batch.download()
    batch.sync()
    rv = batch.results_view()
    meta = np.ctypeslib.as_array(rv.meta, shape=(L,))
    ok_frac = float(((meta & 0xFF) == pb.LOCUS_OK).mean())
    dump = sample_records(pb.ScanResults.from_c(rv), rank * L, world) if args.dump_outputs else None
    # the timed region can be shorter than nvidia-smi's sampling period: keep the same kernel running (untimed) until
    # at least three clock samples were taken under load
    t_end = time.time() + 4.0
    while sampler.proc and sampler.samples_since(t_load) < 3 and time.time() < t_end:
        batch.time_runs(max(1, args.steps))
    sampler.keep_since(t_load)
    clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * L * args.steps / (ms_max * 1e-3)

    # ---- end to end through the C ABI with HOST buffers: pinned counts -> H2D -> ingest -> scan -> D2H records
    slab = args.e2e_slab
    n_slabs = args.e2e_slabs
    # the narrowest count type that holds the slab (the reader knows its maximum count): u8 here, depths are 20..100
    host, hptr = ctx.pinned_empty((3, slab, N_ALLELES, N_POOLS), np.uint8)
    for i in range(3):
        c = pb.synth_counts_host(SEED, rank * L + i * slab, slab, N_POOLS, N_ALLELES)
        assert c.max() < 256
        host[i] = c.astype(np.uint8)
    scan.stream_begin(slab)
    for i in range(3):  # warm-up
        scan.collect(scan.submit_counts(host[i]), copy=False)
    barrier()
    t0 = time.perf_counter()
    pending = []
    kept = 0
    for i in range(n_slabs):
        pending.append(scan.submit_counts(host[i % 3]))
        if len(pending) == 3:
            r = scan.collect(pending.pop(0), copy=False)
            kept += int(r.n_loci)
    while pending:
        r = scan.collect(pending.pop(0), copy=False)
        kept += int(r.n_loci)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * slab * n_slabs / float(te.item())
    h2d = slab * N_ALLELES * N_POOLS * host.dtype.itemsize
    d2h = slab * (8 + 8 * (N_ALLELES - 1) + 32 * (N_ALLELES - 1) * N_PHEN)
    ctx.pinned_free(hptr)

    batch.close()
    scan.close()
    extras = {}
    if not args.no_extras:
        if rank == 0:
            extras = c2_numbers(ctx, pb)
            extras.update(c5_numbers(ctx, pb, args.c5_loci))
            extras.update(text_numbers(ctx, pb))
            extras.update(nm_numbers(ctx, pb))
        kin = c4_numbers(ctx, pb, dist, rank, world)  # every rank takes part (column shards + all-reduce)
        if rank == 0:
            extras.update(kin)

    if rank == 0:
        peak, peak_src = measured_peaks()
        per_launch_ms = ms / args.steps  # one step = the streaming kernel + the (short) fix-up kernel over its deferred loci
        achieved = ALG_BYTES_PER_LOCUS * L / (per_launch_ms * 1e-3) / 1e9
        cpu = None
        if world == 1 and not args.no_cpu:
            n_threads = os.cpu_count() or 1
            step, sample = cpu_reference_rate(12.0, n_threads)
            dt = step()
            tstep, tsample = cpu_reference_rate(6.0, n_threads, tight=True)
            tdt = tstep()
            cpu = {"value": sample / dt, "unit": "loci/s", "cores": n_threads, "kind": "port",
                   "sample": f"{sample} loci of the C3 shape (1000 pools x 4 alleles, 3 phenotypes), in-memory counts, "
                             f"{n_threads} OS threads over contiguous locus ranges, {dt:.1f} s",
                   "variant": "faithful (per-locus allocations, pool-size total re-summed per pool and allele as "
                              "src/base/sync.rs:262-270, X'X refactored per phenotype as src/gwas/ols.rs:180)",
                   "tight": {"value": tsample / tdt, "unit": "loci/s", "cores": n_threads,
                             "sample": f"{tsample} loci, {tdt:.1f} s",
                             "variant": "same arithmetic, bit-identical records: total hoisted, one inversion per "
                                        "locus, no per-locus allocation"}}
        traffic_per_locus, traffic_file = traffic_from_profile(N_POOLS, N_ALLELES, N_PHEN)
        line = {
            "metric": METRIC, "value": value, "unit": "loci/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C3 ols_iter shard: {N_POOLS} pools x {L} loci/GPU x {N_ALLELES} alleles, "
                                   f"{N_PHEN} phenotypes (8 GPUs = the 10M-locus job)",
                       "l2": f"inputs {in_bytes / 1e9:.1f} GB per pass >> 126 MB L2, no flush needed",
                       "filters": "CLI defaults: min depth 1, MAF 0.001, missingness 0", "ok_fraction": ok_frac,
                       "e2e_format": f"u8 counts (every count < 256), slabs of {slab} loci, depth-3 pipeline, {n_slabs} slabs"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         # dram__bytes_read + dram__bytes_write of one step (streaming + fix-up kernel), read at run time
                         # from the committed ncu --set full capture of this shape, scaled to the resident batch
                         "traffic": (traffic_per_locus * L) if traffic_per_locus else None,
                         "traffic_unit": "bytes per launch", "traffic_source": traffic_file,
                         "traffic_bytes_per_locus": traffic_per_locus, "peak_source": peak_src,
                         "algorithmic_bytes_per_locus": ALG_BYTES_PER_LOCUS,
                         "resident_input_bytes_per_locus": in_bytes / L, "kernel_ms": per_launch_ms},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "loci/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        # the other BASELINE configs, top level so that they survive the driver's parse of this line
        for key, names in (("c2", ("c2_ols_iter", "c2_pearson_corr")), ("c5", ("c5_chisq_test", "c5_fisher_exact_test")),
                           ("c4", ("c4_kinship",)), ("text", ("e2e_sync_text", "e2e_text_to_csv")),
                           ("nelder_mead", ("nelder_mead",))):
            got = {n: extras[n] for n in names if n in extras}
            if got:
                line[key] = got[names[0]] if len(names) == 1 else got
        if cpus is not None:
            line["config"]["cpu_affinity"] = f"each rank bound to the {len(cpus)} CPUs next to its GPU (NVML)"
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + (f".rank{rank}" if world > 1 else "") + ".npy"), a)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    os.dup2(real_stdout, 1)
    os.close(real_stdout)
    return 0


def c2_numbers(ctx, pb):
    """BASELINE.json configs[1] (C2): 100 pools x 1M loci x 4 alleles, 1 phenotype, ols_iter + pearson_corr."""
    out = {}
    n, A, k, L = 100, 4, 1, 1_000_000
    phen = pb.synth_phen_host(0x5EED0002, n, k)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    peak, _ = measured_peaks()
    alg = 8 * n * A + 32 * (A - 1) * k
    for name, kind in (("c2_ols_iter", pb.KIND_OLS), ("c2_pearson_corr", pb.KIND_CORR)):
        scan = pb.Scan(ctx, kind, fs, n, np.arange(A, dtype=np.uint8), phen)
        b = scan.batch(L)
        b.synth(0x5EED0002, 0, L)
        b.time_runs(5)
        ms, nl = b.time_runs(20)
        per = ms / 20
        out[name] = {"loci_per_s": L / (per * 1e-3), "kernel_ms": per,
                     "roofline_frac": alg * L / (per * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_locus": alg,
                     "note": "3.3 GB input > L2 (126 MB); time = streaming kernel + fix-up kernel"}
        b.close()
        scan.close()
    return out


def c5_numbers(ctx, pb, L=50_000_000):
    """BASELINE.json configs[4] (C5): chisq_test + fisher_exact_test on 2 pools x 50M loci of synthetic counts
    (count path: u32 [locus][allele][pool] in, 2 f64 + status out; 4*n*6 + 16 = 64 algorithmic bytes per locus)."""
    out = {}
    n, A = 2, 6
    fs = pb.FilterStats(pool_sizes=np.full(n, 0.5))
    peak, _ = measured_peaks()
    alg = 4 * n * 6 + 16
    for name, kind in (("c5_chisq_test", pb.KIND_CHISQ), ("c5_fisher_exact_test", pb.KIND_FISHER)):
        scan = pb.Scan(ctx, kind, fs, n, np.arange(A, dtype=np.uint8))
        b = scan.batch(L)
        b.synth(0x5EED0005, 0, L)
        b.time_runs(3)
        ms, nl = b.time_runs(5)
        per = ms / 5
        out[name] = {"loci_per_s": L / (per * 1e-3), "kernel_ms": per, "loci": L,
                     "roofline_frac": alg * L / (per * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_locus": alg,
                     "note": f"{L * n * A * 4 / 1e9:.1f} GB of counts per pass > L2 (126 MB); Fisher is compute-bound "
                             "(O((n a)^2 (n+a)) log10/pow per locus)"}
        b.close()
        scan.close()
    return out


def nm_numbers(ctx, pb):
    """SURVEY 8f-3 / 8f-4: the Nelder-Mead analyses.  mle_iter on the C2 shape (100 pools, 1 phenotype) and gwalpha (LS,
    ML) on 5 pools: filter-only scan pass + simplex kernel (1,000-iteration cap per search).  Compute-bound by design
    (the reference's own algorithm): reported as loci/s, no roofline claim."""
    out = {}
    n, A, k, L = 100, 4, 1, 200_000
    phen = pb.synth_phen_host(0x5EED0002, n, k)
    fs = pb.FilterStats(pool_sizes=np.full(n, 1.0 / n))
    scan = pb.Scan(ctx, pb.KIND_MLE, fs, n, np.arange(A, dtype=np.uint8), phen)
    b = scan.batch(L)
    b.synth(0x5EED0002, 0, L)
    b.time_runs(1)
    ms, _ = b.time_runs(2)
    out["mle_iter_c2_shape"] = {"loci_per_s": L / (ms / 2 * 1e-3), "ms": ms / 2, "loci": L, "n_pools": n, "n_phen": k}
    b.close()
    scan.close()
    n, L = 5, 20_000
    fmt = np.full((5, 3), -np.inf)
    fmt[:, 0] = 0.2
    fmt[:, 1] = (0.0, 0.1, 0.4, 0.7, 0.9)
    fmt[:3, 2] = (0.02, 0.0, 0.9)
    fs = pb.FilterStats(pool_sizes=np.full(n, 0.2))
    for name, kind in (("gwalpha_ls_5_pools", pb.KIND_GWALPHA_LS), ("gwalpha_ml_5_pools", pb.KIND_GWALPHA_ML)):
        scan = pb.Scan(ctx, kind, fs, n, np.arange(A, dtype=np.uint8), fmt)
        b = scan.batch(L)
        b.synth(0x5EED0005, 0, L)
        ms, _ = b.time_runs(1)
        out[name] = {"loci_per_s": L / (ms * 1e-3), "ms": ms, "loci": L, "n_pools": n}
        b.close()
        scan.close()
    # mle_iter_with_kinship (mle_with_covariate, gwas/mle.rs:307-463): C4's pool count, no PCs (what raw frequencies
    # select), one search over [sigma2, b_0, b_g] per column
    n, P = 2000, 200_000
    kin = pb.Kinship(ctx, n, P)
    kin.synth(0x5EED0004, 0, P // 2)
    kin.set_covariates(np.zeros((n, 0)))
    y = pb.synth_phen_host(0x5EED0004, n, 1)
    kin.mle_scan(y)
    ms = kin.mle_scan(y, timed=True)[3]
    out["mle_iter_with_kinship_c4_pools"] = {"columns_per_s": kin.columns / (ms * 1e-3), "ms": ms, "columns": int(kin.columns),
                                             "n_pools": n, "n_covariates": 0}
    kin.close()
    return {"nelder_mead": out}


def text_numbers(ctx, pb, n_threads=2):
    """SURVEY 8f-1 + 8f-2: the whole stretch of `read_analyse_write` the library replaces, end to end from sync TEXT in
    pinned host memory (what the reference's reader threads start from) to (a) records on the host and (b) the CSV rows
    of the reference's writer: H2D of the raw text, device-side parse, ingest, scan, D2H, pg_format_rows.  C3 shape,
    slabs of 4,096 loci, `n_threads` reader threads with one scan handle each (the reference runs one reader per file
    chunk, src/base/sync.rs:917-939) so that one thread's host synchronisation overlaps another's copy."""
    import ctypes as C
    import threading
    import torch
    slab, slabs_per_thread = 4096, 24   # long enough that the three formats of the pipeline drain weigh little
    per_locus_cap = 16 + N_POOLS * 24
    host, hptr = ctx.pinned_empty((2, slab * per_locus_cap), np.uint8)
    nbytes = [pb.synth_sync_text_host(SEED, i * slab, slab, N_POOLS, N_ALLELES, host[i]) for i in range(2)]
    phen = pb.synth_phen_host(SEED, N_POOLS, N_PHEN)
    fs = pb.FilterStats(pool_sizes=np.full(N_POOLS, 1.0 / N_POOLS))
    lib = pb.capi.lib()
    scans = [pb.Scan(ctx, pb.KIND_OLS, fs, N_POOLS, np.arange(6, dtype=np.uint8), phen) for _ in range(n_threads)]
    for sc in scans:
        sc.stream_begin(slab)
    cap = slab * N_PHEN * 3 * 96
    outs = [C.create_string_buffer(cap) for _ in range(n_threads)]
    fmt_threads = max(1, (os.cpu_count() or 1) // n_threads)
    rows = [0] * n_threads

    def reader(t, n_slabs, to_csv):
        sc = scans[t]
        pending = []

        def finish(item):
            ticket, i = item
            r = sc.collect(ticket, copy=False)
            assert r.n_loci == slab, r.n_loci
            if not to_csv:
                return
            po, pp = C.c_void_p(), C.c_void_p()
            assert lib.pg_scan_text_labels(sc._h, int(ticket), C.byref(po), C.byref(pp)) == 0
            lab = pb.capi._RowLabels()
            lab.positions = C.cast(pp, C.POINTER(C.c_uint64))
            lab.text = C.cast(host[i % 2].ctypes.data, C.c_char_p)
            lab.line_offsets = C.cast(po, C.POINTER(C.c_uint64))
            nb = C.c_size_t()
            rc = lib.pg_format_rows_ex(pb.KIND_OLS, C.byref(r), C.byref(lab), 1 if to_csv == 2 else 0, N_POOLS,
                                       fmt_threads, outs[t], cap, C.byref(nb))
            assert rc == 0, rc
            rows[t] += nb.value

        for i in range(n_slabs):
            tk = C.c_int()
            rc = lib.pg_scan_submit_sync_text(sc._h, host[i % 2].ctypes.data, nbytes[i % 2], C.byref(tk), None)
            assert rc == 0, rc
            pending.append((tk.value, i))
            if len(pending) == 3:
                finish(pending.pop(0))
        while pending:
            finish(pending.pop(0))

    def timed(n_slabs, to_csv):
        th = [threading.Thread(target=reader, args=(t, n_slabs, to_csv)) for t in range(n_threads)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    timed(3, 1)
    dt_rec = min(timed(slabs_per_thread, 0) for _ in range(2))
    dt_csv = dt_exact = 1e30
    for _ in range(2):
        rows[:] = [0] * n_threads
        dt_exact = min(dt_exact, timed(slabs_per_thread, 2))
    for _ in range(2):
        rows[:] = [0] * n_threads
        dt_csv = min(dt_csv, timed(slabs_per_thread, 1))
    for sc in scans:
        sc.close()
    ctx.pinned_free(hptr)
    n_loci = slab * slabs_per_thread * n_threads
    text_bytes = sum(nbytes[i % 2] for i in range(slabs_per_thread)) * n_threads
    note = (f"{N_POOLS} pools, slabs of {slab} loci, {n_threads} reader threads x depth-3 pipeline; "
            "pinned sync text -> H2D -> device parse -> ingest -> scan -> D2H records")
    return {"e2e_sync_text": {"loci_per_s": n_loci / dt_rec, "text_bytes_per_locus": nbytes[0] / slab,
                              "text_gb_per_s": text_bytes / dt_rec / 1e9, "note": note},
            "e2e_text_to_csv": {"loci_per_s": n_loci / dt_csv, "text_gb_per_s": text_bytes / dt_csv / 1e9,
                                "csv_bytes": int(sum(rows)), "csv_gb_per_s": sum(rows) / dt_csv / 1e9,
                                "format_threads": fmt_threads * n_threads,
                                "exact_p_loci_per_s": n_loci / dt_exact,
                                "note": note + " -> pg_format_rows (the reference's CSV rows); exact_p = "
                                               "PG_FORMAT_EXACT_P, p re-derived on the host with the reference's arithmetic"}}


FP64_DMMA_PEAK_TFLOPS = 37.1  # tools/fp64_probe.cu on this pool's B200 (profiles/fp64_probe_r1.txt): mma.sync m8n8k4 f64


def dgemm_peak(torch, seconds: float = 2.0):
    """cuBLAS Dgemm 8192^3 (torch.matmul on f64 operands) burst = best of 10, sustained = back to back for `seconds`:
    the FP64 GEMM denominator BASELINE.md 3 names for the kinship Gram matrix, measured in the same process."""
    n = 8192
    a = torch.rand((n, n), dtype=torch.float64, device="cuda")
    b = torch.rand((n, n), dtype=torch.float64, device="cuda")
    c = torch.empty((n, n), dtype=torch.float64, device="cuda")
    flops = 2.0 * n * n * n
    for _ in range(2):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    reps = max(3, int(seconds * 1e3 / best))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b, out=c)
    e1.record()
    e1.synchronize()
    sustained = e0.elapsed_time(e1) / reps
    del a, b, c
    torch.cuda.empty_cache()
    return flops / best / 1e9, flops / sustained / 1e9


def c4_numbers(ctx, pb, dist, rank, world):
    """BASELINE.json configs[3] (C4): ols_iter_with_kinship, 2,000 pools x 5M biallelic loci = 10M allele columns
    (160 GB of f64) column-sharded over 8 GPUs = 1.25M columns (20 GB) per rank: FP64 DMMA Gram matrix, the exchange
    step (pg_kin_allreduce on the library's own NCCL communicator), eigen step, covariate scan."""
    import torch
    from poolgen_b200 import shard
    n, L_rank, k = 2000, 625_000, 1
    kin = pb.Kinship(ctx, n, 2 * L_rank)
    kin.synth(0x5EED0004, rank * L_rank, L_rank)
    P = kin.columns
    kin.gram_time(1)
    gram_ms = kin.gram_time(3) / 3
    comm = shard.make_comm(ctx, dist)      # rank 0's id travels over torch.distributed; the data path is the library's
    kin.gram()
    comm.kin_allreduce([kin])              # communicator warm-up (the first collective sets up the channels)
    kin.gram()
    P_total, ar_ms = comm.kin_allreduce([kin], timed=True)   # the 32 MB exchange step, CUDA events on the kin's stream
    t0 = time.perf_counter()
    m = kin.eig_select(0, 0.75)
    eig_ms = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    kin.eig_select(0, 0.75)
    eig_warm_ms = 1e3 * (time.perf_counter() - t0)
    phen = pb.synth_phen_host(0x5EED0004, n, k)
    kin.covar_scan(phen, 1)
    *_, covar_ms = kin.covar_scan(phen, 5)
    covar_ms /= 5
    # SURVEY H7: the default threshold selects no PC on frequency data; the covariate scan with m = 10 explicit
    # (orthonormalised by the library) covariates shows the X = [1 | PCs | g] case
    rng = np.random.default_rng(0x5EED0004)
    kin.set_covariates(rng.standard_normal((n, 10)))
    kin.covar_scan(phen, 1)
    *_, covar10_ms = kin.covar_scan(phen, 5)
    covar10_ms /= 5
    kin.close()
    comm.close()
    t = torch.tensor([gram_ms, covar_ms, covar10_ms, ar_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gram_ms, covar_ms, covar10_ms, ar_ms = (float(v) for v in t.tolist())
    if rank != 0:
        return {}
    dgemm_burst, dgemm_sustained = dgemm_peak(torch)
    peak, _ = measured_peaks()
    nt = (n + 127) // 128
    hw_flops = 2.0 * (nt * (nt + 1) // 2) * 128 * 128 * P       # the upper triangle of 128 x 128 tiles that is computed
    alg_flops = 2.0 * n * n * P                                  # what g.dot(&g.t()) does (ols.rs:295)
    alg_bytes = (8.0 * n + 24 * k) * P
    fp64_floor_ms = 2.0 * n * 12 * P / (FP64_DMMA_PEAK_TFLOPS * 1e9)   # Q'G with 12 vectors at the FP64 peak
    bound10_ms = max(alg_bytes / (peak * 1e6), fp64_floor_ms)
    return {"c4_kinship": {
        "columns_per_gpu": P, "columns_total": P_total, "n_pools": n, "n_eigenvecs": m,
        "gram_ms": gram_ms, "gram_algorithmic_tflops_per_gpu": alg_flops / gram_ms / 1e9,
        "gram_hardware_tflops_per_gpu": hw_flops / gram_ms / 1e9,
        "gram_frac_of_fp64_tensor_peak": hw_flops / gram_ms / 1e9 / FP64_DMMA_PEAK_TFLOPS,
        "fp64_tensor_peak_tflops": FP64_DMMA_PEAK_TFLOPS,
        "cublas_dgemm_8192_tflops_burst": dgemm_burst, "cublas_dgemm_8192_tflops_sustained": dgemm_sustained,
        "gram_hardware_frac_of_dgemm_sustained": hw_flops / gram_ms / 1e9 / dgemm_sustained,
        "gram_algorithmic_frac_of_dgemm_sustained": alg_flops / gram_ms / 1e9 / dgemm_sustained,
        "allreduce_ms": ar_ms, "allreduce": "pg_kin_allreduce (library NCCL communicator, %d ranks)" % world,
        "eig_select_ms": eig_ms, "eig_select_warm_ms": eig_warm_ms,
        "covar_scan_ms": covar_ms, "covar_columns_per_s": world * P / (covar_ms * 1e-3),
        "covar_roofline_frac": alg_bytes / (covar_ms * 1e-3) / 1e9 / peak,
        "covar_scan_10_covariates_ms": covar10_ms,
        "covar_10_covariates_roofline_frac": alg_bytes / (covar10_ms * 1e-3) / 1e9 / peak,
        "covar_10_covariates_frac_of_min_hbm_fp64": bound10_ms / covar10_ms,
        "note": "symmetric Gram: the algorithmic rate counts 2 n^2 P flops, the hardware rate the DMMA work issued"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--loci-per-gpu", type=int, default=LOCI_PER_GPU)
    ap.add_argument("--e2e-slab", type=int, default=16384)
    ap.add_argument("--e2e-slabs", type=int, default=24)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--c5-loci", type=int, default=50_000_000, help="loci of the C5 leg (BASELINE: 50M)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--cpu-seconds", type=float, default=2.5, help="target seconds per step of the --impl reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs needs --impl cuda: the reference arm times a sample whose size depends on the CPU")
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
