"""bench.py's output: the reference arm's JSON line (CPU only), the committed bench lines and --dump-outputs."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-seconds", "0.5"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "loci/s" and d["higher_is_better"] is True
    assert d["metric"] == "loci/sec for ols_iter (f64)" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "loci/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    # the reference arm never maps the product library (its inputs come from libpoolgen_synth.so) and reports the
    # "tight" CPU variant next to the faithful one
    assert d["maps_product_library"] is False
    assert d["cpu_baseline"]["tight"]["value"] > d["value"]


def test_traffic_is_read_from_the_committed_capture():
    """roofline.traffic comes from profiles/ncu_raw_r*.csv at run time (dram__bytes_read + dram__bytes_write of the
    streaming kernel and the fix-up kernel), not from a constant"""
    sys.path.insert(0, ROOT)
    import bench
    per_locus, src = bench.traffic_from_profile(1000, 4, 3)
    assert src and src.startswith("profiles/ncu_raw_r")
    assert 32288 <= per_locus <= 1.2 * 32288          # at least the algorithmic bytes, no wasted re-reads
    assert bench.traffic_from_profile(7, 7, 7) == (None, None)


def test_dump_sample_is_seeded_and_fits_the_budget():
    """--dump-outputs keeps a fixed sample of the C3 shard's records (1.25 M loci, 3 slots, 3 phenotypes), all in f64,
    under 64 MB for one rank and for eight; of freq_mean and stats only the output rows (the library leaves the other
    slots NaN)"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from poolgen_b200.capi import LOCUS_FILTERED, LOCUS_OK, ScanResults
    L, S, k = bench.LOCI_PER_GPU, bench.N_ALLELES - 1, bench.N_PHEN
    rng = np.random.default_rng(1)
    status = np.where(rng.random(L) < 0.9, LOCUS_OK, LOCUS_FILTERED).astype(np.uint8)
    n_out = np.where(status == LOCUS_OK, rng.integers(1, S + 1, L), 0).astype(np.uint8)
    rows = (status == LOCUS_OK)[:, None] & (np.arange(S)[None, :] < n_out[:, None])
    fm = np.where(rows, np.arange(L * S, dtype=np.float64).reshape(L, S), np.nan)
    st = np.where(rows[:, :, None, None], rng.random((L, S, k, 4)), np.nan)
    res = ScanResults(status, n_out, np.zeros((L, 6), np.uint8), fm, st)
    for world in (1, 8):
        a = bench.sample_records(res, 5 * L, world)
        b = bench.sample_records(res, 5 * L, world)
        assert a.keys() == b.keys() and all(np.array_equal(a[n], b[n]) for n in a)
        assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in a.values())
        assert world * sum(v.nbytes for v in a.values()) <= 64e6 - 4096
        n = a["locus"].size
        assert n > 10_000 and (np.diff(a["locus"]) > 0).all() and a["locus"][0] >= 5 * L
        idx = a["locus"].astype(np.int64) - 5 * L
        assert np.array_equal(a["status"], status[idx]) and np.array_equal(a["n_out"], n_out[idx])
        assert np.array_equal(a["freq_mean"], fm[idx][rows[idx]]) and np.array_equal(a["stats"], st[idx][rows[idx]])
        assert a["stats"].shape == (int(a["n_out"].sum()), k, 4)
    small = ScanResults(status[:100], n_out[:100], res.alleles[:100], fm[:100], st[:100])
    assert np.array_equal(bench.sample_records(small, 0, 1)["locus"], np.arange(100))


@pytest.mark.gpu
def test_dump_outputs_are_the_records_of_the_timed_scan(ctx, tmp_path):
    """bench.py --dump-outputs writes the records a caller of the timed ols_iter scan receives for the sampled loci: all of
    status, n_out and alleles, and the output rows of freq_mean and stats, every value finite"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    import poolgen_b200 as pb
    L = 20_000
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0",
                          "--loci-per-gpu", str(L), "--no-extras", "--no-cpu", "--dump-outputs", str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("locus", "status", "n_out", "alleles", "freq_mean", "stats")}
    assert np.array_equal(got["locus"], np.arange(L))
    scan = pb.Scan(ctx, pb.KIND_OLS, pb.FilterStats(pool_sizes=np.full(bench.N_POOLS, 1.0 / bench.N_POOLS)),
                   bench.N_POOLS, np.arange(bench.N_ALLELES, dtype=np.uint8),
                   pb.synth_phen_host(bench.SEED, bench.N_POOLS, bench.N_PHEN))
    b = scan.batch(L)
    b.synth(bench.SEED, 0, L)
    b.run()
    want = b.fetch()
    b.close()
    scan.close()
    assert all(np.isfinite(v).all() for v in got.values())
    for n in ("status", "n_out", "alleles"):
        assert np.array_equal(got[n], getattr(want, n).astype(np.float64)), n
    rows = (want.status == pb.LOCUS_OK)[:, None] & (np.arange(want.freq_mean.shape[1])[None, :] < want.n_out[:, None])
    assert rows.sum() > 0.8 * L
    assert np.array_equal(got["freq_mean"], want.freq_mean[rows]) and np.array_equal(got["stats"], want.stats[rows])


def test_committed_bench_lines_follow_the_contract():
    """profiles/bench_*_r2.json (what bench.py printed on the GPU boxes): one JSON line each with the driver's keys, the
    roofline / cpu_baseline / e2e objects and the per-config summaries at the top level"""
    import glob
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = sorted(glob.glob(os.path.join(root, "profiles", "bench_*gpu_r2.json")))
    assert len(files) >= 3
    for f in files:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                    "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "c4"):
            assert key in d, (f, key)
        assert d["unit"] == "loci/s" and d["higher_is_better"] is True and d["scaling"] == "weak" and d["dtype"] == "f64"
        assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and "workload" in d["config"] and "model" not in d["config"]
        r = d["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
        assert r["traffic_source"].startswith("profiles/ncu_raw_r")
        e = d["e2e"]
        assert e["unit"] == "loci/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if d["n_gpus"] == 1:
            cb = d["cpu_baseline"]
            assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "tight" in cb
            for key in ("c2", "c5", "text", "nelder_mead"):
                assert key in d, (f, key)
