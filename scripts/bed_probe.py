"""PLINK 1 .bed writer (k_bed, dnaf_generate_bed*) on bench.py's workload shape; prints one JSON line.

    python scripts/bed_probe.py [windows]

Population: bench.synth_population -- 10 000 + 10 000 samples, genome-wide chromosome mix, `windows` x 32 768 SNP rows
(default 4: 131 072 rows, 655 MB of .bed per call, larger than the 126 MB L2), SNP table resident on the device.
  bed_device     dnaf_generate_bed_device over all rows, wall time of the (synchronous) call; kernel = k_bed event time
  vcf_device     dnaf_generate_device at -z 2 over the same rows, alternated call by call with bed_device
  bed_e2e        dnaf_generate_bed into a page-locked host buffer
  cli            pop_factory -s 10000 -c 10000 -x 65536 -f 0.01 -z 2 --gpu_select, with and without --bed, alternated
  bim_1e7        SnpTable.bim_bytes() on a 10^7-row table (host CPU)
Every device figure repeats until >= 1 s of work has been timed.  No fallback: without a GPU the Engine raises.
"""
import contextlib
import io
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from dna_factory_b200 import _native, pop_factory, snp  # noqa: E402


def gpu_info():
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(0)
    name = nv.nvmlDeviceGetName(h)
    return {"name": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0,
            "sm_max_mhz": nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)}


def timed(fn, min_s=1.0):
    """Calls fn() until min_s seconds have been spent in it; -> (calls, seconds, last stats)."""
    calls, spent, st = 0, 0.0, None
    while spent < min_s:
        t0 = time.perf_counter()
        st = fn()
        spent += time.perf_counter() - t0
        calls += st["calls"]
    return calls, spent, st


def cli(bed, snps=65536):
    d = tempfile.mkdtemp(prefix="dnaf_bed_probe_")
    try:
        args = ["-s", str(bench.N_CASES), "-c", str(bench.N_CONTROLS), "-x", str(snps), "-f", str(bench.MIN_MAF), "-z", "2",
                "-p", os.path.join(ROOT, "tests", "golden", "cli_small", "deleterious_config.yml"), "--outdir", d, "--seed",
                "123456", "--gpu_select"] + (["--bed"] if bed else [])
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            pop_factory.main(args)
        wall = time.perf_counter() - t0
        return wall
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    import torch
    windows = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    R = windows * bench.ROWS_PER_STEP
    n = bench.N_CASES + bench.N_CONTROLS
    sex, ctl, table, orow, osamp = bench.synth_population(R, 0)
    eng = _native.Engine(0)
    eng.set_samples(sex, ctl)
    eng.set_snps(**table.device_arrays())
    eng.set_overrides(orow, osamp)
    seed = bench.PHILOX_SEED
    eng.generate_bed_device(0, R, seed)                      # warm-up: module load, buffer sizes
    eng.generate_device(0, R, seed, level=2)                 # warm-up: code tables
    bed = {"calls": 0, "s": 0.0, "kernel_ms": 0.0, "launches": 0}
    vcf = {"calls": 0, "s": 0.0}
    while bed["s"] < 1.0 or vcf["s"] < 1.0:                  # alternate the two calls
        t0 = time.perf_counter()
        st = eng.generate_bed_device(0, R, seed)
        bed["s"] += time.perf_counter() - t0
        bed["calls"] += st["calls"]
        bed["kernel_ms"] += st["ms_sample"]
        bed["launches"] += st["kernel_launches"]
        t0 = time.perf_counter()
        st = eng.generate_device(0, R, seed, level=2)
        vcf["s"] += time.perf_counter() - t0
        vcf["calls"] += st["calls"]
    bed_bytes = bed["calls"] // n * eng.bed_pitch()          # .bed bytes written by the timed calls
    n_bed_calls = bed["calls"] // (n * R)
    pinned = torch.empty(R * eng.bed_pitch(), dtype=torch.uint8, pin_memory=True).numpy()
    eng.generate_bed_into(0, R, seed, pinned)
    e2e_calls, e2e_s, _ = timed(lambda: eng.generate_bed_into(0, R, seed, pinned))
    eng.close()
    walls = {False: [], True: []}
    for _ in range(2):
        for flag in (False, True):
            walls[flag].append(cli(flag))
    np.random.seed(1)
    big = snp.SnpFactory.init_from_cdf_file().random_snp_table(10_000_000, min_maf=0.01, vector_alt=True).sorted()
    t0 = time.perf_counter()
    bim = big.bim_bytes()
    bim_s = time.perf_counter() - t0
    out = {
        "gpu": gpu_info(),
        "shape": {"rows": R, "samples": n, "bed_bytes_per_call": R * ((n + 3) // 4), "overrides": int(len(orow))},
        "bed_device": {"calls_per_s": bed["calls"] / bed["s"], "seconds": bed["s"],
                       "kernel_calls_per_s": bed["calls"] / (bed["kernel_ms"] * 1e-3),
                       "kernel_output_gb_per_s": bed_bytes / (bed["kernel_ms"] * 1e-3) / 1e9,
                       "launches_per_call": bed["launches"] / n_bed_calls},
        "vcf_device_z2": {"calls_per_s": vcf["calls"] / vcf["s"], "seconds": vcf["s"]},
        "bed_e2e_pinned": {"calls_per_s": e2e_calls / e2e_s, "seconds": e2e_s},
        "cli_65536_snps": {"wall_s_vcf_only": min(walls[False]), "wall_s_with_bed": min(walls[True]),
                           "runs": {"vcf_only": walls[False], "with_bed": walls[True]}},
        "bim_bytes_1e7_rows": {"seconds": bim_s, "bytes": len(bim)},
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
