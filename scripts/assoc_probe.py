"""Case/control allele counts (k_assoc, dnaf_allele_counts*) on bench.py's workload shape; prints one JSON line.

    python scripts/assoc_probe.py [windows]

Population: bench.synth_population -- 10 000 + 10 000 samples, genome-wide chromosome mix, `windows` x 32 768 SNP rows
(default 4: 131 072 rows), SNP table resident on the device.
  assoc_device   dnaf_allele_counts_device over all rows; wall time of the (synchronous) call, kernel = k_assoc event time
  bed_device     dnaf_generate_bed_device over the same rows
  vcf_device_z2  dnaf_generate_device at -z 2 over the same rows
                 the three calls alternate call by call until each has >= 1 s of wall time
  cli            pop_factory -s 10000 -c 10000 -x 65536 -f 0.01 -z 2 --gpu_select, with and without --assoc, alternated
  format_assoc   dnaf_format_assoc over 10^6 and 10^7 rows (host CPU)
No fallback: without a GPU the Engine raises.
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
from scripts.bed_probe import gpu_info  # noqa: E402


def cli(flag, snps=65536):
    d = tempfile.mkdtemp(prefix="dnaf_assoc_probe_")
    try:
        args = ["-s", str(bench.N_CASES), "-c", str(bench.N_CONTROLS), "-x", str(snps), "-f", str(bench.MIN_MAF), "-z", "2",
                "-p", os.path.join(ROOT, "tests", "golden", "cli_small", "deleterious_config.yml"), "--outdir", d, "--seed",
                "123456", "--gpu_select"] + (["--assoc"] if flag else [])
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            pop_factory.main(args)
        return time.perf_counter() - t0
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    windows = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    R = windows * bench.ROWS_PER_STEP
    n = bench.N_CASES + bench.N_CONTROLS
    sex, ctl, table, orow, osamp = bench.synth_population(R, 0)
    eng = _native.Engine(0)
    eng.set_samples(sex, ctl)
    eng.set_snps(**table.device_arrays())
    eng.set_overrides(orow, osamp)
    seed = bench.PHILOX_SEED
    calls = {
        "assoc_device": lambda: eng.allele_counts_device(0, R, seed),
        "bed_device": lambda: eng.generate_bed_device(0, R, seed),
        "vcf_device_z2": lambda: eng.generate_device(0, R, seed, level=2),
    }
    acc = {}
    for name, fn in calls.items():                          # warm-up: module load, buffer sizes, code tables
        fn()
        acc[name] = {"calls": 0, "s": 0.0, "event_ms": 0.0, "launches": 0, "n": 0}
    while min(a["s"] for a in acc.values()) < 1.0:           # alternate the three calls
        for name, fn in calls.items():
            t0 = time.perf_counter()
            st = fn()
            a = acc[name]
            a["s"] += time.perf_counter() - t0
            a["calls"] += st["calls"]
            a["event_ms"] += st["ms_total"]
            a["launches"] += st["kernel_launches"]
            a["n"] += 1
            if name != "vcf_device_z2":
                a.setdefault("kernel_ms", 0.0)
                a["kernel_ms"] += st["ms_sample"]
    counts = eng.allele_counts(0, R, seed)
    eng.close()
    walls = {False: [], True: []}
    for _ in range(2):
        for flag in (False, True):
            walls[flag].append(cli(flag))
    fmt = {}
    np.random.seed(1)
    for rows in (10 ** 6, 10 ** 7):
        big = snp.SnpFactory.init_from_cdf_file().random_snp_table(rows, min_maf=0.01, vector_alt=True).sorted()
        cnt = np.tile(counts, (rows // len(counts) + 1, 1))[:rows]
        t0 = time.perf_counter()
        text = _native.format_assoc(big.ids, big.chrom_idx, big.chrom_labels, big.position, big.n_alleles, big.nts, cnt)
        fmt["rows_%d" % rows] = {"seconds": time.perf_counter() - t0, "bytes": len(text)}
    out = {"gpu": gpu_info(), "shape": {"rows": R, "samples": n, "overrides": int(len(orow))}}
    for name, a in acc.items():
        rec = {"calls_per_s_wall": a["calls"] / a["s"], "calls_per_s_event": a["calls"] / (a["event_ms"] * 1e-3),
               "seconds": a["s"], "n_calls": a["n"], "launches_per_call": a["launches"] / a["n"]}
        if "kernel_ms" in a:
            rec["calls_per_s_kernel"] = a["calls"] / (a["kernel_ms"] * 1e-3)
        out[name] = rec
    out["cli_65536_snps"] = {"wall_s_vcf_only": min(walls[False]), "wall_s_with_assoc": min(walls[True]),
                             "runs": {"vcf_only": walls[False], "with_assoc": walls[True]}}
    out["format_assoc"] = fmt
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
