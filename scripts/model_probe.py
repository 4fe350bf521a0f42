"""Genotype counts (k_geno) and Hardy-Weinberg exact tests (k_hwe) on bench.py's workload shape; prints one JSON line.

    python scripts/model_probe.py [windows]

Population: bench.synth_population -- 10 000 + 10 000 samples, genome-wide chromosome mix, `windows` x 32 768 SNP rows
(default 4: 131 072 rows), SNP table resident on the device.
  geno_device      dnaf_genotype_counts_device without the exact tests (k_geno alone)
  geno_hwe_device  the same with the exact tests (k_geno, then k_hwe over the pass's counts)
  assoc_device     dnaf_allele_counts_device (k_assoc)
  bed_device       dnaf_generate_bed_device (k_bed)
                   the four calls alternate call by call until each has >= 1 s of wall time; kernel = event time of
                   the pass kernels; k_hwe = geno_hwe_device - geno_device
  hwe_1e6          the same two geno calls on a population of 10^6 rows, alternated: k_hwe over 3 x 10^6 tests
  cli              pop_factory -s 10000 -c 10000 -x 65536 -f 0.01 -z 2 --gpu_select, with and without --model --hardy
  format           dnaf_format_model / dnaf_format_hardy over 10^7 rows, ten calls of 10^6 (host CPU)
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


def cli(flags, snps=65536):
    d = tempfile.mkdtemp(prefix="dnaf_model_probe_")
    try:
        args = ["-s", str(bench.N_CASES), "-c", str(bench.N_CONTROLS), "-x", str(snps), "-f", str(bench.MIN_MAF), "-z", "2",
                "-p", os.path.join(ROOT, "tests", "golden", "cli_small", "deleterious_config.yml"), "--outdir", d, "--seed",
                "123456", "--gpu_select"] + flags
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            pop_factory.main(args)
        return time.perf_counter() - t0
    finally:
        shutil.rmtree(d, ignore_errors=True)


def engine(R):
    sex, ctl, table, orow, osamp = bench.synth_population(R, 0)
    eng = _native.Engine(0)
    eng.set_samples(sex, ctl)
    eng.set_snps(**table.device_arrays())
    eng.set_overrides(orow, osamp)
    return eng, len(orow)


def alternate(calls, min_s):
    acc = {}
    for name, fn in calls.items():                          # warm-up: module load, buffer sizes
        fn()
        acc[name] = {"calls": 0, "s": 0.0, "event_ms": 0.0, "kernel_ms": 0.0, "launches": 0, "n": 0}
    while min(a["s"] for a in acc.values()) < min_s:
        for name, fn in calls.items():
            t0 = time.perf_counter()
            st = fn()
            a = acc[name]
            a["s"] += time.perf_counter() - t0
            a["calls"] += st["calls"]
            a["event_ms"] += st["ms_total"]
            a["kernel_ms"] += st["ms_sample"]
            a["launches"] += st["kernel_launches"]
            a["n"] += 1
    out = {}
    for name, a in acc.items():
        out[name] = {"calls_per_s_wall": a["calls"] / a["s"], "calls_per_s_event": a["calls"] / (a["event_ms"] * 1e-3),
                     "calls_per_s_kernel": a["calls"] / (a["kernel_ms"] * 1e-3), "kernel_ms_per_call": a["kernel_ms"] / a["n"],
                     "seconds": a["s"], "n_calls": a["n"], "launches_per_call": a["launches"] / a["n"]}
    return out


def main():
    windows = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    R = windows * bench.ROWS_PER_STEP
    seed = bench.PHILOX_SEED
    out = {"gpu": gpu_info(), "shape": {"rows": R, "samples": bench.N_CASES + bench.N_CONTROLS}}
    eng, n_over = engine(R)
    out["shape"]["overrides"] = n_over
    res = alternate({
        "geno_device": lambda: eng.genotype_counts_device(0, R, seed, hwe=False),
        "geno_hwe_device": lambda: eng.genotype_counts_device(0, R, seed, hwe=True),
        "assoc_device": lambda: eng.allele_counts_device(0, R, seed),
        "bed_device": lambda: eng.generate_bed_device(0, R, seed),
    }, 1.0)
    out.update(res)
    out["k_hwe_ms_per_call"] = res["geno_hwe_device"]["kernel_ms_per_call"] - res["geno_device"]["kernel_ms_per_call"]
    counts, p = eng.genotype_counts(0, R, seed)
    out["hwe_p_nan_rows"] = int(np.isnan(p).any(axis=1).sum())
    eng.close()

    big = 10 ** 6
    eng, _ = engine(big)
    res = alternate({"geno_device": lambda: eng.genotype_counts_device(0, big, seed, hwe=False),
                     "geno_hwe_device": lambda: eng.genotype_counts_device(0, big, seed, hwe=True)}, 1.0)
    eng.close()
    out["rows_1e6"] = res
    out["rows_1e6"]["k_hwe_ms_per_call"] = res["geno_hwe_device"]["kernel_ms_per_call"] - res["geno_device"]["kernel_ms_per_call"]

    walls = {False: [], True: []}
    for _ in range(2):
        for flag in (False, True):
            walls[flag].append(cli(["--model", "--hardy"] if flag else []))
    out["cli_65536_snps"] = {"wall_s_vcf_only": min(walls[False]), "wall_s_with_model_hardy": min(walls[True]),
                             "runs": {"vcf_only": walls[False], "with_model_hardy": walls[True]}}

    rows = 10 ** 7
    np.random.seed(1)
    t = snp.SnpFactory.init_from_cdf_file().random_snp_table(rows, min_maf=0.01, vector_alt=True).sorted()
    cnt = np.tile(counts, (rows // len(counts) + 1, 1))[:rows]
    pp = np.tile(p, (rows // len(p) + 1, 1))[:rows]
    fmt = {"model": {"seconds": 0.0, "bytes": 0}, "hardy": {"seconds": 0.0, "bytes": 0}}
    step = 10 ** 6          # ten calls of 10^6 rows: one call's output buffer would be 9.6 GB
    for r0 in range(0, rows, step):
        s = slice(r0, r0 + step)
        cols = (t.ids[s], t.chrom_idx[s], t.chrom_labels, t.n_alleles[s], t.nts[s])
        t0 = time.perf_counter()
        n = len(_native.format_model(*cols, cnt[s]))
        fmt["model"]["seconds"] += time.perf_counter() - t0
        fmt["model"]["bytes"] += n
        t0 = time.perf_counter()
        n = len(_native.format_hardy(*cols, cnt[s], pp[s]))
        fmt["hardy"]["seconds"] += time.perf_counter() - t0
        fmt["hardy"]["bytes"] += n
    out["format_1e7_rows"] = fmt
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
