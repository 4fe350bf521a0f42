"""Fisher's exact tests (k_fisher) beside the genotype counts (k_geno) on bench.py's workload shape; prints one JSON line.

    python scripts/fisher_probe.py [windows]

Population: bench.synth_population -- 10 000 + 10 000 samples, genome-wide chromosome mix, `windows` x 32 768 SNP rows
(default 4: 131 072 rows), SNP table resident on the device.
  geno               dnaf_genotype_tests_device without exact tests (k_geno alone)
  geno_fisher        the same with the Fisher tests (k_geno, then k_fisher over the pass's counts)
  geno_hwe_fisher    the same with the Hardy-Weinberg and the Fisher tests (k_geno, k_hwe, k_fisher)
                     the three calls alternate call by call until each has >= 1 s of wall time; kernel = event time of
                     the pass kernels; k_fisher = geno_fisher - geno
  split              dnaf_fisher_exact over the GENO tables alone and over the three 2x2 tables (ALLELIC, DOM, REC) alone
                     of the same rows: wall time of the synchronous call, upload and download included
  rows_1e6           geno / geno_fisher / geno_hwe_fisher on a population of 10^6 rows, alternated
  cli                pop_factory -s 10000 -c 10000 -x 65536 -f 0.01 -z 2 --gpu_select, with and without --fisher
  format             dnaf_format_assoc_fisher / dnaf_format_model_fisher over 10^6 rows (host CPU)
No fallback: without a GPU the Engine raises.
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from dna_factory_b200 import _native, snp  # noqa: E402
from scripts.bed_probe import gpu_info  # noqa: E402
from scripts.model_probe import alternate, cli, engine  # noqa: E402


def tables(counts):
    """[rows][4][6] Fisher tables (GENO, ALLELIC, DOM, REC) of [rows][10] counts, as k_fisher builds them."""
    c = np.asarray(counts, np.int64)
    a11, a12, a22 = c[:, 2], c[:, 1], c[:, 0] - c[:, 1] - c[:, 2]
    u11, u12, u22 = c[:, 7], c[:, 6], c[:, 5] - c[:, 6] - c[:, 7]
    alt_a, alt_u = 2 * a11 + a12 + c[:, 4], 2 * u11 + u12 + c[:, 9]
    z = np.zeros_like(a11)
    t = [(a11, a12, a22, u11, u12, u22), (alt_a, 2 * c[:, 0] + c[:, 3] - alt_a, z, alt_u, 2 * c[:, 5] + c[:, 8] - alt_u, z),
         (a11 + a12, a22, z, u11 + u12, u22, z), (a11, a12 + a22, z, u11, u12 + u22, z)]
    return np.stack([np.stack(q, 1) for q in t], 1).astype(np.uint32)


def three_calls(eng, R, seed):
    res = alternate({
        "geno": lambda: eng.genotype_tests_device(0, R, seed, hwe=False, fisher=False),
        "geno_fisher": lambda: eng.genotype_tests_device(0, R, seed, hwe=False, fisher=True),
        "geno_hwe_fisher": lambda: eng.genotype_tests_device(0, R, seed, hwe=True, fisher=True),
    }, 1.0)
    res["k_fisher_ms_per_call"] = res["geno_fisher"]["kernel_ms_per_call"] - res["geno"]["kernel_ms_per_call"]
    return res


def main():
    windows = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    R = windows * bench.ROWS_PER_STEP
    seed = bench.PHILOX_SEED
    out = {"gpu": gpu_info(), "shape": {"rows": R, "samples": bench.N_CASES + bench.N_CONTROLS}}
    eng, n_over = engine(R)
    out["shape"]["overrides"] = n_over
    out.update(three_calls(eng, R, seed))
    counts, _, l = eng.genotype_tests(0, R, seed, hwe=False)
    out["nan_tests"] = {t: int(np.isnan(l[:, j]).sum()) for j, t in enumerate(("GENO", "ALLELIC", "DOM", "REC"))}
    out["p_below_0.05"] = {t: int((l[:, j] < np.log10(0.05)).sum()) for j, t in enumerate(("GENO", "ALLELIC", "DOM", "REC"))}
    tabs = tables(counts)
    split = {}
    for name, sel in (("geno", tabs[:, 0]), ("2x2", tabs[:, 1:].reshape(-1, 6))):
        eng.fisher_exact(sel)                                # warm-up
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            got = eng.fisher_exact(sel)
            ts.append(time.perf_counter() - t0)
        split[name] = {"tests": len(sel), "wall_ms_min": 1e3 * min(ts), "wall_ms": [1e3 * t for t in ts]}
        split[name]["bitwise_equal_to_the_pass"] = bool(np.array_equal(
            got.reshape(len(counts), -1), l[:, :1] if name == "geno" else l[:, 1:], equal_nan=True))
    out["split"] = split
    eng.close()

    big = 10 ** 6
    eng, _ = engine(big)
    out["rows_1e6"] = three_calls(eng, big, seed)
    eng.close()

    walls = {False: [], True: []}
    for _ in range(2):
        for flag in (False, True):
            walls[flag].append(cli(["--fisher"] if flag else []))
    out["cli_65536_snps"] = {"wall_s_vcf_only": min(walls[False]), "wall_s_with_fisher": min(walls[True]),
                             "runs": {"vcf_only": walls[False], "with_fisher": walls[True]}}

    rows = 10 ** 6
    np.random.seed(1)
    t = snp.SnpFactory.init_from_cdf_file().random_snp_table(rows, min_maf=0.01, vector_alt=True).sorted()
    cnt = np.tile(counts, (rows // len(counts) + 1, 1))[:rows]
    ll = np.tile(l, (rows // len(l) + 1, 1))[:rows]
    cols = (t.ids, t.chrom_idx, t.chrom_labels)
    fmt = {}
    t0 = time.perf_counter()
    n = len(_native.format_assoc_fisher(*cols, t.position, t.n_alleles, t.nts, cnt, ll))
    fmt["assoc_fisher"] = {"seconds": time.perf_counter() - t0, "bytes": n}
    t0 = time.perf_counter()
    n = len(_native.format_model_fisher(*cols, t.n_alleles, t.nts, cnt, ll))
    fmt["model_fisher"] = {"seconds": time.perf_counter() - t0, "bytes": n}
    out["format_1e6_rows"] = fmt
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
