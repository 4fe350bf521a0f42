"""max(T) permutation tests (k_perm_masks, k_mperm_planes, k_mperm) beside the genotype counts (k_geno) on bench.py's
workload shape; prints one JSON line.

    python scripts/mperm_probe.py [windows]

Population: bench.synth_population -- 10 000 + 10 000 samples, genome-wide chromosome mix, `windows` x 32 768 SNP rows
(default 4: 131 072 rows), SNP table resident on the device.
  geno, mperm_<P>  dnaf_genotype_tests_device without exact tests (k_geno alone) and dnaf_mperm_device at P = 100,
                   1 000 and 10 000 permutations, alternated call by call until each has >= 1 s of wall time; kernel =
                   event time of the pass kernels (k_perm_masks included)
  kernels          torch.profiler (CUDA activity) over one call of each: device time per kernel name, and k_mperm's rate
                   in row x permutation x sample tests per second (rows x P x N / k_mperm time)
  cli              pop_factory -s 10000 -c 10000 -x 65536 -f 0.01 -z 2 --gpu_select, with and without --mperm 1000
The card's name, power limit and maximum SM clock are read before, and the SM clock after the timed calls.
No fallback: without a GPU the Engine raises.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from scripts.bed_probe import gpu_info  # noqa: E402
from scripts.model_probe import alternate, cli, engine  # noqa: E402

PERMS = (100, 1000, 10000)


def sm_clock_mhz():
    import pynvml as nv
    nv.nvmlInit()
    return nv.nvmlDeviceGetClockInfo(nv.nvmlDeviceGetHandleByIndex(0), nv.NVML_CLOCK_SM)


def kernel_times(fn):
    """{kernel name: device ms} of one fn() under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        if us > 0:
            out[e.key] = out.get(e.key, 0.0) + us * 1e-3
    return out


def main():
    windows = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    R = windows * bench.ROWS_PER_STEP
    N = bench.N_CASES + bench.N_CONTROLS
    seed = bench.PHILOX_SEED
    out = {"gpu": gpu_info(), "shape": {"rows": R, "samples": N}}
    eng, n_over = engine(R)
    out["shape"]["overrides"] = n_over
    calls = {"geno": lambda: eng.genotype_tests_device(0, R, seed, hwe=False, fisher=False)}
    for P in PERMS:
        calls["mperm_%d" % P] = (lambda P=P: eng.mperm_device(0, R, seed, P))
    out.update(alternate(calls, 1.0))
    out["sm_clock_mhz_after"] = sm_clock_mhz()
    ker = {}
    for P in PERMS:
        k = kernel_times(lambda P=P: eng.mperm_device(0, R, seed, P))
        short = {}
        for name, ms in k.items():
            for tag in ("k_perm_masks", "k_mperm_planes", "k_mperm(", "k_geno"):
                if tag in name:
                    short[tag.rstrip("(")] = short.get(tag.rstrip("("), 0.0) + ms
        short["k_mperm_tests_per_s"] = R * P * N / (short["k_mperm"] * 1e-3)
        ker[str(P)] = short
    out["kernels"] = ker
    eng.close()
    walls = {False: [], True: []}
    for _ in range(2):
        for flag in (False, True):
            walls[flag].append(cli(["--mperm", "1000"] if flag else []))
    out["cli_65536_snps"] = {"wall_s_vcf_only": min(walls[False]), "wall_s_with_mperm_1000": min(walls[True]),
                             "runs": {"vcf_only": walls[False], "with_mperm_1000": walls[True]}}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
