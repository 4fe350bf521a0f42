#!/usr/bin/env python
"""Benchmark of the population-generation hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload: BASELINE.json configs[1] (README 8-core scenario): 10 000 cases + 10 000 controls, -f 0.01,
-z 2, SNPs drawn like SnpFactory (MAF from the RefSNP CDF, chromosomes by CHROMOSOME_PROB, sorted by
(chromosome string, position)).  One "step" = one batch of ROWS_PER_STEP consecutive SNP rows of that
5 000 000-row population through the hot path: allele draws -> VCF text -> BGZF blocks.  Every step uses
a new row window (and every rank its own contiguous SNP range), so inputs never repeat.

  value   calls/s with the SNP table already resident in HBM and the BGZF stream left in HBM
          (dnaf_generate_device), timed with CUDA events on the stream the kernels run on
  e2e     calls/s through the public API with HOST buffers: every step uploads that step's SNP metadata
          (H2D) and receives the BGZF bytes in host memory (D2H) inside the timed region
  roofline / cpu_baseline: see DESIGN.md section 6
Extra keys of the N = 1 line: value_sustained (>= 1 s of back-to-back device-only calls), level_sweep (-z 1..9: ratio,
value, e2e on the C5 sample shape), cli_to_file (the drop-in CLI writing population.vcf.gz), allele_chi_square
(dna_factory_b200/allele_stats.py), cpu_baseline (the UNMODIFIED reference CLI from oracle/_ref, `-n <cores-1>`),
cpu_baseline_c1_full (BASELINE config 1 in full) and cpu_baseline_port (the C port).  N > 1: multi_gpu_parity.
--dump-outputs DIR: rank 0 writes what the last timed step of `value` and of `e2e` returned to DIR/*.npy (dump_outputs).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CASES = 10000
N_CONTROLS = 10000
TOTAL_SNPS = 5_000_000
MIN_MAF = 0.01
LEVEL = 2
MALE_ODDS = 0.5
ROWS_PER_STEP = 32768
PHILOX_SEED = 0x5EED000000000001
HOST_SEED = 20260101
E2E_CHUNK = 1024 << 20   # the library default: passes ramp 1/4, 1/2 of it at the start of a call (1/2 for device-only calls), then whole chunks
WORKLOAD = ("C2 pop_factory -s 10000 -c 10000 -x 5000000 -f 0.01 -z 2: one step = %d consecutive SNP rows "
            "x 20000 samples (sample -> VCF GT text -> BGZF)" % ROWS_PER_STEP)


def synth_population(n_rows, rank=0, window=ROWS_PER_STEP):
    """Sex vector, control flags and `n_rows` sorted SNP rows shaped like the reference's own generator."""
    from dna_factory_b200 import snp
    rs_state = np.random.get_state()
    np.random.seed(HOST_SEED + rank)
    n = N_CASES + N_CONTROLS
    sex = np.where(np.random.rand(n) <= MALE_ODDS, 1, 2).astype(np.uint8)       # pop_factory.py:352,365
    ctl = (np.arange(n) < N_CONTROLS).astype(np.uint8)                          # pop_factory.py:358
    # every step's row window is its own sorted draw from the genome-wide distribution, so each step sees the
    # whole-job chromosome mix (about 4.8 % X and 0.25 % Y rows) instead of ROWS_PER_STEP rows of chromosome 1
    fac = snp.SnpFactory.init_from_cdf_file()
    wins, orows, osamps = [], [], []
    for w0 in range(0, n_rows, window):
        wn = min(window, n_rows - w0)
        t = fac.random_snp_table(wn, min_maf=MIN_MAF, vector_alt=True).sorted()
        t.ids = t.ids + w0
        wins.append(t)
        # polygenic overrides: ~6 deleterious SNPs per case over the whole job, as deleterious.yml's groups produce;
        # drawn window by window, so that a window's forced cells do not depend on how many windows follow it
        n_over = 6 * N_CASES * wn // TOTAL_SNPS + 2
        orows.append(np.sort(np.random.randint(w0, w0 + wn, n_over)).astype(np.uint64))
        osamps.append(np.random.randint(N_CONTROLS, n, n_over).astype(np.uint32))
    table = snp.SnpTable.concat(wins)
    orow, osamp = np.concatenate(orows), np.concatenate(osamps)
    np.random.set_state(rs_state)
    return sex, ctl, table, orow, osamp


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU; started before the warm-up so that NVML is up when the
    timed region begins, reports the samples that fall inside [mark_begin, mark_end]."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []          # (time, sm_mhz, reason bits)
        self.max_mhz = None
        self.error = None
        self.t0 = self.t1 = None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), r))
                time.sleep(0.005)
        except Exception as e:  # noqa: clocks are reported as unknown, never fatal
            self.error = "unavailable:%s" % type(e).__name__

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        inside = [x for x in self.samples if self.t0 is not None and self.t0 <= x[0] <= self.t1]
        if not inside and self.samples and self.t0 is not None:   # region shorter than the poll interval
            inside = [min(self.samples, key=lambda x: abs(x[0] - 0.5 * (self.t0 + self.t1)))]
        reasons = sorted({k for x in inside for k, bit in names.items() if x[2] & bit})
        if self.error:
            reasons.append(self.error)
        return {"sm_mhz": float(np.median([x[1] for x in inside])) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside)}


def cpu_reference_run(steps, warmup, budget_s=20.0):
    """The reference's path on host cores: C port of the row loop + zlib BGZF (oracle/), all host threads.
    Each step is a bounded sample of the workload (same sample count and level, fewer SNP rows)."""
    from oracle import oracle
    oracle.build()
    # every host thread the box offers, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    rows = 512   # 6 timed steps = 6.1e7 calls: about 1 s of wall clock, ~15 s of CPU time on 16 threads
    sex, ctl, table, orow, osamp = synth_population(rows * (steps + warmup), window=rows)
    snps_all = table.to_snps()
    from types import SimpleNamespace
    fam = [SimpleNamespace(sex=int(s), is_control=bool(c), deleterious_snps=None if c else {}, person_id=i) for i, (s, c) in
           enumerate(zip(sex, ctl))]
    flat_batches = []
    for k in range(steps + warmup):
        flat = oracle.flatten(fam, snps_all[k * rows:(k + 1) * rows])
        sel = (orow >= k * rows) & (orow < (k + 1) * rows)
        flat["over_row"] = (orow[sel] - k * rows).astype(np.uint64)
        flat["over_sample"] = osamp[sel]
        flat_batches.append(flat)
    times = []
    text_bytes = 0
    comp_bytes = 0
    for k, flat in enumerate(flat_batches):
        t0 = time.perf_counter()
        text, _ = oracle.rows_from_flat(flat, PHILOX_SEED, k * rows, n_threads=cores)
        blob = oracle.bgzf(text.tobytes(), level=LEVEL, with_eof=False, n_threads=cores)
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
            text_bytes += len(text)
            comp_bytes += len(blob)
    calls = rows * (N_CASES + N_CONTROLS) * len(times)
    total = sum(times)
    return {"value": calls / total, "ms_per_step": 1e3 * total / len(times), "cores": cores,
            "sample": "%d steps x %d SNP rows x %d samples, -z %d (C port of pop_factory.py:471-513 + zlib BGZF, "
                      "OpenMP over rows and blocks)" % (len(times), rows, N_CASES + N_CONTROLS, LEVEL),
            "text_bytes": text_bytes, "bgzf_bytes": comp_bytes}


def _inflate_bgzf(blob):
    """Decompressed bytes of a BGZF stream without EOF block (zlib, block by block, CRC32 / ISIZE checked)."""
    from dna_factory_b200 import allele_stats
    return allele_stats.inflate_bgzf(blob)


DUMP_STATS = ("rows", "calls", "text_bytes", "bgzf_bytes", "bgzf_blocks", "crc_xor")
DUMP_SEED = 20260101
DUMP_WINDOW = 1 << 16


def _sample_windows(n_bytes, n, rng):
    """Sorted offsets of n windows of min(DUMP_WINDOW, n_bytes) bytes inside n_bytes bytes, and that width."""
    width = min(DUMP_WINDOW, n_bytes)
    return np.sort(rng.integers(0, n_bytes - width + 1, n)), width


def dump_outputs(out_dir, value_stats, e2e_stats, blob):
    """What the last timed step handed its caller, as .npy files for comparing two builds output for output (~50 MB).

    value_stats / e2e_stats   float64[6]: rows, calls, text_bytes, bgzf_bytes, bgzf_blocks, crc_xor of the last step
                              of the `value` pass (dnaf_generate_device returns nothing else) and of the `e2e` pass
    e2e_bgzf_blocks           float32[blocks, 2]: compressed and text size of every BGZF block of the e2e step's stream
    e2e_bgzf, e2e_text        float32[windows, 64 KiB]: bytes of that stream and of its decompressed VCF text in
                              windows at seeded offsets (e2e_bgzf_offsets, e2e_text_offsets: float64)
    The text is inflated only around the windows; every block inflated is checked against its CRC32 and ISIZE.
    """
    from dna_factory_b200 import _native, allele_stats
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    csize, usize = _native.bgzf_scan(blob)
    coff = np.concatenate(([0], np.cumsum(csize, dtype=np.int64)))
    uoff = np.concatenate(([0], np.cumsum(usize, dtype=np.int64)))
    b_off, b_w = _sample_windows(len(blob), 64, rng)
    t_off, t_w = _sample_windows(int(uoff[-1]), 128, rng)
    text = []
    for o in t_off:
        b0, b1 = np.searchsorted(uoff, o, "right") - 1, np.searchsorted(uoff, o + t_w, "left")
        t = allele_stats.inflate_bgzf(blob[coff[b0]:coff[max(b0 + 1, b1)]])
        text.append(np.frombuffer(t, np.uint8)[o - uoff[b0]:o - uoff[b0] + t_w])
    arrays = {"value_stats": np.array([value_stats[k] for k in DUMP_STATS], np.float64),
              "e2e_stats": np.array([e2e_stats[k] for k in DUMP_STATS], np.float64),
              "e2e_bgzf_blocks": np.stack([csize, usize], axis=1).astype(np.float32),
              "e2e_bgzf_offsets": b_off.astype(np.float64),
              "e2e_bgzf": np.stack([blob[o:o + b_w] for o in b_off]).astype(np.float32),
              "e2e_text_offsets": t_off.astype(np.float64),
              "e2e_text": np.stack(text).astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _lap(what, t0=[time.perf_counter()]):
    """Phase timing on stderr (the JSON line on stdout stays alone)."""
    now = time.perf_counter()
    print("[bench] %-34s +%.1f s" % (what, now - t0[0]), file=sys.stderr, flush=True)
    t0[0] = now


def run_extras(eng, torch, stream, R, n_steps_total, arrays, orow, osamp, row_base, local_rank):
    """Extra keys of the 1-GPU line (module docstring)."""
    from dna_factory_b200 import _native, allele_stats
    out = {}
    eng.set_snps(**arrays)          # the e2e pass left one step's slice in the context: the whole table again
    eng.set_overrides(orow, osamp)
    eng.set_row_base(row_base)
    n_rows = 2 * n_steps_total * R
    n = N_CASES + N_CONTROLS
    # ---- value_sustained: back-to-back device-only calls over the whole resident table for >= 1 s (the timed `value`
    # region is a few tens of ms, during which the GPU never leaves its burst power state)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.generate_device(0, n_rows, PHILOX_SEED, level=LEVEL)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    calls = 0
    ev0.record(stream)
    while time.perf_counter() - t0 < 1.2:
        calls += eng.generate_device(0, n_rows, PHILOX_SEED, level=LEVEL)["calls"]
    ev1.record(stream)
    torch.cuda.synchronize()
    out["value_sustained"] = {"value": calls / (ev0.elapsed_time(ev1) * 1e-3), "unit": "calls/s", "seconds": ev0.elapsed_time(ev1) * 1e-3,
                              "what": "dnaf_generate_device over %d resident rows x %d samples, repeated back to back, -z %d" % (n_rows, n, LEVEL)}
    _lap("value_sustained")
    # ---- level_sweep: BASELINE config 5 (-z 1..9 on 20 000 samples), one window of rows per level
    sweep_rows = min(n_rows, 4 * R)
    out_buf = torch.empty(int(eng.plan(0, sweep_rows)[1]) + (1 << 20), dtype=torch.uint8, pin_memory=True).numpy()
    sweep = {}
    for lv in range(1, 10):
        eng.generate_device(0, sweep_rows, PHILOX_SEED, level=lv)                  # the tier's tables are built here
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = eng.generate_device(0, sweep_rows, PHILOX_SEED, level=lv)
        e1.record(stream)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        st2 = eng.generate_into(0, sweep_rows, PHILOX_SEED, out_buf, level=lv)
        dt = time.perf_counter() - t1
        sweep[str(lv)] = {"ratio": st["text_bytes"] / st["bgzf_bytes"], "value": st["calls"] / (e0.elapsed_time(e1) * 1e-3),
                          "e2e": st2["calls"] / dt, "bgzf_bytes_per_call": st["bgzf_bytes"] / st["calls"]}
    out["level_sweep"] = {"rows": sweep_rows, "samples": n, "note": "value: device only; e2e: one call, BGZF bytes into pinned host memory "
                          "(SNP table resident)", "levels": sweep}
    _lap("level_sweep")
    # ---- the drop-in CLI writing a real population.vcf.gz (C2 shape, SNP axis cut to 65536 rows)
    try:
        out["cli_to_file"] = cli_to_file(65536)
    except Exception as e:   # noqa: a full disk or a missing tmp dir must not cost the bench line
        out["cli_to_file"] = {"error": "%s: %s" % (type(e).__name__, e)}
    # ---- BASELINE config 1 in full through the same CLI (200 samples x 100 000 SNPs: rows of 800 bytes take the
    # generic three-kernel path), to set beside cpu_baseline_c1_full
    try:
        out["c1_full_cli"] = cli_to_file(100000, cases=100, controls=100)
    except Exception as e:   # noqa
        out["c1_full_cli"] = {"error": "%s: %s" % (type(e).__name__, e)}
    _lap("cli_to_file")
    # ---- allele-frequency chi-square of the draws (north_star), >= 1e8 calls
    out["allele_chi_square"] = allele_stats.chi_square_report(level=LEVEL, device=local_rank)
    _lap("allele_chi_square")
    return out


def cli_to_file(snps, level=LEVEL, cases=N_CASES, controls=N_CONTROLS):
    """`pop_factory -s <cases> -c <controls> -x <snps> -f 0.01 -z 2 --gpu_select` of the re-hosted CLI into a temp dir."""
    import contextlib
    import io
    import shutil
    import tempfile
    from dna_factory_b200 import pop_factory
    d = tempfile.mkdtemp(prefix="dnaf_cli_")
    try:
        buf = io.StringIO()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(buf):
            pop_factory.main(["-s", str(cases), "-c", str(controls), "-x", str(snps), "-f", str(MIN_MAF), "-z", str(level), "-p",
                              os.path.join(ROOT, "tests", "golden", "cli_small", "deleterious_config.yml"), "--outdir", d, "--seed", "123456", "--gpu_select"])
        wall = time.perf_counter() - t0
        import re
        m = re.findall(r"Finished write_vcf_snps chunk Elapsed time: ([0-9.]+) seconds", buf.getvalue())
        write_s = sum(float(x) for x in m)
        calls = (cases + controls) * snps
        size = os.path.getsize(os.path.join(d, "population.vcf.gz"))
        return {"calls_per_s_write_vcf_snps": calls / write_s if write_s else None, "calls_per_s_wall": calls / wall, "wall_s": wall,
                "write_vcf_snps_s": write_s, "vcf_gz_bytes": size, "snps": snps, "samples": cases + controls, "level": level}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def python_reference_run(steps, warmup, rows=600):
    """The UNMODIFIED reference CLI (oracle/_ref, materialised by oracle/make_ref.py) on the host cores:
    `pop_factory.py -s 10000 -c 10000 -x <rows> -f 0.01 -n <cores-1> -z 2`, one process run per step; the time of a
    step is the reference's own write_vcf_snps timer (pop_factory.py:417)."""
    from oracle import ref_cli
    runs = [ref_cli.run(N_CONTROLS, N_CASES, rows, LEVEL, min_maf=MIN_MAF) for _ in range(steps + warmup)][warmup:]
    total = sum(r["write_s"] for r in runs)
    calls = sum(r["calls"] for r in runs)
    return {"value": calls / total, "ms_per_step": 1e3 * total / len(runs), "cores": runs[0]["procs"] + 1, "procs": runs[0]["procs"],
            "wall_s_per_step": sum(r["wall_s"] for r in runs) / len(runs),
            "sample": "%d runs of the unmodified reference CLI `pop_factory.py -s %d -c %d -x %d -f %s -n %d -z %d` "
                      "(C2 with the SNP axis cut from 5 000 000 to %d rows); time = its own write_vcf_snps timer lines" % (
                          len(runs), N_CONTROLS, N_CASES, rows, MIN_MAF, runs[0]["procs"], LEVEL, rows)}


def python_reference_c1():
    """BASELINE config 1 in full through the unmodified reference CLI: -s 100 -c 100 -x 100000 -f 0.01 -z 2."""
    from oracle import ref_cli
    r = ref_cli.run(100, 100, 100000, LEVEL, min_maf=MIN_MAF)
    return {"value": r["calls_per_s"], "unit": "calls/s", "cores": r["procs"] + 1, "kind": "reference", "write_vcf_snps_s": r["write_s"],
            "wall_s": r["wall_s"], "vcf_bytes": r["vcf_bytes"],
            "sample": "config 1 in full: pop_factory.py -s 100 -c 100 -x 100000 -f 0.01 -n %d -z %d (2e7 calls)" % (r["procs"], LEVEL)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows-per-step", type=int, default=ROWS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip level_sweep / value_sustained / cli_to_file / chi-square")
    ap.add_argument("--level", type=int, default=LEVEL, help="-z of the timed steps (default: the workload's 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # debugging aid: DNAF_BENCH_ONE_GPU=1 runs all ranks of a torchrun launch on GPU 0 over gloo, so that the N > 1
    # code path (ranges, reductions, multi_gpu_parity) can be exercised on a 1-GPU box; such a line is not a result
    shared_gpu = os.environ.get("DNAF_BENCH_ONE_GPU") == "1"
    if shared_gpu:
        local_rank = 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        if rank != 0:
            return 0
        from oracle import make_ref
        make_ref.materialise()
        if make_ref.available():
            r = python_reference_run(args.steps, args.warmup)
            kind = "reference"
        else:
            r = cpu_reference_run(args.steps, args.warmup)
            kind = "port"
        line = {"impl": "reference", "metric": "genotype calls/sec to bgzf VCF", "value": r["value"],
                "unit": "calls/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic", "config": {"workload": WORKLOAD},
                "cpu_baseline": {"value": r["value"], "unit": "calls/s", "cores": r["cores"], "kind": kind,
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "calls/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from dna_factory_b200 import _native, host, partition

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: dna_factory_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if shared_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    red_dev = "cpu" if shared_gpu else "cuda"

    R = args.rows_per_step
    n_steps_total = warmup + args.steps
    # this rank's contiguous SNP range of the population: rows for the device-resident pass, then for e2e
    rows_needed = 2 * n_steps_total * R
    sex, ctl, table, orow, osamp = synth_population(rows_needed, rank, window=R)
    arrays = table.device_arrays()
    n = len(sex)
    row_base = partition.row_bounds(TOTAL_SNPS, world)[rank]   # this rank's contiguous SNP range of the job

    eng = _native.Engine(local_rank)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_samples(sex, ctl)
    eng.set_snps(**arrays)
    eng.set_overrides(orow, osamp)
    eng.set_row_base(row_base)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return partition.reduce_max(x, dist if world > 1 else None, red_dev)

    def sum_over_ranks(x):
        return partition.reduce_sum(x, dist if world > 1 else None, red_dev)

    _lap("population + context ready")
    # ------------------------------------------------------------------ device-resident pass (`value`)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for k in range(warmup):
        eng.generate_device(k * R, (k + 1) * R, PHILOX_SEED, level=args.level)
    barrier()
    sampler.mark_begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats = []
    ev0.record(stream)
    for k in range(warmup, n_steps_total):
        stats.append(eng.generate_device(k * R, (k + 1) * R, PHILOX_SEED, level=args.level))
    ev1.record(stream)
    barrier()
    sampler.mark_end()
    clocks = sampler.stop()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    calls = sum_over_ranks(sum(s["calls"] for s in stats))
    text_bytes = sum(s["text_bytes"] for s in stats)
    bgzf_bytes = sum(s["bgzf_bytes"] for s in stats)
    launches = int(sum(s["kernel_launches"] for s in stats))
    value = calls / (ms * 1e-3)

    # dominant kernel: algorithmic bytes = uncompressed text bytes it emits (DESIGN.md 6), live CUDA-event time
    stage_ms = {k: sum(s[k] for s in stats) for k in ("ms_sample", "ms_format", "ms_deflate", "ms_fused")}
    dom = max(stage_ms, key=stage_ms.get)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic, traffic_note = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tr = json.load(f)["k_auto" if args.level <= 2 else "k_lz"]
        traffic = tr["dram_bytes_per_launch"]
        traffic_note = "%s, one ncu --set full capture: %d-block launch emitting %.0f MB of text" % (
            tr["kernel"], tr["blocks"], tr["text_bytes_of_that_launch"] / 1e6)
    except Exception:
        pass
    stage_achieved = text_bytes / (stage_ms[dom] * 1e-3) / 1e9 if stage_ms[dom] > 0 else 0.0
    # the dominant KERNEL: k_auto, CUDA events right around its launches on the stream it is launched on
    ms_auto = sum(s["ms_auto"] for s in stats)
    auto_text = sum(s["auto_text_bytes"] for s in stats)
    auto_launches = sum(s["auto_launches"] for s in stats)
    if ms_auto > 0:
        achieved, kernel = auto_text / (ms_auto * 1e-3) / 1e9, ("k_auto" if args.level <= 2 else "k_lz")
    else:
        achieved, kernel = stage_achieved, dom.replace("ms_", "")
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "launches": auto_launches, "avg_launch_ms": ms_auto / max(1, auto_launches),
                "algorithmic_bytes_per_launch": auto_text / max(1, auto_launches),
                "stage": {"kernels": "k_auto + k_x + k_fused_text (side streams) between two events on the main stream",
                          "achieved": stage_achieved, "frac": stage_achieved / peak},
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "algorithmic_bytes": "uncompressed VCF text bytes emitted (%.3f B/call)" % (text_bytes / max(1, sum(
                    s["calls"] for s in stats))),
                "stage_ms_per_step": {k.replace("ms_", ""): v / len(stats) for k, v in stage_ms.items()},
                "pipeline_frac": (text_bytes / (sum(s["ms_total"] for s in stats) * 1e-3) / 1e9) / peak}

    _lap("value pass")
    # ------------------------------------------------------------------ end-to-end pass (`e2e`)
    # host buffers in, host buffer out: per step the step's SNP metadata goes H2D, the BGZF bytes come D2H
    # page-locked output buffer: the library DMAs straight into it; smaller passes so that the copy of one pass
    # overlaps the kernels of the next inside a step
    # Two contexts on this GPU, one host thread each, double-buffer whole steps: inside a call the passes are
    # pipelined (kernels of pass i+1 run while pass i crosses PCIe), and while one context's last pass drains the
    # other uploads its step's SNP metadata and starts its kernels.  Every step still does its own H2D, kernels and
    # D2H inside the timed region.  (1 context: 5.3 ms per step, 2: 4.2-4.7 ms, PCIe floor 4.1 ms.)
    n_ctx = int(os.environ.get("DNAF_BENCH_CTX", "2"))
    engines = [eng] + [_native.Engine(local_rank) for _ in range(n_ctx - 1)]
    for e in engines[1:]:
        e.set_samples(sex, ctl)
    out_bytes = int(eng.plan(0, R)[1]) + (1 << 20)
    outs = [torch.empty(out_bytes, dtype=torch.uint8, pin_memory=True).numpy() for _ in engines]
    for e in engines:
        e.set_chunk_bytes(E2E_CHUNK)
    base = n_steps_total * R

    def step_arrays(k):
        lo, hi = base + k * R, base + (k + 1) * R
        p0, p1 = int(arrays["prefix_off"][lo]), int(arrays["prefix_off"][hi])
        sel = (orow >= lo) & (orow < hi)
        return (dict(chrom_class=arrays["chrom_class"][lo:hi], n_alleles=arrays["n_alleles"][lo:hi],
                     thresholds=arrays["thresholds"][lo:hi], prefix_bytes=arrays["prefix_bytes"][p0:p1 + 1],
                     prefix_off=arrays["prefix_off"][lo:hi + 1] - np.uint64(p0)),
                (orow[sel] - np.uint64(lo)).astype(np.uint64), osamp[sel], lo)

    batches = [step_arrays(k) for k in range(n_steps_total)]

    e2e_level = [args.level]

    def e2e_step(j, b):
        a, o_r, o_s, lo = b
        e = engines[j]
        e.set_snps(**a)
        e.set_overrides(o_r, o_s)
        e.set_row_base(row_base + lo)
        return e.generate_into(0, R, PHILOX_SEED, outs[j], level=e2e_level[0])

    def run_steps(ks):
        """Steps ks, dealt round-robin to the contexts; every context runs its steps in order on its own thread."""
        res = [None] * len(ks)

        def worker(j):
            torch.cuda.set_device(local_rank)
            for i in range(j, len(ks), n_ctx):
                res[i] = e2e_step(j, batches[ks[i]])

        ts = [threading.Thread(target=worker, args=(j,)) for j in range(n_ctx)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return res

    run_steps([k for k in range(warmup) for _ in range(n_ctx)])   # every context runs every warm-up step
    barrier()
    t0 = time.perf_counter()
    e2e_stats = run_steps(list(range(warmup, n_steps_total)))
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    # the last step's stream, taken before the -z runs below reuse the output buffers
    last_blob = outs[(args.steps - 1) % n_ctx][:e2e_stats[-1]["bgzf_bytes"]].copy() if args.dump_outputs else None
    e2e_calls = sum_over_ranks(sum(s["calls"] for s in e2e_stats))
    h2d = int(np.mean([sum(v.nbytes for v in b[0].values()) + b[1].nbytes + b[2].nbytes for b in
                       batches[warmup:]]))
    d2h = int(np.mean([s["bgzf_bytes"] for s in e2e_stats]))
    launches += 0  # e2e launches are outside the `value` region
    # the same end-to-end steps at the reference's default -z 6 and at -z 4 / 5: past one GPU the host's PCIe fabric bounds
    # the rate, so fewer compressed bytes per call are worth more than kernel time (BASELINE config 5 at 1/2/4/8 GPUs)
    e2e_by_level = {str(args.level): e2e_calls / e2e_s}
    if not args.no_extras:
        for lv in (4, 5, 6):
            if lv == args.level:
                continue
            e2e_level[0] = lv
            ks = list(range(warmup, n_steps_total))[:6]
            run_steps(ks[:2] * n_ctx)                       # tables of the tier, warm-up
            barrier()
            t1 = time.perf_counter()
            st_l = run_steps(ks)
            torch.cuda.synchronize()
            dt = max_over_ranks(time.perf_counter() - t1)
            barrier()
            e2e_by_level[str(lv)] = sum_over_ranks(sum(x["calls"] for x in st_l)) / dt
        e2e_level[0] = args.level


    _lap("e2e pass")
    # ------------------------------------------------------------------ multi-GPU parity (N > 1)
    # Every rank regenerates nothing on trust: it inflates a window at the START of its own SNP range (produced with
    # its own row_base) and publishes (text bytes, blocks, CRC32 of the text); rank 0 recomputes every rank's window
    # on ITS GPU with that rank's row base -- rows are a pure function of (seed, global row, sample) -- and checks the
    # last rank's window against the CPU oracle as well.
    multi_gpu_parity = None
    if world > 1:
        W = 24
        eng.set_snps(**host.slice_snps(arrays, 0, W))     # the e2e pass left one of its steps in the context
        eng.set_overrides(*host.slice_overrides(orow, osamp, 0, W))
        eng.set_row_base(row_base)
        blob, st_w = eng.generate(0, W, PHILOX_SEED, level=args.level)
        mine = partition.window_signature(_inflate_bgzf(blob), st_w["bgzf_blocks"], st_w["crc_xor"])
        bounds = partition.row_bounds(TOTAL_SNPS, world)
        last_text = {}

        def recompute(r):   # runs on rank 0 only
            sex_r, ctl_r, table_r, orow_r, osamp_r = synth_population(R, r, window=R)
            chk = _native.Engine(local_rank)
            chk.set_samples(sex_r, ctl_r)
            chk.set_snps(**host.slice_snps(table_r.device_arrays(), 0, W))
            chk.set_overrides(*host.slice_overrides(orow_r, osamp_r, 0, W))
            chk.set_row_base(bounds[r])
            b2, st2 = chk.generate(0, W, PHILOX_SEED, level=args.level)
            chk.close()
            t2 = _inflate_bgzf(b2)
            if r == world - 1:
                last_text.update(text=t2, pop=(sex_r, ctl_r, table_r, orow_r, osamp_r))
            return partition.window_signature(t2, st2["bgzf_blocks"], st2["crc_xor"])

        multi_gpu_parity = partition.check_rank_windows(mine, recompute, dist, red_dev)
        if rank == 0 and multi_gpu_parity == "ok":      # and the last rank's window against the CPU oracle
            from oracle import oracle
            from types import SimpleNamespace
            sex_r, ctl_r, table_r, orow_r, osamp_r = last_text["pop"]
            fam = [SimpleNamespace(sex=int(a), is_control=bool(c), deleterious_snps=None if c else {}, person_id=i)
                   for i, (a, c) in enumerate(zip(sex_r, ctl_r))]
            flat = oracle.flatten(fam, [table_r.snp(q) for q in range(W)])
            flat["over_row"], flat["over_sample"] = host.slice_overrides(orow_r, osamp_r, 0, W)
            want, _ = oracle.rows_from_flat(flat, PHILOX_SEED, bounds[world - 1], n_threads=8)
            if want.tobytes() != last_text["text"]:
                multi_gpu_parity = "FAILED: rank %d window differs from the CPU oracle" % (world - 1)
        if rank == 0 and multi_gpu_parity != "ok":
            raise SystemExit("multi-GPU parity check failed: " + str(multi_gpu_parity))

    # ------------------------------------------------------------------ extras (rank 0 of a 1-GPU run)
    extras = {}
    if world == 1 and not args.no_extras:
        extras = run_extras(eng, torch, stream, R, n_steps_total, arrays, orow, osamp, row_base, local_rank)

    if rank == 0:
        cpu = None
        cpu_port = cpu_c1 = None
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(6, 1)
            cpu_port = {"value": r["value"], "unit": "calls/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
            cpu = cpu_port
            from oracle import make_ref
            make_ref.materialise()
            if make_ref.available():      # the reference's own `-n <cores-1>` multiprocess path, same box, same run
                r = python_reference_run(2, 0, rows=800)
                cpu = {"value": r["value"], "unit": "calls/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"],
                       "worker_processes": r["procs"], "wall_s_per_run": r["wall_s_per_step"]}
                cpu_c1 = python_reference_c1()
        line = {"metric": "genotype calls/sec to bgzf VCF", "value": value, "unit": "calls/s", "n_gpus": world,
                "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "samples": n, "rows_per_step": R, "level": args.level,
                           "l2_policy": "inputs larger than L2: each step draws a new %d MB text window" % (
                               text_bytes // len(stats) >> 20),
                           "partition": "contiguous SNP ranges per rank, no collective",
                           "e2e_pipeline": "2 contexts per GPU alternate whole steps; %d MB passes, 3 output buffers in rotation, DMA into the caller's pinned buffer" % (E2E_CHUNK >> 20)},
                "e2e": {"value": e2e_calls / e2e_s, "unit": "calls/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
                "compression_ratio": text_bytes / max(1, bgzf_bytes), "text_gb_per_s": text_bytes / (ms * 1e-3) / 1e9}
        if shared_gpu:
            line["debug"] = "DNAF_BENCH_ONE_GPU=1: every rank ran on GPU 0 over gloo -- plumbing check, not a result"
        _lap("cpu baselines")
        if cpu_port is not None:
            line["cpu_baseline_port"] = cpu_port
            line["cpu_baseline_python"] = cpu if cpu is not cpu_port else None
            line["cpu_baseline_c1_full"] = cpu_c1
        line["e2e_by_level"] = e2e_by_level
        if multi_gpu_parity is not None:
            line["multi_gpu_parity"] = multi_gpu_parity
        line.update(extras)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, stats[-1], e2e_stats[-1], last_blob)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
