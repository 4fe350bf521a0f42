"""Call timeline of bench.py's device-only workload (`value`): back-to-back generate_device calls on one GPU.

    python scripts/pass_probe.py [--calls 200] [--windows 40] [--level 2] [--profile-calls 20] [--out DIR]

Population and step size are bench.py's (20 000 samples, 32 768-row sorted windows); the calls cycle over --windows
distinct windows.  Three parts, each in a run of its own so that one does not perturb the other:

  passes    one child process with DNAF_TRACE=1 (read once at library load) lists every pass of a few calls: rows,
            rows run implicitly by k_auto, blocks per kernel, host planning time
  timeline  the timed calls: per call ms_auto, ms_fused - ms_auto and ms_deflate (the library's CUDA events,
            dnaf_stats), the device span of the call (CUDA events on its stream), the host wall time of the call and
            the host gap to the next call
  profile   torch.profiler (CUDA activities) over --profile-calls calls: time per launch of every kernel, H2D copies,
            and the idle time of the GPU between kernels, inside calls and between them

The card's name, power limit and SM clocks are read (nvidia-smi) in the same run and printed with the numbers.
Prints one JSON line; with --out also writes it to DIR/pass_probe.json.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

R = bench.ROWS_PER_STEP
PASS_RE = re.compile(r"\[dnaf\] pass rows (\d+)(?: implicit (\d+) blocks (\d+) auto (\d+) x (\d+) text (\d+) generic (\d+))?"
                     r": plan (\d+) us, launch (\d+) us")


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:   # noqa: the numbers are still printed, marked with what could not be read
        return {"error": "nvidia-smi unavailable: %s" % type(e).__name__}


def engine(n_windows):
    import torch
    from dna_factory_b200 import _native
    sex, ctl, table, orow, osamp = bench.synth_population(n_windows * R, 0, window=R)
    eng = _native.Engine(0)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_samples(sex, ctl)
    eng.set_snps(**table.device_arrays())
    eng.set_overrides(orow, osamp)
    return eng, stream


def passes_child(args):
    """Runs with DNAF_TRACE=1: a few calls, the library prints one line per pass to stderr."""
    eng, _ = engine(args.windows)
    for k in range(args.windows):
        sys.stderr.write("[probe] call %d\n" % k)
        sys.stderr.flush()
        eng.generate_device(k * R, (k + 1) * R, bench.PHILOX_SEED, level=args.level)
    return 0


def pass_list(args):
    env = dict(os.environ, DNAF_TRACE="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--passes-child", "--windows", "3", "--level", str(args.level)],
                       capture_output=True, text=True, env=env, timeout=1800)
    if r.returncode:
        raise SystemExit("pass listing failed:\n" + r.stderr[-3000:])
    calls, cur = [], None
    for line in r.stderr.splitlines():
        if line.startswith("[probe] call"):
            cur = []
            calls.append(cur)
            continue
        m = PASS_RE.search(line)
        if m and cur is not None:
            g = [None if x is None else int(x) for x in m.groups()]
            p = {"rows": g[0], "plan_us": g[7], "launch_us": g[8]}
            if g[1] is not None:
                p.update(implicit_rows=g[1], blocks=g[2], auto_blocks=g[3], x_blocks=g[4], text_blocks=g[5], generic_blocks=g[6],
                         kind="implicit" if g[1] == g[0] else ("split" if g[1] else "planned"))
            cur.append(p)
    return calls[-1] if calls else []   # the last call: tables and buffers warm


def timeline(args, eng, stream):
    import torch
    for k in range(3):
        eng.generate_device(k * R, (k + 1) * R, bench.PHILOX_SEED, level=args.level)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
    rows, t_in, t_out = [], [], []
    t_begin = time.perf_counter()
    for k in range(args.calls):
        w = k % args.windows
        t_in.append(time.perf_counter())
        ev[k][0].record(stream)
        st = eng.generate_device(w * R, (w + 1) * R, bench.PHILOX_SEED, level=args.level)
        ev[k][1].record(stream)
        t_out.append(time.perf_counter())
        rows.append(st)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_begin
    span = np.array([a.elapsed_time(b) for a, b in ev])
    auto = np.array([s["ms_auto"] for s in rows])
    fused = np.array([s["ms_fused"] for s in rows])
    defl = np.array([s["ms_deflate"] for s in rows])
    call_wall = 1e3 * (np.array(t_out) - np.array(t_in))
    gap = 1e3 * (np.array(t_in[1:]) - np.array(t_out[:-1]))
    calls = sum(s["calls"] for s in rows)

    def stat(x):
        return {"median": float(np.median(x)), "mean": float(np.mean(x)), "p10": float(np.percentile(x, 10)),
                "p90": float(np.percentile(x, 90))}
    return {"calls": args.calls, "calls_per_s": calls / wall, "ms_per_call_wall": 1e3 * wall / args.calls,
            "ms_auto": stat(auto), "ms_fused_minus_auto": stat(fused - auto), "ms_deflate": stat(defl),
            "device_span_ms": stat(span), "host_wall_ms": stat(call_wall), "host_gap_ms": stat(gap),
            "per_call": [{"ms_auto": float(a), "ms_fused_minus_auto": float(f - a), "ms_deflate": float(d), "span_ms": float(s),
                          "wall_ms": float(w)} for a, f, d, s, w in zip(auto, fused, defl, span, call_wall)]}


def profile(args, eng, stream):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    n = args.profile_calls
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(n):
            w = k % args.windows
            eng.generate_device(w * R, (w + 1) * R, bench.PHILOX_SEED, level=args.level)
        torch.cuda.synchronize()
    kern, copies = [], []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        t0 = e.time_range.start
        t1 = e.time_range.end
        name = e.name
        if "memcpy" in name.lower() or "memset" in name.lower():
            copies.append((name, t0, t1))
        else:
            kern.append((re.sub(r"^(?:void )?(?:dnaf::)?([A-Za-z_0-9]+).*$", r"\1", name), t0, t1))
    by = {}
    for name, t0, t1 in kern:
        by.setdefault(name, []).append(t1 - t0)
    kernels = {k: {"launches": len(v), "us_per_launch_median": float(np.median(v)), "us_per_launch_mean": float(np.mean(v)),
                   "us_total_per_call": float(np.sum(v)) / n} for k, v in sorted(by.items())}
    cby = {}
    for name, t0, t1 in copies:
        cby.setdefault(name, []).append(t1 - t0)
    copy_sum = {k: {"count": len(v), "us_total_per_call": float(np.sum(v)) / n} for k, v in cby.items()}
    # GPU idle: the union of kernel intervals over all streams, gaps between consecutive busy intervals
    iv = sorted((t0, t1) for _, t0, t1 in kern)
    busy, gaps = [], []
    for t0, t1 in iv:
        if busy and t0 <= busy[-1][1]:
            busy[-1][1] = max(busy[-1][1], t1)
        else:
            if busy:
                gaps.append(t0 - busy[-1][1])
            busy.append([t0, t1])
    span = (iv[-1][1] - iv[0][0]) if iv else 0.0
    gaps = np.array(gaps) if gaps else np.zeros(1)
    return {"calls": n, "kernels_us": kernels, "copies_us": copy_sum, "window_us_per_call": span / n,
            "idle_us_per_call": float(gaps.sum()) / n, "gaps_over_5us_per_call": float((gaps > 5).sum()) / n,
            "largest_gaps_us": [float(x) for x in sorted(gaps)[-8:][::-1]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--windows", type=int, default=40, help="distinct 32768-row windows the calls cycle over")
    ap.add_argument("--level", type=int, default=bench.LEVEL)
    ap.add_argument("--profile-calls", type=int, default=20)
    ap.add_argument("--out", metavar="DIR")
    ap.add_argument("--passes-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.passes_child:
        return passes_child(args)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pass_probe.py needs a CUDA device: dna_factory_b200 has no CPU fallback")
    info = {"card": card(), "level": args.level, "rows_per_call": R, "full_plan": bool(os.environ.get("DNAF_FULL_PLAN"))}
    info["passes"] = pass_list(args)
    eng, stream = engine(args.windows)
    info["timeline"] = timeline(args, eng, stream)
    info["profile"] = profile(args, eng, stream)
    info["card_after"] = card()
    line = json.dumps(info)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "pass_probe.json"), "w") as f:
            f.write(line + "\n")
    summary = {k: info["timeline"][k] for k in ("calls_per_s", "ms_per_call_wall")}
    summary.update({k: info["timeline"][k]["median"] for k in ("ms_auto", "ms_fused_minus_auto", "ms_deflate", "device_span_ms",
                                                                "host_gap_ms")})
    summary["k_x_us_per_launch"] = info["profile"]["kernels_us"].get("k_x", {}).get("us_per_launch_median")
    summary["idle_us_per_call"] = info["profile"]["idle_us_per_call"]
    print(json.dumps({"card": info["card"], "passes": info["passes"], "summary": summary}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
