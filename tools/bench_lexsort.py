#!/usr/bin/env python
"""What a sort by several key columns costs through lsb.lexsort / DistributedSorter.lexsort_device, against torch's
chained stable argsorts, on one GPU, in one process.

    python tools/bench_lexsort.py --out profiles/r9_lexsort.json [--reps 3] [--log2n 28 30]

Workloads (columns least significant first, made on the device, no NaNs so that torch's order is the same):
  i32_f32        (int32 uniform bits, float32 normal)            one round of 64 bits: 4 passes at radix 16
  bf16_i16_i32   (bfloat16 normal, int16, int32 uniform bits)    one round of 64 bits
  i64_i64        (int64, int64 uniform bits)                     two rounds: 8 passes and one gather pack
  i64x3          3 x int64 uniform bits                          three rounds
  i64x2_low      2 x int64 of 2^10 values                        two rounds whose constant digits are skipped
  i32_f32_vals   i32_f32 with float64 vals gathered by the unpack
Arms, alternated in a rotating order, one warm-up round and then `reps` rounds, medians of the whole synchronous call
(host clock to a device synchronise):
  lsb      lsb.lexsort(columns): a fresh one-GPU sorter per call
  kept     DistributedSorter.lexsort_device(columns) on a sorter made once
  torch    p = argsort(col_0, stable); p = p[argsort(col_c[p], stable)] for c = 1 .. K-1 (then vals[p])
Every arm's output is compared bit for bit with lsb's.  A second, profiled run (torch.profiler, CUDA activities) of
the kept sorter takes the times of the pack, gather pack and unpack kernels; their bytes per element over those
times are reported beside the HBM copy peak.  The card's name and power limit are read in the same run
(nvidia-smi --query-gpu, read only)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import distributed_lsb_b200 as lsb  # noqa: E402

COPY_PEAK_GBS = 6446.9  # HBM copy peak of the B200 these numbers were taken on, DESIGN.md
WORKLOADS = {
    "i32_f32": ["int32", "float32"],
    "bf16_i16_i32": ["bfloat16", "int16", "int32"],
    "i64_i64": ["int64", "int64"],
    "i64x3": ["int64", "int64", "int64"],
    "i64x2_low": ["int64_low", "int64_low"],
    "i32_f32_vals": ["int32", "float32"],
}
WIDTH = {"int64": 8, "int64_low": 8, "int32": 4, "float32": 4, "int16": 2, "bfloat16": 2}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def make_column(kind, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind in ("float32", "bfloat16"):
        return torch.randn(n, dtype=torch.float32, device="cuda", generator=g).to(getattr(torch, kind))
    if kind == "int64_low":
        return torch.randint(0, 1 << 10, (n,), dtype=torch.int64, device="cuda", generator=g)
    w = {"int64": 64, "int32": 32, "int16": 16}[kind]
    return torch.randint(-(1 << (w - 1)), (1 << (w - 1)) - 1, (n,), dtype=getattr(torch, kind), device="cuda", generator=g)


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def torch_chain(cols, vals):
    p = torch.argsort(cols[0], stable=True)
    for c in cols[1:]:
        p = p[torch.argsort(c[p], stable=True)]
    return p if vals is None else vals[p]


def same(a, b):
    return torch.equal(a.view(torch.int64), b.view(torch.int64))


def run_config(wl, n, reps, log):
    cols = [make_column(k, n, seed=c + 1) for c, k in enumerate(WORKLOADS[wl])]
    vals = torch.randn(n, dtype=torch.float64, device="cuda") if wl.endswith("_vals") else None
    ref = lsb.lexsort(cols, vals=vals)
    torch.cuda.empty_cache()
    sorter = lsb.DistributedSorter(n, ranks=1)
    samples = {a: [] for a in ("lsb", "kept", "torch")}
    checks, stats = {}, {}

    def arm_lsb():
        ms, v = host_ms(lambda: lsb.lexsort(cols, vals=vals))
        checks["lsb"] = same(v, ref)
        return ms

    def arm_kept():
        ms, (v, st) = host_ms(lambda: sorter.lexsort_device(cols, vals))
        checks["kept"] = same(v, ref)
        stats.update(passes=st.passes, skipped=st.skipped, subpasses=st.subpasses, kernel_launches=st.kernel_launches,
                     device_ms=st.device_ms)
        return ms

    def arm_torch():
        ms, v = host_ms(lambda: torch_chain(cols, vals))
        checks["torch"] = same(v, ref)
        return ms

    arms = [("lsb", arm_lsb), ("kept", arm_kept), ("torch", arm_torch)]
    for r in range(reps + 1):  # round 0 warms every arm up
        for a, fn in arms[r % len(arms):] + arms[:r % len(arms)]:
            ms = fn()
            if r:
                samples[a].append(ms)
            torch.cuda.empty_cache()
    sorter.close()
    med = {a: statistics.median(v) for a, v in samples.items()}
    res = {"n": n, "workload": wl, "columns": WORKLOADS[wl], "vals": vals is not None, "median_ms": med,
           "samples_ms": samples, "stats": stats, "verified": checks}
    log(f"2^{n.bit_length() - 1} {wl:13s} " + " ".join(f"{a}={m:.2f}" for a, m in med.items()) +
        f"  passes={stats['passes']} skipped={stats['skipped']}  checks={checks}")
    return res


def kernel_bytes(kernel, wl):
    """bytes per element a kernel must move (read + write): the pack reads round 0's columns, a gather pack the records
    and its round's columns (random reads, each of which touches a whole 32-byte DRAM sector this count leaves out)"""
    widths = [WIDTH[k] for k in WORKLOADS[wl]]
    rounds = lsb.hostlogic.lexsort_rounds([8 * w for w in widths], 16)
    round_bytes = lambda r: sum(widths[r[0]:r[0] + r[1]])  # noqa: E731
    if "lexsort_unpack" in kernel:
        return 16 + 8 + 8
    if "unpack_kernel" in kernel:
        return 16 + 8
    if "<true," in kernel:
        return 16 + statistics.mean(round_bytes(r) for r in rounds[1:]) + 16
    return round_bytes(rounds[0]) + 16


def profile_kernels(wl, n):
    """device time of the lexsort kernels of lexsort_device from torch.profiler (CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    cols = [make_column(k, n, seed=c + 1) for c, k in enumerate(WORKLOADS[wl])]
    vals = torch.randn(n, dtype=torch.float64, device="cuda") if wl.endswith("_vals") else None
    out = {}
    with lsb.DistributedSorter(n, ranks=1) as s:
        s.lexsort_device(cols, vals)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                s.lexsort_device(cols, vals)
                torch.cuda.synchronize()
    for e in prof.key_averages():
        if "lexsort" not in e.key and "unpack_kernel" not in e.key:
            continue
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        ms = us / e.count / 1e3
        nbytes = kernel_bytes(e.key, wl) * n
        which = ("gather_pack" if "<true," in e.key else "pack") if "pack_kernel" in e.key and "unpack" not in e.key \
            else "unpack"
        out[which] = {"kernel": e.key, "calls": e.count, "ms": ms, "bytes_per_element": nbytes / n,
                      "GBps": nbytes / ms / 1e6, "of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2n", type=int, nargs="+", default=[28, 30])
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_lexsort: no CUDA device (there is no CPU fallback)")
    log = lambda m: print(m, flush=True)  # noqa: E731
    res = {"gpu": gpu_info(), "torch": torch.__version__, "copy_peak_GBps": COPY_PEAK_GBS, "reps": args.reps,
           "configs": [], "kernels": []}
    log(f"{res['gpu']}")
    for lg in args.log2n:
        for wl in args.workloads:
            res["configs"].append(run_config(wl, 1 << lg, args.reps, log))
            torch.cuda.empty_cache()
    for wl in args.workloads:
        lg = max(args.log2n)
        k = profile_kernels(wl, 1 << lg)
        res["kernels"].append({"n": 1 << lg, "workload": wl, **k})
        log(f"2^{lg} {wl}: " + " ".join(f"{w}={v['ms']:.3f}ms/{v['GBps']:.0f}GB/s ({v['of_copy_peak']:.2f})"
                                        for w, v in k.items()))
        torch.cuda.empty_cache()
    res["all_verified"] = all(v is True for c in res["configs"] for v in c["verified"].values())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    log(f"all arms verified: {res['all_verified']}")
    sys.exit(0 if res["all_verified"] else 1)


if __name__ == "__main__":
    main()
