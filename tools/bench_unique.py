#!/usr/bin/env python
"""What the distinct keys or rows of a CUDA tensor cost through lsb.unique / DistributedSorter.unique_device, against
torch.unique / torch.unique_consecutive, on one GPU, in one process.

    python tools/bench_unique.py --out profiles/r11_unique.json [--reps 3] [--log2n 28 30]

Workloads (n elements or rows, made on the device, no NaNs so that torch's groups are the same; every call asks for
the values, the inverse and the counts):
  i64_uniform   int64 uniform bits: U ~ n
  i64_2p20      int64 of 2^20 distinct values
  f32_normal    float32 normal
  u64_uniform   uint64 uniform bits (torch.unique has no CUDA kernel for uint64: no torch arm)
  edges_i64     int64[n, 2] rows of 2^20 x 2^10 values, dim=0: two rounds, one gather-flag launch
  edges_i32     int32[n, 2] rows of 2^20 x 2^10 values, dim=0: one round of 64 bits
  consec_i64    unique_consecutive of sorted int64 of 2^20 distinct values
Arms, alternated in a rotating order, one warm-up round and then `reps` rounds, medians of the whole synchronous call
(host clock to a device synchronise):
  lsb      lsb.unique / lsb.unique_consecutive: a fresh one-GPU sorter per call, values gathered by index
  kept     DistributedSorter.unique_device(columns) on a sorter made once (the columns made once too)
  torch    torch.unique(sorted=True, return_inverse=True, return_counts=True[, dim=0]) / torch.unique_consecutive
Every arm's output is compared bit for bit with lsb's.  A second, profiled run (torch.profiler, CUDA activities) of the
kept sorter takes the times of the unique kernels; their bytes per element over those times are reported beside the
HBM copy peak.  The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read only)."""
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
WORKLOADS = ["i64_uniform", "i64_2p20", "f32_normal", "u64_uniform", "edges_i64", "edges_i32", "consec_i64"]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def make_input(wl, n):
    """(input, dim, consecutive)"""
    g = torch.Generator(device="cuda").manual_seed(len(wl))
    ri = lambda lo, hi, dt=torch.int64: torch.randint(lo, hi, (n,), dtype=dt, device="cuda", generator=g)  # noqa: E731
    if wl == "i64_uniform":
        return ri(-(1 << 63), (1 << 63) - 1), None, False
    if wl == "i64_2p20":
        return ri(0, 1 << 20) * 7919, None, False
    if wl == "f32_normal":
        return torch.randn(n, device="cuda", generator=g), None, False
    if wl == "u64_uniform":
        return ri(-(1 << 63), (1 << 63) - 1).view(torch.uint64), None, False
    if wl.startswith("edges"):
        dt = torch.int64 if wl == "edges_i64" else torch.int32
        return torch.stack([ri(0, 1 << 20, dt), ri(0, 1 << 10, dt)], dim=1), 0, False
    return torch.sort(ri(0, 1 << 20))[0], None, True


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def same(a, b):
    return a.shape == b.shape and torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


def lsb_call(x, dim, consecutive):
    if consecutive:
        return lsb.unique_consecutive(x, return_inverse=True, return_counts=True, dim=dim)
    return lsb.unique(x, return_inverse=True, return_counts=True, dim=dim)


def torch_call(x, dim, consecutive):
    if consecutive:
        return torch.unique_consecutive(x, return_inverse=True, return_counts=True, dim=dim)
    return torch.unique(x, sorted=True, return_inverse=True, return_counts=True, dim=dim)


def columns_of(x, dim):
    return lsb.lsbsort._unique_columns(torch, x, dim)[2]


def run_config(wl, n, reps, log):
    x, dim, consecutive = make_input(wl, n)
    ref = lsb_call(x, dim, consecutive)
    cols = columns_of(x, dim)
    torch.cuda.empty_cache()
    sorter = lsb.DistributedSorter(n, ranks=1)
    samples = {"lsb": [], "kept": [], "torch": []}
    checks, stats = {}, {}

    def arm_lsb():
        ms, out = host_ms(lambda: lsb_call(x, dim, consecutive))
        checks["lsb"] = all(same(a, b) for a, b in zip(out, ref))
        return ms

    def arm_kept():
        ms, (index, inverse, counts, u, st) = host_ms(lambda: sorter.unique_device(cols, consecutive=consecutive))
        bits = x.view({8: torch.int64, 4: torch.int32}[x.element_size()])  # torch indexes no uint64 CUDA tensor
        values = (bits.reshape(-1)[index[:u]] if dim is None else bits.index_select(dim, index[:u])).view(x.dtype)
        checks["kept"] = same(values, ref[0]) and same(inverse, ref[1].reshape(-1)) and same(counts[:u], ref[2])
        stats.update(unique=u, passes=st.passes, skipped=st.skipped, kernel_launches=st.kernel_launches,
                     device_ms=st.device_ms)
        return ms

    def arm_torch():
        ms, out = host_ms(lambda: torch_call(x, dim, consecutive))
        checks["torch"] = all(same(a, b) for a, b in zip(out, ref))
        return ms

    arms = [("lsb", arm_lsb), ("kept", arm_kept), ("torch", arm_torch)]
    try:
        torch_call(x[:16], dim, consecutive)
    except (RuntimeError, NotImplementedError) as e:  # torch has no CUDA kernel for the dtype
        arms = arms[:2]
        samples.pop("torch")
        log(f"{wl}: no torch arm ({str(e).splitlines()[0][:100]})")
    for r in range(reps + 1):  # round 0 warms every arm up
        for a, fn in arms[r % len(arms):] + arms[:r % len(arms)]:
            ms = fn()
            if r:
                samples[a].append(ms)
            torch.cuda.empty_cache()
    sorter.close()
    med = {a: statistics.median(v) for a, v in samples.items()}
    res = {"n": n, "workload": wl, "dtype": str(x.dtype), "shape": list(x.shape), "dim": dim, "consecutive": consecutive,
           "median_ms": med, "samples_ms": samples, "stats": stats, "verified": checks}
    log(f"2^{n.bit_length() - 1} {wl:12s} " + " ".join(f"{a}={m:.2f}" for a, m in med.items()) +
        f"  U={stats['unique']} passes={stats['passes']} launches={stats['kernel_launches']}  checks={checks}")
    return res


def kernel_bytes(kernel, col_bytes, nrounds_first_bytes, frac):
    """bytes per element a unique kernel must move (read + write), `frac` = U / n.  Random accesses (the gathers of the
    flag kernel, the inverse scatter of sorted mode) each touch a whole 32-byte DRAM sector this count leaves out."""
    if "unique_flag_kernel" in kernel:
        rec = 16 if "<true" in kernel else 0
        return rec + nrounds_first_bytes + 1
    if "unique_counts_kernel" in kernel:
        return 16 * frac
    reads = (16 if ", 0>" in kernel else col_bytes) + (1 if nrounds_first_bytes else 0)  # + the earlier rounds' flag
    if "unique_tile_kernel<0" in kernel:
        return reads
    return reads + 8 + 16 * frac


def profile_kernels(wl, n):
    """device time of every unique kernel of unique_device from torch.profiler (CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    x, dim, consecutive = make_input(wl, n)
    cols = columns_of(x, dim)
    out = {}
    with lsb.DistributedSorter(n, ranks=1) as s:
        u = s.unique_device(cols, consecutive=consecutive)[3]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                s.unique_device(cols, consecutive=consecutive)
                torch.cuda.synchronize()
    # the last round's columns (read by the tile kernels in consecutive mode) and the earlier rounds' (flag kernels)
    widths = [c.element_size() for c in cols]
    rounds = lsb.hostlogic.lexsort_rounds([8 * w for w in widths], 16)
    last = sum(widths[rounds[-1][0]:rounds[-1][0] + rounds[-1][1]])
    earlier = statistics.mean(sum(widths[r[0]:r[0] + r[1]]) for r in rounds[:-1]) if len(rounds) > 1 else 0
    for e in prof.key_averages():
        if "unique_" not in e.key and "global_scan_kernel" not in e.key:
            continue
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        ms = us / e.count / 1e3
        per = 16 * (n // 2048 + 1) / n if "global_scan" in e.key else kernel_bytes(e.key, last, earlier, u / n)
        nbytes = per * n
        out[e.key] = {"calls": e.count, "ms": ms, "bytes_per_element": per, "GBps": nbytes / ms / 1e6,
                      "of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2n", type=int, nargs="+", default=[28, 30])
    ap.add_argument("--workloads", nargs="+", default=WORKLOADS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_unique: no CUDA device (there is no CPU fallback)")
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
        res["kernels"].append({"n": 1 << lg, "workload": wl, "kernels": k})
        for name, v in k.items():
            log(f"2^{lg} {wl}: {name[:60]} {v['ms']:.3f} ms, {v['bytes_per_element']:.2f} B/elt, {v['GBps']:.0f} GB/s "
                f"({v['of_copy_peak']:.2f})")
        torch.cuda.empty_cache()
    res["all_verified"] = all(v is True for c in res["configs"] for v in c["verified"].values())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    log(f"all arms verified: {res['all_verified']}")
    sys.exit(0 if res["all_verified"] else 1)


if __name__ == "__main__":
    main()
