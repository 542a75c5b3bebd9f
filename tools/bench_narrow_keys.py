#!/usr/bin/env python
"""What sorting 4- and 2-byte keys costs through lsb.sort (lsb_sort_device_typed / lsb_sort_segments_device_typed),
against torch.sort and against the same keys widened to 64 bits, on one GPU, in one process.

    python tools/bench_narrow_keys.py --out profiles/r7_narrow_keys.json [--reps 3] [--log2n 28 30]

Workloads: 2^28 and 2^30 keys made on the device -- float32 / float16 / bfloat16 standard normal, int32 / int16 /
uint32 / uint16 uniform bits -- sorted ascending with indices, as one 1-D array, as 2^10 rows (dim=-1) and as rows of
2^10.  Arms, alternated in a rotating order, one warm-up round and then `reps` rounds, medians of the whole synchronous
call (host clock to a device synchronise):
  lsb      lsb.sort(x, dim=-1): a fresh one-GPU sorter, pack, ceil(W / 16) key passes (+ the segment pass), unpack
  torch    torch.sort(x, dim=-1, stable=True) ("not measured" where torch has no CUDA sort of the dtype)
  widened  x cast to float64 / int64 / uint64, sort_tensor (1-D) or sort_segments (rows), values cast back
Every arm's values (bit for bit) and indices are compared with lsb's.  A second, profiled run (torch.profiler, CUDA
activities) takes the times of the pack and unpack kernels; their bytes per element over those times are reported
beside the HBM copy peak.  The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read
only)."""
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

DTYPES = ["float32", "bfloat16", "float16", "int32", "int16", "uint32", "uint16"]
COPY_PEAK_GBS = 6446.9  # HBM copy peak of the B200 these numbers were taken on, DESIGN.md
WIDE = {"float32": torch.float64, "bfloat16": torch.float64, "float16": torch.float64, "int32": torch.int64,
        "int16": torch.int64, "uint32": torch.uint64, "uint16": torch.uint64}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def make_keys(name, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if name.startswith("float") or name == "bfloat16":
        return torch.randn(n, dtype=torch.float32, device="cuda", generator=g).to(getattr(torch, name))
    w = 32 if name.endswith("32") else 16
    signed = torch.int32 if w == 32 else torch.int16
    bits = torch.randint(-(1 << (w - 1)), 1 << (w - 1), (n,), dtype=signed, device="cuda", generator=g)
    return bits.view(getattr(torch, name))


def bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def widen(x, name):
    if WIDE[name] == torch.uint64:  # no CUDA cast to uint64: zero-extend through int64, same bits
        return x.to(torch.int64).view(torch.uint64)
    return x.to(WIDE[name])


def narrow(v, x, name):
    return (v.view(torch.int64) if WIDE[name] == torch.uint64 else v).to(x.dtype)


def run_config(name, n, rows, reps, log):
    x = make_keys(name, n, 1).view(rows, n // rows) if rows > 1 else make_keys(name, n, 1)
    ref_v, ref_i = lsb.sort(x)
    samples = {a: [] for a in ("lsb", "torch", "widened")}
    checks = {}

    def arm_lsb():
        ms, (v, i) = host_ms(lambda: lsb.sort(x))
        checks["lsb"] = torch.equal(bits(v), bits(ref_v)) and torch.equal(i, ref_i)
        return ms

    def arm_torch():
        try:
            ms, (v, i) = host_ms(lambda: torch.sort(x, dim=-1, stable=True))
        except (RuntimeError, NotImplementedError) as e:
            checks["torch"] = f"not measured: {str(e).splitlines()[0]}"
            return None
        checks["torch"] = torch.equal(bits(v), bits(ref_v)) and torch.equal(i, ref_i)
        return ms

    def arm_widened():
        def f():
            w = widen(x, name)
            v, i = lsb.sort_tensor(w) if rows == 1 else lsb.sort_segments(w)
            return narrow(v, x, name), i
        try:
            ms, (v, i) = host_ms(f)
        except (RuntimeError, NotImplementedError) as e:  # a cast torch lacks on CUDA
            checks["widened"] = f"not measured: {str(e).splitlines()[0]}"
            return None
        checks["widened"] = torch.equal(bits(v), bits(ref_v)) and torch.equal(i, ref_i)
        return ms

    arms = [("lsb", arm_lsb), ("torch", arm_torch), ("widened", arm_widened)]
    for r in range(reps + 1):  # round 0 warms every arm up
        for a, fn in arms[r % len(arms):] + arms[:r % len(arms)]:
            ms = fn()
            if r and ms is not None:
                samples[a].append(ms)
            torch.cuda.empty_cache()
    med = {a: (statistics.median(v) if v else None) for a, v in samples.items()}
    shape = "1d" if rows == 1 else f"{rows}x{n // rows}"
    res = {"n": n, "dtype": name, "shape": shape, "median_ms": med, "samples_ms": samples, "verified": checks}
    log(f"2^{n.bit_length() - 1} {name:8s} {shape:12s} " +
        " ".join(f"{a}={m:.2f}" for a, m in med.items() if m is not None) + f"  checks={checks}")
    return res


def kernel_bytes(kernel, w_bytes):
    """bytes a pack / unpack kernel must move per element (read + write) with indices and both outputs"""
    if "unpack" in kernel:
        return 16 + w_bytes + 8
    return w_bytes + 16


def profile_kernels(name, n, rows):
    """device time of the pack / unpack kernels of lsb.sort from torch.profiler (CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    x = make_keys(name, n, 1).view(rows, n // rows) if rows > 1 else make_keys(name, n, 1)
    lsb.sort(x)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            lsb.sort(x)
            torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "pack_kernel" not in e.key:
            continue
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        ms = us / e.count / 1e3
        nbytes = kernel_bytes(e.key, x.element_size()) * n
        which = ("segsort_" if "segsort" in e.key else "") + ("unpack" if "unpack_kernel" in e.key else "pack")
        out[which] = {"kernel": e.key, "calls": e.count, "ms": ms, "bytes_per_element": nbytes // n,
                      "GBps": nbytes / ms / 1e6, "of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2n", type=int, nargs="+", default=[28, 30])
    ap.add_argument("--dtypes", nargs="+", default=DTYPES)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_narrow_keys: no CUDA device (there is no CPU fallback)")
    log = lambda m: print(m, flush=True)  # noqa: E731
    res = {"gpu": gpu_info(), "torch": torch.__version__, "copy_peak_GBps": COPY_PEAK_GBS, "reps": args.reps,
           "configs": [], "kernels": []}
    log(f"{res['gpu']}")
    layouts = lambda lg: [1, 1 << 10, 1 << (lg - 10)]  # noqa: E731  1-D, 2^10 long rows, rows of 2^10
    for lg in args.log2n:
        for name in args.dtypes:
            for rows in layouts(lg):
                res["configs"].append(run_config(name, 1 << lg, rows, args.reps, log))
                torch.cuda.empty_cache()
    for lg in args.log2n:
        for name in args.dtypes:
            for rows in layouts(lg):
                k = profile_kernels(name, 1 << lg, rows)
                shape = "1d" if rows == 1 else f"{rows}x{(1 << lg) // rows}"
                res["kernels"].append({"n": 1 << lg, "dtype": name, "shape": shape, **k})
                log(f"2^{lg} {name} {shape}: " + " ".join(f"{w}={v['ms']:.3f}ms/{v['GBps']:.0f}GB/s"
                                                           for w, v in k.items()))
                torch.cuda.empty_cache()
    res["all_verified"] = all(v is True or (isinstance(v, str) and v.startswith("not measured"))
                              for c in res["configs"] for v in c["verified"].values())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    log(f"all arms verified: {res['all_verified']}")
    sys.exit(0 if res["all_verified"] else 1)


if __name__ == "__main__":
    main()
