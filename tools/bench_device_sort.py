#!/usr/bin/env python
"""What sorting CUDA tensors costs through DistributedSorter.sort_device (lsb_sort_device), against the sort alone, torch.sort
and the host-memory path, on one GPU, in one process.

    python tools/bench_device_sort.py --out profiles/r4_device_sort.json [--reps 5] [--log2n 28 30]

Workloads: 2^28 and 2^30 keys made on the device -- uint64 random bits, int64 random bits, float64 standard normal --
with no vals (the values are the input index: the stable argsort) and with random int64 vals.  Arms, alternated in a
rotating order, one warm-up round and then `reps` rounds, medians reported:
  floor        lsb_sort's device_ms on the same records already in the shard (written there by a device copy)
  sort_device  the whole synchronous call, host clock (pack + sort + unpack + call overhead)
  torch_sort   torch.sort(keys, stable=True) (+ vals[indices] with vals), host clock to a device synchronise
  sort_tensor  the one-shot convenience, context creation included
  sort_pairs   numpy arrays through host memory (2^28 only), host clock
  create       lsb_create of a one-GPU context of n elements
Every arm's keys and values are compared with sort_device's, bit for bit, and verify() passes after every floor sort.
A second, profiled run (torch.profiler, CUDA activities) takes the pack_kernel / unpack_kernel times; their bytes per
element over those times are reported beside the HBM copy peak.  The card's name and power limit are read in the same
run (nvidia-smi --query-gpu, read only)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

KEYS = {"u64": (torch.uint64, 0), "i64": (torch.int64, L.FLAG_KEY_I64), "f64": (torch.float64, L.FLAG_KEY_F64)}
# bytes each kernel must move per element (read + write)
PACK_BYTES = {False: 8 + 16, True: 16 + 16}      # vals given?
UNPACK_BYTES = {2: 16 + 16, 1: 16 + 8}           # outputs written
COPY_PEAK_GBS = 6446.9                           # HBM copy peak of the B200 these numbers were taken on, DESIGN.md


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def make_keys(kind, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "f64":
        return torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    bits = torch.randint(-(1 << 63), (1 << 63) - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    return bits.view(KEYS[kind][0])


class _Shard:
    """the sorter's current shard as an (n, 2) int64 tensor, zero copy"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n, 2), "typestr": "<i8", "data": (ptr, False), "version": 3}


def same(a, b):
    return a is not None and b is not None and torch.equal(a.view(torch.int64), b.view(torch.int64))


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def run_config(n, kind, with_vals, reps, log):
    dtype, flags = KEYS[kind]
    keys = make_keys(kind, n, 1)
    vals = make_keys("i64", n, 2) if with_vals else None
    records = torch.stack((keys.view(torch.int64), (vals if with_vals else torch.arange(n, device="cuda"))), 1)
    t0 = time.perf_counter()
    s = lsb.DistributedSorter(n, ranks=1, flags=flags)
    create_first = (time.perf_counter() - t0) * 1e3
    ref_k, ref_v, _ = s.sort_device(keys, vals)  # the answer every arm is compared with
    samples = {a: [] for a in ("floor", "sort_device", "sort_device_sort_ms", "torch_sort", "sort_tensor", "sort_pairs",
                               "create")}
    checks = {}
    host_k = keys.view(torch.int64).cpu().numpy().view(np.dtype(str(dtype).replace("torch.", ""))) if n <= 1 << 28 else None
    host_v = vals.cpu().numpy() if (with_vals and host_k is not None) else None

    def floor():
        torch.as_tensor(_Shard(s.device_ptr(), n), device="cuda").copy_(records)
        torch.cuda.synchronize()
        st = s.my_sort()
        got = torch.as_tensor(_Shard(s.device_ptr(), n), device="cuda")
        v = s.verify(raise_on_failure=False)
        checks["floor"] = same(got[:, 0], ref_k) and same(got[:, 1], ref_v) and (with_vals or v.order_violations == 0)
        return st.device_ms

    def sort_device():
        ms, (k, v, st) = host_ms(lambda: s.sort_device(keys, vals))
        checks["sort_device"] = same(k, ref_k) and same(v, ref_v)
        samples["sort_device_sort_ms"].append(st.device_ms)
        return ms

    def torch_sort():
        def f():
            k, i = torch.sort(keys, stable=True)
            return k, (vals[i] if with_vals else i)
        try:
            ms, (k, v) = host_ms(f)
        except RuntimeError as e:  # torch has no CUDA sort for this dtype
            checks["torch_sort"] = f"not measured: {str(e).splitlines()[0]}"
            return None
        checks["torch_sort"] = same(k, ref_k) and same(v, ref_v)
        return ms

    def sort_tensor():
        ms, (k, v) = host_ms(lambda: lsb.sort_tensor(keys, vals))
        checks["sort_tensor"] = same(k, ref_k) and same(v, ref_v)
        return ms

    def sort_pairs():
        if host_k is None:
            return None
        t = time.perf_counter()
        k, v = lsb.sort_pairs(host_k, host_v)
        ms = (time.perf_counter() - t) * 1e3
        checks["sort_pairs"] = (np.array_equal(k.view(np.int64), ref_k.view(torch.int64).cpu().numpy()) and
                                np.array_equal(v.view(np.int64), ref_v.view(torch.int64).cpu().numpy()))
        return ms

    def create():
        t = time.perf_counter()
        c = lsb.DistributedSorter(n, ranks=1, flags=flags)
        ms = (time.perf_counter() - t) * 1e3
        c.close()
        return ms

    arms = [("floor", floor), ("sort_device", sort_device), ("torch_sort", torch_sort), ("sort_tensor", sort_tensor),
            ("sort_pairs", sort_pairs), ("create", create)]
    for r in range(reps + 1):  # round 0 warms every arm up
        for name, fn in arms[r % len(arms):] + arms[:r % len(arms)]:
            ms = fn()
            if r and ms is not None:
                samples[name].append(ms)
        if r == 0:
            samples["sort_device_sort_ms"].clear()
    s.close()
    med = {a: (statistics.median(v) if v else None) for a, v in samples.items()}
    res = {"n": n, "keys": kind, "vals": "int64" if with_vals else "index", "median_ms": med, "samples_ms": samples,
           "create_first_ms": create_first, "verified": checks}
    log(f"2^{n.bit_length() - 1} {kind:3s} vals={res['vals']:5s} " +
        " ".join(f"{a}={m:.2f}" for a, m in med.items() if m is not None) + f"  checks={checks}")
    return res


def profile_kernels(n, kind, with_vals):
    """device time of pack_kernel / unpack_kernel from torch.profiler (CUDA activities), both outputs and one output"""
    from torch.profiler import ProfilerActivity, profile
    dtype, flags = KEYS[kind]
    keys = make_keys(kind, n, 1)
    vals = make_keys("i64", n, 2) if with_vals else None
    out = {}
    with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
        s.sort_device(keys, vals)
        for outputs, kw in ((2, {}), (1, {"keys_out": False})):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    s.sort_device(keys, vals, **kw)
            for e in prof.key_averages():
                if "pack_kernel" not in e.key:
                    continue
                us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                which = "unpack" if "unpack_kernel" in e.key else "pack"
                if which == "pack" and outputs == 1:
                    continue
                ms = us / e.count / 1e3
                nbytes = (PACK_BYTES[with_vals] if which == "pack" else UNPACK_BYTES[outputs]) * n
                out[f"{which}" + (f"_{outputs}out" if which == "unpack" else "")] = {
                    "kernel": e.key, "calls": e.count, "ms": ms, "bytes_per_element": nbytes // n,
                    "GBps": nbytes / ms / 1e6, "of_copy_peak": nbytes / ms / 1e6 / COPY_PEAK_GBS}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--log2n", type=int, nargs="+", default=[28, 30])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_device_sort: no CUDA device (there is no CPU fallback)")
    log = lambda m: print(m, flush=True)  # noqa: E731
    res = {"gpu": gpu_info(), "torch": torch.__version__, "copy_peak_GBps": COPY_PEAK_GBS, "reps": args.reps,
           "configs": [], "kernels": []}
    log(f"{res['gpu']}")
    for lg in args.log2n:
        for kind in KEYS:
            for with_vals in (False, True):
                res["configs"].append(run_config(1 << lg, kind, with_vals, args.reps, log))
                torch.cuda.empty_cache()
    for lg in args.log2n:
        for kind in KEYS:
            for with_vals in (False, True):
                k = profile_kernels(1 << lg, kind, with_vals)
                res["kernels"].append({"n": 1 << lg, "keys": kind, "vals": "int64" if with_vals else "index", **k})
                log(f"2^{lg} {kind} vals={with_vals}: " + " ".join(f"{w}={v['ms']:.3f}ms/{v['GBps']:.0f}GB/s"
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
