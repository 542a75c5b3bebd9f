#!/usr/bin/env python
"""What sorting many groups of a CUDA tensor at once costs through DistributedSorter.sort_segments
(lsb_sort_segments_device), against the one-segment sort and what a torch user runs today, on one GPU, in one process.

    python tools/bench_segments.py --out profiles/r5_segments.json [--reps 3] [--log2n 28 30]

Workloads: 2^28 and 2^30 keys made on the device -- uint64 random bits and float64 standard normal -- with no vals (the
values are indices) and with random int64 vals, in five segmentations:
  one       1 segment
  rows1k    2^10 rows of n / 2^10               (2-D [B, L]: the values are indices within the row)
  width1k   n / 2^10 rows of 2^10
  width32   n / 32 rows of 32
  ragged    2^16 segments with lognormal sizes (sigma 1), given as CSR offsets (the values are global indices)
Arms, alternated per workload after a warm-up round, `reps` rounds, medians reported:
  segments     sort_segments on a sorter kept across calls, host clock of the synchronous call (its device_ms too)
  sort_device  sort_device of the same keys on the same sorter: the one-segment floor
  torch        float64 only (torch has no CUDA sort of uint64): rows -- torch.sort(x2d, dim=-1, stable=True) and a
               gather of vals; ragged -- a stable sort by key, a gather of the segment ids (precomputed, not timed),
               a stable sort by segment id and the gathers of keys and vals: what torch offers for ragged groups
Every torch arm's keys and values are compared with sort_segments' bit for bit, and sort_segments of one segment with
sort_device.  A second, profiled run (torch.profiler, CUDA activities) takes the times of the four segsort_* kernels at
2^30; their bytes per element over those times are reported beside the HBM copy peak.  The card's name and power limit
are read in the same run (nvidia-smi --query-gpu, read only)."""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from bench_device_sort import COPY_PEAK_GBS, gpu_info, host_ms, make_keys, same  # noqa: E402

KEYS = {"u64": (torch.uint64, 0), "f64": (torch.float64, L.FLAG_KEY_F64)}
SHAPES = ["one", "rows1k", "width1k", "width32", "ragged"]
RAGGED_SEGMENTS = 1 << 16


def offsets_for(shape, n, device="cuda"):
    """(offsets, rows or None): rows is the row count of a 2-D shape"""
    rows = {"one": 1, "rows1k": 1 << 10, "width1k": n >> 10, "width32": n >> 5}.get(shape)
    if rows is not None:
        return torch.arange(rows + 1, dtype=torch.int64, device=device) * (n // rows), rows
    w = np.random.default_rng(3).lognormal(0.0, 1.0, RAGGED_SEGMENTS)
    sizes = np.floor(w / w.sum() * n).astype(np.int64)
    sizes[-1] += n - sizes.sum()
    return torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)])).to(device), None


def torch_arm(keys, vals, offsets, rows, seg_ids):
    if rows is not None:
        k, i = torch.sort(keys.view(rows, -1), dim=-1, stable=True)
        v = vals.view(rows, -1).gather(1, i) if vals is not None else i
        return k.reshape(-1), v.reshape(-1)
    _, i1 = torch.sort(keys, stable=True)
    _, i2 = torch.sort(seg_ids[i1], stable=True)
    perm = i1[i2]
    return keys[perm], (vals[perm] if vals is not None else perm)


def run_workload(s, n, kind, with_vals, shape, reps, floor):
    keys = make_keys(kind, n, 1)
    vals = make_keys("i64", n, 2).view(torch.int64) if with_vals else None
    offsets, rows = offsets_for(shape, n)
    local = rows is not None
    seg_ids = None
    if kind == "f64" and rows is None:
        seg_ids = torch.repeat_interleave(torch.arange(len(offsets) - 1, device="cuda"), offsets.diff())
    k_out, v_out = torch.empty_like(keys), (torch.empty_like(vals) if with_vals else torch.empty(n, dtype=torch.int64, device="cuda"))
    arms = {"segments": lambda: s.sort_segments(keys, offsets, vals, k_out, v_out, local_index=local)}
    if kind == "f64":
        arms["torch"] = lambda: torch_arm(keys, vals, offsets, rows, seg_ids)
    times = {a: [] for a in arms}
    dev_ms, st = [], None
    outs = {}
    for r in range(reps + 1):
        order = list(arms)[r % len(arms):] + list(arms)[:r % len(arms)]
        for a in order:
            t, out = host_ms(arms[a])
            if r:
                times[a].append(t)
            if a == "segments":
                st = out[2]
                if r:
                    dev_ms.append(st.device_ms)
            elif r == 0:
                outs[a] = out
            del out
    rec = {"n": n, "keys": kind, "vals": with_vals, "shape": shape, "segments": len(offsets) - 1,
           "ms": {a: statistics.median(v) for a, v in times.items()}, "segments_device_ms": statistics.median(dev_ms),
           "passes": st.passes, "skipped": st.skipped, "subpasses": st.subpasses, "kernel_launches": st.kernel_launches,
           "sort_device_ms": floor["ms"], "sort_device_device_ms": floor["device_ms"]}
    rec["ms_over_sort_device"] = rec["ms"]["segments"] / floor["ms"]
    equal = {}
    if "torch" in outs:
        tk, tv = outs.pop("torch")
        equal["torch"] = same(tk, k_out) and same(tv, v_out)
        rec["torch_over_segments"] = rec["ms"]["torch"] / rec["ms"]["segments"]
        del tk, tv
    if shape == "one":
        fk, fv, _ = s.sort_device(keys, vals)
        equal["sort_device"] = same(fk, k_out) and same(fv, v_out)
        del fk, fv
    rec["equal"] = equal
    del keys, vals, k_out, v_out, offsets, seg_ids
    torch.cuda.empty_cache()
    return rec


def floor_arm(s, n, kind, with_vals, reps):
    keys = make_keys(kind, n, 1)
    vals = make_keys("i64", n, 2).view(torch.int64) if with_vals else None
    k_out, v_out = torch.empty_like(keys), (torch.empty_like(vals) if with_vals else torch.empty(n, dtype=torch.int64, device="cuda"))
    ms, dev = [], []
    for r in range(reps + 1):
        t, out = host_ms(lambda: s.sort_device(keys, vals, k_out, v_out))
        if r:
            ms.append(t)
            dev.append(out[2].device_ms)
    del keys, vals, k_out, v_out
    return {"ms": statistics.median(ms), "device_ms": statistics.median(dev)}


def kernel_bytes(name, shape):
    """bytes each segsort kernel must move per element (check: per segment), read + write, in the profiled workloads:
    ragged with vals (the unpack gathers) and width-1k rows without vals (the unpack reads offsets[seg], L1/L2 hits)"""
    for kernel, b in (("check", 16), ("pack", 8 + 16), ("retag", 16 + 16)):
        if f"segsort_{kernel}_kernel" in name:
            return b
    return 16 + 8 + 8 + (8 if shape == "ragged" else 0)  # unpack: record, two outputs, the gather


def profile_kernels(n, out_dir):
    """torch.profiler over sort_segments at n, float64 keys: ragged with vals (gather) and width-1k rows (local index)"""
    from torch.profiler import ProfilerActivity, profile
    keys = make_keys("f64", n, 1)
    vals = make_keys("i64", n, 2).view(torch.int64)
    res = {}
    with lsb.DistributedSorter(n, ranks=1, flags=L.FLAG_KEY_F64) as s:
        for shape, v in (("ragged", vals), ("width1k", None)):
            offsets, rows = offsets_for(shape, n)
            s.sort_segments(keys, offsets, v, local_index=rows is not None)  # warm-up
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    s.sort_segments(keys, offsets, v, local_index=rows is not None)
                torch.cuda.synchronize()
            for e in prof.key_averages():
                if "segsort_" not in e.key:
                    continue
                total_us = getattr(e, "device_time_total", None)
                if total_us is None:
                    total_us = e.cuda_time_total
                ms = total_us / e.count / 1e3
                elems = len(offsets) - 1 if "check" in e.key else n
                b = kernel_bytes(e.key, shape)
                gbs = elems * b / (ms * 1e-3) / 1e9
                res[f"{shape}: {e.key}"] = {"ms_per_launch": ms, "launches": e.count, "elements": elems,
                                            "bytes_per_element": b, "gbs": gbs, "share_of_copy_peak": gbs / COPY_PEAK_GBS}
            if out_dir:
                prof.export_chrome_trace(os.path.join(out_dir, f"segments_{shape}.pt.trace.json"))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default="profiles/r5_segments.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2n", type=int, nargs="+", default=[28, 30])
    ap.add_argument("--trace-dir", default=None, help="write the profiled run's chrome traces here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_segments: no CUDA device")
    out = {"gpu": gpu_info(), "copy_peak_gbs": COPY_PEAK_GBS, "reps": args.reps, "workloads": []}
    for lg in args.log2n:
        n = 1 << lg
        for kind in KEYS:
            with lsb.DistributedSorter(n, ranks=1, flags=KEYS[kind][1]) as s:
                for with_vals in (False, True):
                    floor = floor_arm(s, n, kind, with_vals, args.reps)
                    for shape in SHAPES:
                        rec = run_workload(s, n, kind, with_vals, shape, args.reps, floor)
                        print(json.dumps(rec), flush=True)
                        out["workloads"].append(rec)
    out["kernels"] = profile_kernels(1 << max(args.log2n), args.trace_dir)
    out["all_equal"] = all(all(r["equal"].values()) for r in out["workloads"])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"kernels": out["kernels"], "all_equal": out["all_equal"]}, indent=1))


if __name__ == "__main__":
    main()
