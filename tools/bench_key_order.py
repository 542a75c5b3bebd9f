#!/usr/bin/env python
"""Cost of the key orders (LSB_FLAG_KEY_I64 / KEY_F64 / DESCENDING) on one GPU, alternating the orders so that drift
of the shared machine spreads over all of them.

    python tools/bench_key_order.py --out profiles/r3_key_order_2p30.json [--reps 5]

Workloads: 2^30 pcg64 keys made on the device (read as uint64, int64, float64, float64 descending), and 2^28
standard-normal doubles uploaded from the host (a narrow exponent range: the high digits are nearly constant).  Each
(workload, order, shape) gets one warm-up sort and `reps` timed sorts; the round-robin visits every configuration once
per round.  Every sort is verified on the device (order and multiset checksum).  A context holds two 16 GiB shards at
2^30, so each sort runs in its own context.  The card's name, power limit and max SM clock are read in the same run
(nvidia-smi --query-gpu, read only)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

ORDERS = {"u64": 0, "i64": L.FLAG_KEY_I64, "f64": L.FLAG_KEY_F64, "f64_desc": L.FLAG_KEY_F64 | L.FLAG_DESCENDING}
SHAPES = {"default": 0, "one_pass": L.FLAG_ONE_PASS}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def one_sort(n, flags, host=None):
    with lsb.DistributedSorter(n, ranks=1, flags=flags | L.FLAG_PHASE_EVENTS) as s:
        if host is None:
            s.generate()
        else:
            s.upload(host)
        before = s.checksum()
        st = s.my_sort()
        v = s.verify(raise_on_failure=False)
        ok = v.order_violations == 0 and v.elements == n and list(v.checksum) == before
        return {"device_ms": st.device_ms, "hist_ms": st.hist_ms, "partition_ms": st.partition_ms,
                "launches": st.partition_launches, "skipped": st.skipped, "verified": ok,
                "subpass_ms": [round(x, 4) for x in st.subpass_ms[:min(st.partition_launches, L.LSB_MAX_SUBPASSES)]]}


def summary(runs):
    def med_spread(xs):
        return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4)}
    return {"device_ms": med_spread([r["device_ms"] for r in runs]),
            "hist_ms": med_spread([r["hist_ms"] for r in runs]),
            "partition_ms_per_launch": med_spread([r["partition_ms"] / max(r["launches"], 1) for r in runs]),
            "launches": runs[0]["launches"], "skipped": runs[0]["skipped"],
            "verified": all(r["verified"] for r in runs), "timed_sorts": len(runs),
            "subpass_ms_last": runs[-1]["subpass_ms"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--log2n", type=int, default=30)
    ap.add_argument("--log2n-upload", type=int, default=28)
    args = ap.parse_args()
    info = gpu_info()
    n_gen, n_up = 1 << args.log2n, 1 << args.log2n_upload
    host = np.zeros(n_up, dtype=L.ELT)
    host["key"] = np.random.default_rng(0).standard_normal(n_up).view(np.uint64)
    host["val"] = np.arange(n_up, dtype=np.uint64)
    work = {f"generated_2p{args.log2n}": (n_gen, None), f"normal_doubles_2p{args.log2n_upload}": (n_up, host)}
    configs = [(w, o, sh) for w in work for o in ORDERS for sh in SHAPES]
    runs = {c: [] for c in configs}
    t0 = time.time()
    for rnd in range(args.reps + 1):  # round 0 is the warm-up of every configuration
        for c in configs:
            w, o, sh = c
            n, h = work[w]
            r = one_sort(n, ORDERS[o] | SHAPES[sh], h)
            if not r["verified"]:
                raise SystemExit(f"verification failed: {c}")
            if rnd:
                runs[c].append(r)
            print(f"round {rnd} {w} {o} {sh}: {r['device_ms']:.3f} ms", flush=True)
    res = {"gpu": info, "reps": args.reps, "wall_s": round(time.time() - t0, 1),
           "note": "device_ms with LSB_FLAG_PHASE_EVENTS (one event per kernel); default skipping of constant digits",
           "results": [{"workload": w, "order": o, "shape": sh, **summary(runs[(w, o, sh)])} for w, o, sh in configs]}
    for w in work:
        for sh in SHAPES:
            base = next(r for r in res["results"] if r["workload"] == w and r["order"] == "u64" and r["shape"] == sh)
            for r in res["results"]:
                if r["workload"] == w and r["shape"] == sh:
                    r["vs_u64"] = round(r["device_ms"]["median"] / base["device_ms"]["median"], 4)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in res["results"]:
        print(json.dumps({k: r[k] for k in ("workload", "order", "shape", "device_ms", "partition_ms_per_launch",
                                             "vs_u64", "verified")}))


if __name__ == "__main__":
    main()
