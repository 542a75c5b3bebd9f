#!/usr/bin/env python
"""The bucket pass (bucket_sort_kernel) of the one-GPU 64-bit sort: its launch time from LSB_FLAG_PHASE_EVENTS for
several builds alternated (one child process per build and round, LSB_LIBRARY), and where its time goes in the
stage-clock build (`make -C distributed-lsb_b200/csrc prof`).  Every sort is verified.
    python tools/bench_bucket.py --lib parent=/path/liblsbsort.so --lib branch=distributed-lsb_b200/liblsbsort.so \\
        --rounds 3 --log2n 30 31 22 [--stages tools/bin/liblsbsort_prof.so]
Inputs: `uniform` = the bench's generated keys (pcg64 streams); `fallback` = 2^28 uploaded keys whose top 3 bytes are
uniform, next 3 bytes constant and low 2 bytes random, so every chunk of the 32-bit keys has ties and is sorted again
by the 64-bit keys."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MHZ = 1965.0  # clock64() ticks per microsecond at the B200's boost clock (only scales the per-CTA figures)
STAGES = ["load wait", "boundary bits", "key build (ordinals, 32-bit keys)", "network (32-bit)", "tie check",
          "perm + gather + store", "64-bit fallback (tie check + whole 64-bit chunk)", "long bucket"]
BK_PROF0, NPROF = 40, 56  # BK_PROF0 / OP_NPROF of csrc/lsb_bucket.cuh / lsb_onepass.cuh


def fallback_keys(n, seed=5):
    import numpy as np
    rng = np.random.default_rng(seed)
    top = rng.integers(0, 1 << 24, size=n, dtype=np.uint64)
    return top << np.uint64(40) | np.uint64(0x5A5A5A << 16) | rng.integers(0, 1 << 16, size=n, dtype=np.uint64)


def child(a):
    sys.path.insert(0, ROOT)
    import numpy as np
    import distributed_lsb_b200 as lsb
    from distributed_lsb_b200 import lsbsort as L
    lib = lsb.load_library()
    prof = a.child_stages
    if prof:
        lib.lsb_debug_prof.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    flags = L.FLAG_NO_SKIP | L.FLAG_PHASE_EVENTS
    cases = [("uniform", x) for x in a.log2n] + ([("fallback", 28)] if a.fallback else [])
    for name, log2n in cases:
        n = 1 << log2n
        with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
            if name == "fallback":
                src = np.empty(n, dtype=L.ELT)
                src["key"] = fallback_keys(n)
                src["val"] = np.arange(n, dtype=np.uint64)
                want = np.sort(src["key"])
            out = (ctypes.c_uint64 * NPROF)()
            for it in range(a.warmup + a.iters):
                if name == "fallback":
                    s.upload(src)
                    st = s.my_sort()
                    got = s.download()
                    k, v = got["key"], got["val"]
                    tie = k[1:] == k[:-1]  # a stable sort keeps equal keys in input order
                    ok = bool((k == want).all() and (src["key"][v] == k).all() and (v[1:][tie] > v[:-1][tie]).all()
                              and (np.bincount(v.astype(np.int64), minlength=n) == 1).all())
                else:
                    s.generate()
                    before = s.checksum()
                    st = s.my_sort()
                    v = s.verify()
                    ok = list(v.checksum) == before and v.elements == n and not v.order_violations
                if prof:
                    lib.lsb_debug_prof(s._ctx, out)
                if it < a.warmup:
                    continue
                sub = [round(st.subpass_ms[i], 3) for i in range(min(st.partition_launches, L.LSB_MAX_SUBPASSES))]
                rec = {"lib": a.child_name, "input": name, "log2n": log2n, "iter": it - a.warmup,
                       "sort_ms": round(st.device_ms, 3), "hist_ms": round(st.hist_ms, 3), "launches_ms": sub,
                       "bucket_ms": sub[-1] if st.partition_launches < st.subpasses else None,
                       "subpasses": st.subpasses, "partition_launches": st.partition_launches, "verified": ok}
                if prof:
                    p = [out[BK_PROF0 + i] for i in range(12)]
                    total = sum(p[:8])
                    rec["ctas"], rec["chunks"], rec["fallback_chunks"], rec["long_buckets"] = p[8:12]
                    rec["fallback_rate"] = p[10] / max(p[9], 1)
                    rec["stages"] = {STAGES[i]: {"share": round(p[i] / max(total, 1), 4),
                                                 "us_per_cta": round(p[i] / max(p[8], 1) / MHZ, 3)} for i in range(8)}
                print(json.dumps(rec), flush=True)
                if not ok:
                    sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="name=path of a liblsbsort.so (alternated in this order)")
    ap.add_argument("--stages", default="", help="stage-clock build to report the stage split with (after the A/B)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--log2n", type=int, nargs="+", default=[30])
    ap.add_argument("--no-fallback", dest="fallback", action="store_false", help="skip the every-chunk-falls-back input")
    ap.add_argument("--child-name", default="")
    ap.add_argument("--child-stages", action="store_true")
    a = ap.parse_args()
    if a.child_name:
        return child(a)
    common = ["--iters", str(a.iters), "--warmup", str(a.warmup), "--log2n", *map(str, a.log2n)]
    if not a.fallback:
        common.append("--no-fallback")
    runs = [(name, path, []) for name, path in (x.split("=", 1) for x in a.lib)]
    plan = [r for _ in range(a.rounds) for r in runs]
    if a.stages:
        plan.append(("stages", a.stages, ["--child-stages"]))
    for name, path, extra in plan:
        env = dict(os.environ, LSB_LIBRARY=os.path.abspath(path))
        subprocess.run([sys.executable, os.path.abspath(__file__), "--child-name", name, *common, *extra], env=env,
                       check=True)


if __name__ == "__main__":
    main()
