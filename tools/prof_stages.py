#!/usr/bin/env python
"""Where a one-pass work item spends its time: needs the stage-clock build
(`make -C distributed-lsb_b200/csrc prof`), loaded through LSB_LIBRARY.
    LSB_LIBRARY=tools/bin/liblsbsort_prof.so python tools/prof_stages.py --log2n 28 [--tune op_t1=128]"""
import argparse
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
os.environ.setdefault("LSB_LIBRARY", os.path.join(ROOT, "tools", "bin", "liblsbsort_prof.so"))
sys.path.insert(0, ROOT)
import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

NAMES = {1: "dispatch (claim, slot wait, load issue)", 3: "K1 tile load", 7: "K1 rank + scan + write", 8: "K1 completion (warp 0)",
         11: "K2 piece table", 12: "K2 gather", 13: "K2 rank", 14: "K2 scan + frontier", 15: "K2 permutation", 20: "K2 scatter"}
ap = argparse.ArgumentParser()
ap.add_argument("--log2n", type=int, default=28)
ap.add_argument("--mhz", type=float, default=1965.0)
ap.add_argument("--tune", action="append", default=[])
ap.add_argument("--two-step", action="store_true", help="stage clocks of partition_kernel (default shape) instead")
a = ap.parse_args()
for kv in a.tune:
    k, v = kv.split("=")
    lsb.tune(k, int(v))
n = 1 << a.log2n
lib = lsb.load_library()
lib.lsb_debug_prof.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
PT_NAMES = ["ticket (atomic) + clear counters + barrier", "segment lookup + bulk-load issue + barrier", "wait for the tile (TMA)",
            "early counts (shared atomics) + barrier", "tile totals published, scan over bins + barrier", "ranks (ballots) -> permutation",
            "look-back (thread 0's bin)", "barrier after the look-back", "gather + stores issued"]
if a.two_step:
    with lsb.DistributedSorter(n, ranks=1, flags=L.FLAG_NO_SKIP) as s:
        out = (ctypes.c_uint64 * 56)()
        s.generate()
        s.my_sort()
        lib.lsb_debug_prof(s._ctx, out)
        s.generate()
        st = s.my_sort()
        lib.lsb_debug_prof(s._ctx, out)
        tiles = out[39]
        total = sum(out[24 + i] for i in range(9))
        print(f"n=2^{a.log2n}: sort {st.device_ms:.3f} ms, {st.partition_launches} partition launches, {tiles} tiles; "
              f"thread-0 clocks per tile {total / tiles / a.mhz:.2f} us")
        for i, name in enumerate(PT_NAMES):
            print(f"  {name:52s} {100.0 * out[24 + i] / total:6.2f} %   {out[24 + i] / tiles / a.mhz:7.3f} us per tile")
        print(f"  look-back of bin 0: {out[24 + 10] / tiles:.2f} round trips per tile"
              + (f", {out[24 + 9] / tiles / a.mhz:.3f} us per tile (walker thread)" if out[24 + 9] else ""))
    sys.exit(0)
with lsb.DistributedSorter(n, ranks=1, flags=L.FLAG_NO_SKIP | L.FLAG_ONE_PASS) as s:
    s.generate()
    s.my_sort()
    out = (ctypes.c_uint64 * 56)()
    lib.lsb_debug_prof(s._ctx, out)
    s.generate()
    st = s.my_sort()
    lib.lsb_debug_prof(s._ctx, out)
    ctas = out[23] / 4  # 4 passes
    total = sum(out[i] for i in range(21))
    print(f"n=2^{a.log2n}: sort {st.device_ms:.3f} ms; {ctas:.0f} CTAs; thread-0 clocks per CTA per pass "
          f"{total / out[23] / a.mhz / 1e3:.3f} ms")
    for i, name in NAMES.items():
        print(f"  {name:40s} {100.0 * out[i] / total:6.2f} %   {out[i] / out[23] / a.mhz:9.1f} us per CTA per pass")
