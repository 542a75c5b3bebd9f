#!/usr/bin/env python
"""Every sorting entry point on seeded inputs, dumped as a digest of each call's output bytes beside its stats: run it
once with each of two builds of liblsbsort.so (LSB_LIBRARY, one process each) and compare the dumps. They are
identical when a change leaves what the library computes, and the launches it makes, as they were.

    LSB_LIBRARY=a/liblsbsort.so python tools/same_results.py --out a.txt
    LSB_LIBRARY=b/liblsbsort.so python tools/same_results.py --out b.txt
    cmp a.txt b.txt

For each key type (uint64, int64, float64, float32, int32, bfloat16), order (ascending, descending), pass shape
(default, one-pass, two-level) and radix (8, 13, 16), one sorter of 2^20 + 7 keys runs in turn: sort_device without and
with vals, sort_segments over one segment, over rows of 2^10 (local index) and over ragged segments (vals gathered), an
upload / my_sort / download of 16-byte records, an upload / global_shuffle(0) / download, then num_passes and
digit_bits. lsb.sort (2^10 rows) and lsb.argsort (1-D) run once per key type and order. A line of the dump is one call:
the first 16 hex digits of the sha256 of its outputs' bytes, then passes, subpasses, skipped, elements,
kernel_launches, partition_launches and partition_elements."""
import argparse
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import narrow_keys as NK  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

N = (1 << 20) + 7
WIDE = {"uint64": 0, "int64": L.FLAG_KEY_I64, "float64": L.FLAG_KEY_F64}
NAMES = ["uint64", "int64", "float64", "float32", "int32", "bfloat16"]
SHAPES = {"default": 0, "one_pass": L.FLAG_ONE_PASS, "two_level": L.FLAG_TWO_LEVEL}
RADICES = [8, 13, 16]
STATS = ["passes", "subpasses", "skipped", "elements", "kernel_launches", "partition_launches", "partition_elements"]


def keys_of(name, seed):
    if name in WIDE:
        return torch.from_numpy(KO.special_mix(N, seed=seed).view(np.int64)).cuda().view(getattr(torch, name))
    return NK.to_device(torch, NK.special_mix(N, name, seed=seed), name)


def digest(outputs):
    h = hashlib.sha256()
    for t in outputs:
        if isinstance(t, torch.Tensor):
            t = t.contiguous().view(torch.uint8).cpu().numpy()
        h.update(np.ascontiguousarray(t).tobytes())
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    rng = np.random.default_rng(20)
    vals = torch.from_numpy(rng.integers(0, 1 << 62, N)).cuda()
    recs = np.empty(N, dtype=L.ELT)
    recs["key"] = KO.special_mix(N, seed=21)
    recs["val"] = np.arange(N)
    segmentations = {
        "one": (np.array([0, N]), {}),
        "rows": (np.append(np.arange(0, N, 1 << 10), N), {"local_index": True}),
        "ragged": (np.concatenate([[0], np.sort(rng.integers(0, N, 999)), [N]]), {"vals": vals}),
    }
    segmentations = {k: (torch.from_numpy(o.astype(np.int64)).cuda(), kw) for k, (o, kw) in segmentations.items()}
    lines = []

    def put(what, outputs, st=None):
        stats = [f"{f}={getattr(st, f)}" for f in STATS] if st is not None else []
        lines.append(" ".join([what, digest(outputs)] + stats))

    for i, name in enumerate(NAMES):
        keys = keys_of(name, 30 + i)
        key_dtype = None if name in WIDE else getattr(torch, name)
        for desc in (False, True):
            order = "desc" if desc else "asc"
            for shape, shape_flags in SHAPES.items():
                for radix in RADICES:
                    tag = f"{name} {order} {shape} r{radix}"
                    flags = WIDE.get(name, 0) | shape_flags | (L.FLAG_DESCENDING if desc else 0)
                    with lsb.DistributedSorter(N, ranks=1, radix_bits=radix, flags=flags, key_dtype=key_dtype) as s:
                        k, v, st = s.sort_device(keys)
                        put(f"{tag} sort_device", (k, v), st)
                        k, v, st = s.sort_device(keys, vals)
                        put(f"{tag} sort_device+vals", (k, v), st)
                        for seg, (offsets, kw) in segmentations.items():
                            k, v, st = s.sort_segments(keys, offsets, **kw)
                            put(f"{tag} sort_segments/{seg}", (k, v), st)
                        s.upload(recs)
                        st = s.my_sort()
                        put(f"{tag} my_sort", (s.download(),), st)
                        s.upload(recs)
                        st = s.global_shuffle(0)
                        put(f"{tag} global_shuffle(0)", (s.download(),), st)
                        lines.append(f"{tag} plan {s.num_passes()} {[s.digit_bits(d) for d in range(s.num_passes())]}")
            r = lsb.sort(keys[:1 << 20].view(1 << 10, 1 << 10), dim=-1, descending=desc)
            put(f"{name} {order} lsb.sort rows", (r.values, r.indices))
            put(f"{name} {order} lsb.argsort", (lsb.argsort(keys, descending=desc),))
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print(f"{len(lines)} calls -> {args.out}")


if __name__ == "__main__":
    main()
