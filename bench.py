#!/usr/bin/env python
"""bench.py -- headline benchmark: M 16-byte elements sorted / s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU path
    torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU

A "step" is one full mySort (all passes) over one freshly generated synthetic input.
  N = 1 : BASELINE configs[1] -- single B200, n = 2^30 uniform pcg64 keys, 16-bit digits.
  N > 1 : BASELINE configs[2] weak scaling -- 2^31 elements per GPU, R = N pcg64 streams.
  --strong        configs[2] strong scaling: n = 2^33 in total at N = 4/8, 2^32 at N = 1/2 (2^33 does not fit)
  --key-mask / --and-draws   configs[3] skewed keys;  --radix 8|11|16   configs[4] digit-width sweep
Constant-digit passes are NOT skipped in the measured line (the reference always runs them); a skewed
run also reports the skipping variant as `skip_variant`.
`value` is device time (CUDA events on the sort stream, inputs already in HBM, max over ranks);
`e2e` is the same metric through the host-buffer C-ABI call lsb_sort_host (pinned host memory
in, pinned host memory out, copies inside the timed region, wall clock); `e2e.overlapped` (N = 1)
is two sorters fed from two threads, so one batch's copy in shares the link with another's copy out.
`--dump-outputs DIR` writes a fixed sample of the last timed step's sorted output as .npy files (see dump_outputs),
so that two builds run with the same arguments can be compared output for output.
`cpu_baseline` and --impl reference need oracle/_ref, which oracle/build_ref.sh builds only where the reference's
source is present; without it `cpu_baseline.value` is null.
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "M 16-byte elements sorted/s"
ALL_BITS = 0xFFFFFFFFFFFFFFFF
UNIT = "M elements/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period_ms=100):
        self.device, self.rows, self.proc, self.period_ms = device, [], None, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms), "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the UNMODIFIED mpi_lsbsort.cpp (oracle/_ref, ranks = threads)
# --------------------------------------------------------------------------------------
def reference_binary():
    """path of the reference program oracle/build_ref.sh builds, or None: it needs the reference's source,
    which the repository does not contain, and bench.py never compiles into the tree itself"""
    from oracle import oracle as O  # the one place bench.py may execute oracle/: the CPU baseline
    return O.REF_BIN if os.path.exists(O.REF_BIN) else None


def run_reference_once(n, ranks):
    from oracle import oracle as O
    env = dict(os.environ, SHIM_RANKS=str(ranks))
    out = subprocess.run([O.REF_BIN, "--n", str(n), "--no-verify"], env=env, check=True, capture_output=True,
                         text=True).stdout
    m = re.search(r"That's ([0-9.eE+-]+) M elements sorted / s", out)
    s = re.search(r"Sorted \d+ values in ([0-9.eE+-]+)", out)
    return float(m.group(1)), float(s.group(1))


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline(sample_log2=None):
    """bounded sample of the same workload on the host cores; ~10-30 s of CPU work"""
    cores = host_threads()
    ranks = max(1, min(cores, 64))
    if reference_binary() is None:
        return {"value": None, "unit": UNIT, "kind": "reference",
                "note": "not measured: the reference program oracle/_ref/mpi_lsbsort_shim is not built "
                        "(oracle/build_ref.sh needs the reference's source)"}
    n = 1 << (sample_log2 or 24)
    rate, secs = run_reference_once(n, ranks)
    if sample_log2 is None and secs < 1.5:  # fast host: take a bigger, steadier sample (~10-20 s of CPU work)
        n = 1 << 28
        rate, secs = run_reference_once(n, ranks)
    return {"value": rate, "unit": UNIT, "cores": ranks, "kind": "reference",
            "sample": f"unmodified mpi/mpi_lsbsort.cpp over the ranks-as-threads mpi.h shim (oracle/_ref), "
                      f"{ranks} ranks, n=2^{n.bit_length() - 1} --no-verify, {secs:.2f} s sort time"}


def bench_shape(args, world):
    """(elements per GPU as log2, n total, scaling) of the workload both arms report"""
    if args.strong:
        total_log2 = args.strong_log2 or (33 if world >= 4 else 32)
        per = total_log2 - (world.bit_length() - 1)
        return per, 1 << total_log2, "strong"
    per = args.log2n if args.log2n else (30 if world == 1 else 31)
    return per, world << per, "weak"


DUMP_ELEMENTS = 1 << 20  # in all ranks together: 4 float64 arrays of this length are 32 MiB
DUMP_BLOCKS = 1024
DUMP_SEED = 20261020


def dump_outputs(sorter, out_dir, rank, world):
    """--dump-outputs: the sorted shard the last timed step left on this GPU, as a fixed sample.

    A shard with more than DUMP_ELEMENTS / world elements is sampled as DUMP_BLOCKS contiguous blocks, one at a
    seeded offset inside each of DUMP_BLOCKS equal strata; the offsets depend on the shard size only, so two builds
    run with the same arguments dump the same positions.  Written as float64, which holds every value exactly:
    index.npy (global position), key_hi.npy / key_lo.npy (upper and lower 32 bits of the key), val.npy.
    With several GPUs each rank writes rank<r>_<name>.npy for its shard."""
    import numpy as np
    here, want = sorter.here, DUMP_ELEMENTS // world
    if here <= want:
        starts, blen = np.array([0], dtype=np.int64), here
    else:
        blen = want // DUMP_BLOCKS
        stratum = here // DUMP_BLOCKS
        rng = np.random.default_rng([DUMP_SEED, here])
        starts = np.arange(DUMP_BLOCKS, dtype=np.int64) * stratum + rng.integers(0, stratum - blen + 1, DUMP_BLOCKS)
    elts = np.concatenate([sorter.download(local_off=int(s), count=blen) for s in starts])
    index = (sorter.first_global + starts[:, None] + np.arange(blen, dtype=np.int64)[None, :]).reshape(-1)
    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    for name, a in (("index", index), ("key_hi", elts["key"] >> np.uint64(32)),
                    ("key_lo", elts["key"] & np.uint64(0xFFFFFFFF)), ("val", elts["val"])):
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a.astype(np.float64))


def config_dict(args, world, n, here, npass):
    return {"workload": workload_name(world, args), "n_total": n, "n_per_gpu": here, "radix_bits": args.radix,
            "passes": npass, "pcg_streams": world, "key_mask": hex(args.key_mask), "and_draws": args.and_draws,
            "skip_constant_digits": False, "one_pass_kernel": bool(args.one_pass),
            "l2": "inputs (16-64 GiB per GPU) are far larger than the 126 MB L2; no flush needed"}


def main_reference(args, rank):
    if rank != 0:
        return 0
    if reference_binary() is None:
        raise SystemExit("bench.py --impl reference: oracle/_ref/mpi_lsbsort_shim is not built "
                         "(oracle/build_ref.sh needs the reference's source)")
    world = args.gpus
    cores = host_threads()
    ranks = max(1, min(cores, 64))
    per_log2, n_total, scaling = bench_shape(args, world)
    n = 1 << args.ref_log2
    for _ in range(args.warmup and 1):
        run_reference_once(n, ranks)
    rates, secs = [], []
    for _ in range(args.steps):
        r, s = run_reference_once(n, ranks)
        rates.append(r)
        secs.append(s)
    value = n * len(secs) / sum(secs) / 1e6
    npass = -(-64 // args.radix)
    sample = (f"unmodified mpi/mpi_lsbsort.cpp via oracle/_ref (ranks-as-threads mpi.h shim, no MPI on the box), {ranks} ranks "
              f"on {cores} host threads, each step = a 2^{args.ref_log2}-element sample of the workload, --no-verify, uniform keys, "
              f"16-bit digits (the reference has neither a skew nor a radix knob)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs),
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_dict(args, world, n_total, n_total // world, npass),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ranks, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_name(gpus, args):
    per_log2, n, scaling = bench_shape(args, gpus)
    keys = "uniform-random"
    if args.key_mask != ALL_BITS or args.and_draws > 1:
        keys = f"skewed (configs[3]: key = AND of {args.and_draws} pcg64 draws & {hex(args.key_mask)})"
    npass = -(-64 // args.radix)
    what = f"{keys} 16-byte elements, {args.radix}-bit digits ({npass} passes)"
    if scaling == "strong":
        return f"configs[2] strong scaling: {gpus}xB200, 2^{n.bit_length() - 1} elements in total, {what}"
    if gpus == 1:
        tag = "configs[1]" if (per_log2 == 30 and args.radix == 16 and keys == "uniform-random") else "single-GPU point"
        return f"{tag}: single B200, 2^{per_log2} {what}"
    tag = "configs[4] digit-width sweep" if args.radix != 16 else "configs[2] weak scaling"
    return f"{tag}: {gpus}xB200, 2^{per_log2} elements per GPU, {what}"


# --------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------
def main_cuda(args, rank, world, local_rank, own_process_group=True, tag=None):
    import torch
    import torch.distributed as dist
    import distributed_lsb_b200 as lsb
    from distributed_lsb_b200 import lsbsort as L

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1 and own_process_group:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    per_gpu_log2, n, scaling = bench_shape(args, world)
    for kv in args.tune:
        k_, v_ = kv.split("=")
        lsb.tune(k_, int(v_))

    def make_sorter(n_total, flags, skip=False, one_pass=None):
        one_pass = args.one_pass if one_pass is None else one_pass
        s_ = lsb.DistributedSorter(n_total, ranks=world, world_size=world, world_rank=rank, device=local_rank,
                                   radix_bits=args.radix, key_mask=args.key_mask, and_draws=args.and_draws,
                                   flags=flags | (0 if skip else L.FLAG_NO_SKIP) | (L.FLAG_ONE_PASS if one_pass else 0))
        if world > 1:
            ids = [lsb.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            s_.comm_init(ids[0])
        return s_

    sorter = make_sorter(n, L.FLAG_PHASE_EVENTS if args.phases else 0)

    # ---- warm-up (also the correctness gate: a wrong sort is not a benchmark) ----
    # mpi/mpi_lsbsort.cpp:722-736: the output must be the stable sort of the input.  On every rank:
    # (key,val) strictly increasing within and across shards, n elements, and the GLOBAL multiset
    # hash (all-gathered by lsb_verify_device) unchanged by the sort -- for any world size.
    for w in range(args.warmup):
        sorter.generate()
        before = sorter.verify(raise_on_failure=False) if w == 0 else None
        sorter.my_sort()
        if w == 0:
            v = sorter.verify()
            if list(v.checksum) != list(before.checksum) or v.elements != n or before.elements != n:
                raise SystemExit(f"bench.py: rank {rank}: the sort changed the multiset of elements "
                                 f"({v.elements} of {n} elements, hash {list(v.checksum)} vs {list(before.checksum)})")

    # ---- timed: exactly K steps, device time per step, max over ranks ----
    sampler = ClockSampler(local_rank, args.clock_period_ms)
    step_ms, launches, part_ms, part_launches = [], 0, 0.0, 0
    if rank == 0:
        sampler.start()
    try:  # the nvidia-smi sampler must not outlive a failed step
        for _ in range(args.steps):
            sorter.generate()          # fresh input, resident in HBM before the timed region
            barrier()
            st = sorter.my_sort()      # CUDA events bracket the kernels on the sort stream
            barrier()
            step_ms.append(max_over_ranks(st.device_ms))
            launches += st.kernel_launches
            part_ms += st.partition_ms
            part_launches += st.partition_launches
    finally:
        clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(sorter, args.dump_outputs, rank, world)
    total_s = sum(step_ms) / 1e3
    value = n * args.steps / total_s / 1e6

    # ---- per-kernel durations for the roofline (phase events; separate, untimed-for-value step) ----
    sorter.close()
    skip_variant = None
    if args.key_mask != ALL_BITS or args.and_draws > 1:  # the same workload with constant-digit passes skipped
        sk = make_sorter(n, 0, skip=True)
        sk_ms, sk_skipped = [], 0
        for i in range(1 + min(args.steps, 3)):
            sk.generate()
            barrier()
            st = sk.my_sort()
            barrier()
            if i:
                sk_ms.append(max_over_ranks(st.device_ms))
            sk_skipped = st.skipped
        sk.close()
        skip_variant = {"value": n / (statistics.mean(sk_ms) / 1e3) / 1e6, "unit": UNIT, "ms_per_step": statistics.mean(sk_ms),
                        "passes_skipped": sk_skipped}
    alt_path = None
    if world == 1 and not args.no_alt:  # the other pass shape on the same workload, for the record
        alt = make_sorter(n, L.FLAG_PHASE_EVENTS, one_pass=not args.one_pass)
        alt_ms, alt_launch = [], []
        for i in range(1 + min(args.steps, 3)):
            alt.generate()
            before_alt = alt.checksum()
            st = alt.my_sort()
            if i == 0 and list(alt.verify().checksum) != before_alt:
                raise SystemExit("bench.py: alternative pass shape: multiset hash changed across the sort")
            if i:
                alt_ms.append(st.device_ms)
                alt_launch.append(st.partition_ms / max(st.partition_launches, 1))
        alt.close()
        tname = "onepass_traffic.json" if not args.one_pass else "partition_traffic.json"
        tfile = os.path.join(ROOT, "profiles", tname)
        per_elem = None
        if os.path.exists(tfile):
            with open(tfile) as f:
                per_elem = json.load(f).get("dram_bytes_per_element")
        alt_path = {"path": "two 8-bit steps per pass (default)" if args.one_pass else "LSB_FLAG_ONE_PASS (one-pass kernel)",
                    "value": n / (statistics.mean(alt_ms) / 1e3) / 1e6, "unit": UNIT, "ms_per_step": statistics.mean(alt_ms),
                    "scatter_launch_ms": statistics.mean(alt_launch), "ncu_dram_bytes_per_element_per_launch": per_elem}
    sorter = make_sorter(n, L.FLAG_PHASE_EVENTS)
    kp_ms, kp_n, hist_ms = [], 0, []
    for _ in range(max(2, min(args.steps, 3))):
        sorter.generate()
        barrier()
        st = sorter.my_sort()
        kp_ms.append(st.partition_ms / max(st.partition_launches, 1))
        kp_n = st.partition_launches
        kp_elems = st.partition_elements / max(st.partition_launches, 1)  # elements per launch (a part when G > 1)
        hist_ms.append(st.hist_ms)
        exch_ms = st.exchange_ms
    peak, peak_src = _peaks()
    here = sorter.here
    launch_ms = statistics.mean(kp_ms)
    achieved = kp_elems * 32 / (launch_ms * 1e-3) / 1e9
    npass = sorter.num_passes()
    sort_ms = statistics.mean(step_ms)
    # SURVEY 8(d): t_pass >= max(m*32 B / BW_hbm, m*16 B*f_remote / BW_nvlink); NVLink denominator =
    # the measured peer-copy figure of B200_PROFILING.md (770 GB/s per direction per GPU, 900 nominal)
    nvlink_gbs = 770.0
    f_remote = lsb.hostlogic.remote_fraction(list(st.sent[:world]), rank) if world > 1 else 0.0
    t_pass_min = lsb.hostlogic.pass_roofline_ms(here, f_remote, peak, nvlink_gbs)
    pass_bound = "hbm" if here * 32 / (peak * 1e9) >= here * 16 * f_remote / (nvlink_gbs * 1e9) else "nvlink"
    pass_frac = t_pass_min * npass / sort_ms
    traffic = None
    if args.one_pass and args.radix > 8:
        kernel_name = "lsb::onepass_kernel (one stable scatter on a 9..16-bit digit = one reference pass per launch)"
        tp = os.path.join(ROOT, "profiles", "onepass_traffic.json")
    else:
        kernel_name = ("lsb::partition_kernel (one stable counting-sort step on <= 8 bits; "
                       + ("two launches" if args.radix > 8 else "one launch") + " per reference pass)")
        tp = os.path.join(ROOT, "profiles", "partition_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get("dram_bytes_per_element", 0) * kp_elems or None  # per launch

    # ---- end to end through the host-buffer C-ABI entry point ----
    # Every rank pins an input and an output buffer for its whole shard; if the host cannot hold
    # 2 x 16 B x n (8 ranks x 2^31 elements = 512 GiB), the e2e leg drops to the largest power of two
    # per GPU that fits and says so.
    e2e = None
    if not args.no_e2e:
        def mem_available():
            try:
                with open("/proc/meminfo") as f:
                    for line in f:
                        if line.startswith("MemAvailable:"):
                            return int(line.split()[1]) * 1024
            except OSError:
                pass
            return 1 << 62
        e2e_log2 = per_gpu_log2
        while e2e_log2 > 20 and 2 * 16 * (world << e2e_log2) * 1.15 > mem_available():
            e2e_log2 -= 1
        if world > 1:  # all ranks must agree
            t = torch.tensor([e2e_log2], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            e2e_log2 = int(t.item())
        es = sorter
        if e2e_log2 != per_gpu_log2:
            sorter.close()
            es = sorter = make_sorter(world << e2e_log2, 0)
        e_n, e_here = world << e2e_log2, es.here
        es.generate()
        hin, hout = L.PinnedBuffer(e_here), L.PinnedBuffer(e_here)
        es.download(out=hin.array)
        walls = []
        for i in range(1 + args.e2e_steps):
            barrier()
            t0 = time.perf_counter()
            es.sort_host(hin.array, hout.array)
            barrier()
            if i:  # first one is warm-up
                walls.append(max_over_ranks(time.perf_counter() - t0))
        chk = min(e_here, 1 << 20)
        ok = bool((hout.array["key"][:chk][:-1] <= hout.array["key"][:chk][1:]).all())
        e2e = {"value": e_n / statistics.mean(walls) / 1e6, "unit": UNIT, "h2d_bytes_per_step": e_here * 16 * world,
               "d2h_bytes_per_step": e_here * 16 * world, "ms_per_step": 1e3 * statistics.mean(walls),
               "api": "lsb_sort_host (pinned host in/out)", "output_sorted": ok, "n_total": e_n}
        if e2e_log2 != per_gpu_log2:
            e2e["note"] = f"host memory holds 2^{e2e_log2} elements per GPU for the pinned in/out buffers, not 2^{per_gpu_log2}"
        # One lsb_sort_host call is H2D -> sort -> D2H back to back and nothing of it can overlap (the
        # first scatter needs every input element, the copy out needs the last scatter), so a single
        # sorter is bound by the two PCIe copies.  A caller with a stream of batches runs TWO sorters
        # from two threads: the copy in of one batch then shares the (full-duplex) link with the copy
        # out of the other.  Reported beside `e2e`, never instead of it; the time includes filling and
        # draining the two-deep pipeline.
        if (world == 1 and not args.no_e2e_overlap and 3 * 16 * e_here * 1.15 < mem_available()
                and 2 * (2 * 16 * e_here) * 1.1 < torch.cuda.get_device_properties(local_rank).total_memory):
            es2 = make_sorter(e_n, 0)
            hout2 = L.PinnedBuffer(e_here)
            errors = []

            def stream_of_batches(s_, out, k):
                try:
                    for _ in range(k):
                        s_.sort_host(hin.array, out.array)
                except Exception as ex:  # surfaced below, the bench must not hang on a dead thread
                    errors.append(repr(ex))

            es2.sort_host(hin.array, hout2.array)  # warm-up of the second sorter
            k = 1 + args.e2e_steps
            threads = [threading.Thread(target=stream_of_batches, args=(es, hout, k)),
                       threading.Thread(target=stream_of_batches, args=(es2, hout2, k))]
            t0 = time.perf_counter()
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            wall = time.perf_counter() - t0
            if errors:
                raise SystemExit(f"bench.py: overlapped e2e leg failed: {errors}")
            same = bool((hout.array[:chk] == hout2.array[:chk]).all()) and \
                bool((hout.array[-chk:] == hout2.array[-chk:]).all())
            e2e["overlapped"] = {"value": 2 * k * e_n / wall / 1e6, "unit": UNIT, "ms_per_step": 1e3 * wall / (2 * k),
                                 "sorts": 2 * k, "sorters": 2, "h2d_bytes_per_step": e_here * 16, "d2h_bytes_per_step": e_here * 16,
                                 "outputs_identical": same,
                                 "api": "two lsb contexts on one GPU, each calling lsb_sort_host from its own thread "
                                        "(wall clock over all sorts, pipeline fill and drain included)"}
            hout2.free()
            es2.close()
        hin.free()
        hout.free()
    sorter.close()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sort_ms, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_dict(args, world, n, here, npass),
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches,
            # SURVEY 8(d): frac = (slower of 32 B/element of HBM traffic and 16 B x f_remote of NVLink traffic per
            # reference pass) / measured time per pass, over the WHOLE sort (counts, scans, scatters, exchange)
            "roofline": {"bound": pass_bound, "achieved": (here * 32 if pass_bound == "hbm" else here * 16 * f_remote) * npass
                         / (sort_ms * 1e-3) / 1e9,
                         "peak": peak if pass_bound == "hbm" else nvlink_gbs, "unit": "GB/s", "frac": pass_frac,
                         "peak_source": peak_src if pass_bound == "hbm" else "B200_PROFILING.md peer-copy figure (770 GB/s per direction)",
                         "t_pass_min_ms": t_pass_min, "t_pass_ms": sort_ms / npass, "f_remote": f_remote,
                         "hbm_gbs": peak, "nvlink_gbs": nvlink_gbs,
                         "algorithmic_bytes_per_pass_hbm": here * 32,
                         "algorithmic_bytes_per_pass_nvlink": here * 16 * f_remote,
                         "kernel": kernel_name, "launch_ms": launch_ms, "launches_per_sort": kp_n,
                         "algorithmic_bytes_per_launch": kp_elems * 32, "launch_gbs": achieved,
                         "launch_frac": achieved / peak, "traffic": traffic,
                         "note": "frac is the per-pass fraction of SURVEY 8(d) over the whole step; launch_frac is the "
                                 "dominant kernel alone (32 B/element per launch / its CUDA-event duration / HBM peak); "
                                 "traffic = ncu dram bytes of one launch of that kernel (profiles/partition_traffic.json or "
                                 "profiles/onepass_traffic.json, scaled to the launch's elements)"},
            "hist_ms_per_sort": statistics.mean(hist_ms),
            "exchange_kernel_ms_per_sort": exch_ms,
        }
        if skip_variant:
            line["skip_variant"] = skip_variant
        if alt_path:
            line["alt_path"] = alt_path
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        if tag:
            line = dict({"suite": tag}, **line)
        print(json.dumps(line), flush=True)
    if world > 1 and own_process_group:
        dist.destroy_process_group()
    return 0


def main_suite(args, rank, world, local_rank, parser):
    """several configurations in ONE set of processes (a multi-GPU box is charged per GPU-minute: import, NCCL and
    rendezvous are paid once).  --suite 'weak:;strong:--strong;mask24:--key-mask 0xFFFFFF --no-e2e;...'"""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rc = 0
    for item in filter(None, (x.strip() for x in args.suite.split(";"))):
        name, _, extra = item.partition(":")
        sub = parser.parse_args(["--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)] + extra.split())
        try:
            main_cuda(sub, rank, world, local_rank, own_process_group=False, tag=name)
        except SystemExit as e:  # keep going: the other configurations are still worth their GPU time
            if rank == 0:
                print(json.dumps({"suite": name, "error": str(e)}), flush=True)
            rc = 1
    if world > 1:
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--log2n", type=int, default=0, help="log2 elements per GPU (default 30 at N=1, 31 at N>1)")
    ap.add_argument("--radix", type=int, default=16)
    ap.add_argument("--phases", action="store_true", help="record per-kernel events inside the timed steps too")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e-overlap", action="store_true", help="skip the two-sorter overlapped e2e leg (N = 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-log2", type=int, default=28, help="--impl reference: log2 of the per-step sample")
    ap.add_argument("--strong", action="store_true", help="strong scaling: fixed total (2^33 at 4/8 GPUs, 2^32 at 1/2)")
    ap.add_argument("--strong-log2", type=int, default=0, help="override the fixed total of --strong")
    ap.add_argument("--key-mask", type=lambda x: int(x, 0), default=ALL_BITS, help="configs[3]: keep only these key bits")
    ap.add_argument("--and-draws", type=int, default=1, help="configs[3]: key = AND of k pcg64 draws (Zipf-like digits)")
    ap.add_argument("--tune", action="append", default=[], help="key=value for lsb_tune (experiments)")
    ap.add_argument("--one-pass", action="store_true", help="measure LSB_FLAG_ONE_PASS (the one-pass kernel) as the main path")
    ap.add_argument("--no-alt", action="store_true", help="skip the short run of the other pass shape (N = 1)")
    ap.add_argument("--clock-period-ms", type=int, default=100, help="nvidia-smi sampling period during the timed region")
    ap.add_argument("--suite", default="", help="'name:flags;name:flags;...': several configurations in one launch, one JSON line each")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the last step's sorted output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.suite:
        ap.error("--dump-outputs writes one configuration's outputs; it does not combine with --suite")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1 and args.impl == "cuda":
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.impl == "reference":
        return main_reference(args, rank)
    try:
        if args.suite:
            return main_suite(args, rank, world, local_rank, ap)
        return main_cuda(args, rank, world, local_rank)
    except BaseException:  # a rank that dies quietly would leave its peers waiting in a collective
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)


if __name__ == "__main__":
    sys.exit(main())
