"""Host-side mirror of the reference driver's interface for the sort path, over the C ABI.

The reference (mpi/mpi_lsbsort.cpp) is C++ with no Python surface, so this module is a thin
ctypes binding whose names follow the reference: `DistributedSorter.create` ~
DistributedArray<SortElement>::create for A and B (:138-161,:638-639), `generate` ~ the pcg64
fill loop (:650-656), `my_sort` ~ mySort (:580-585), `global_shuffle(digit)` ~ globalShuffle
(:481-577), `verify` ~ the verify block (:710-739).  All compute happens in
liblsbsort.so (CUDA, sm_100a).  There is no CPU fallback: if the library is missing or there
is no GPU, calls raise.
"""
import ctypes
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_LIB_PATH = os.environ.get("LSB_LIBRARY", os.path.join(_HERE, "liblsbsort.so"))  # override: kernel experiments
_HEADER = os.path.join(_ROOT, "include", "lsbsort.h")

ELT = np.dtype([("key", "<u8"), ("val", "<u8")])  # SortElement, mpi/mpi_lsbsort.cpp:29-32

LSB_MAX_GPUS = 8
LSB_MAX_SUBPASSES = 32
LSB_COMM_ID_BYTES = 128
FLAG_PHASE_EVENTS = 1
FLAG_TWO_LEVEL = 2
FLAG_ONE_PASS = 4
FLAG_NO_SKIP = 8
# key orders (include/lsbsort.h): the sort is stable and ascending by order_key(key); key bits are never rewritten
FLAG_KEY_I64 = 16
FLAG_KEY_F64 = 32
FLAG_DESCENDING = 64
SEG_LOCAL_INDEX = 1  # lsb_sort_segments_device without vals_in: index within the segment, not the global input index
KEY_DTYPE_FLAGS = {np.dtype(np.uint64): 0, np.dtype(np.int64): FLAG_KEY_I64, np.dtype(np.float64): FLAG_KEY_F64}
# key types of lsb_sort_device_typed / lsb_sort_segments_device_typed (LSB_KEY_*), by torch dtype name
KEY_CONTEXT = 0
NARROW_KEY_TYPES = {"uint32": 1, "int32": 2, "float32": 3, "uint16": 4, "int16": 5, "float16": 6, "bfloat16": 7}


class LsbError(RuntimeError):
    def __init__(self, code, what, detail=""):
        super().__init__(f"{what} failed: status {code}" + (f" ({detail})" if detail else ""))
        self.code = code


class _Config(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int64), ("ranks", ctypes.c_int32), ("world_size", ctypes.c_int32),
                ("world_rank", ctypes.c_int32), ("device", ctypes.c_int32), ("radix_bits", ctypes.c_int32),
                ("and_draws", ctypes.c_int32), ("seed_base", ctypes.c_uint64), ("key_mask", ctypes.c_uint64),
                ("flags", ctypes.c_uint32), ("reserved", ctypes.c_uint32)]


class Stats(ctypes.Structure):
    _fields_ = [("device_ms", ctypes.c_double), ("passes", ctypes.c_int32), ("subpasses", ctypes.c_int32), ("skipped", ctypes.c_int32), ("reserved0", ctypes.c_int32),
                ("elements", ctypes.c_int64), ("hist_ms", ctypes.c_double), ("scan_ms", ctypes.c_double),
                ("partition_ms", ctypes.c_double), ("exchange_ms", ctypes.c_double), ("subpass_ms", ctypes.c_double * LSB_MAX_SUBPASSES),
                ("sent", ctypes.c_int64 * LSB_MAX_GPUS), ("partition_launches", ctypes.c_int64), ("partition_elements", ctypes.c_int64),
                ("kernel_launches", ctypes.c_int64)]


class KeyColumn(ctypes.Structure):
    """lsb_key_column: one key column of lsb_lexsort_device"""
    _fields_ = [("keys", ctypes.c_void_p), ("key_type", ctypes.c_uint32), ("flags", ctypes.c_uint32)]


class Verify(ctypes.Structure):
    _fields_ = [("order_violations", ctypes.c_int64), ("elements", ctypes.c_int64),
                ("checksum", ctypes.c_uint64 * 4)]


def library_path():
    return _LIB_PATH


def header_symbols():
    """names of every function include/lsbsort.h declares"""
    with open(_HEADER) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(lsb_[a-z0-9_]+)\s*\(", text)))


_lib = None


def load_library():
    """dlopen liblsbsort.so; raises (never falls back) if it has not been built"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise LsbError(-4, "load_library", f"{_LIB_PATH} not built; run python -c 'import __graft_entry__ as g; g.build()'")
    L = ctypes.CDLL(_LIB_PATH)
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    pvp = ctypes.POINTER(ctypes.c_void_p)
    L.lsb_abi_version.restype = ci
    L.lsb_create.argtypes = [pvp, ctypes.POINTER(_Config)]
    L.lsb_destroy.argtypes = [vp]
    L.lsb_destroy.restype = None
    L.lsb_last_error.argtypes = [vp]
    L.lsb_last_error.restype = ctypes.c_char_p
    L.lsb_status_string.argtypes = [ci]
    L.lsb_status_string.restype = ctypes.c_char_p
    L.lsb_tune.argtypes = [ctypes.c_char_p, ci]
    L.lsb_comm_unique_id.argtypes = [vp]
    L.lsb_comm_init.argtypes = [vp, vp]
    L.lsb_barrier.argtypes = [vp]
    L.lsb_shard_info.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64)]
    L.lsb_generate.argtypes = [vp]
    L.lsb_upload.argtypes = [vp, vp, i64, i64]
    L.lsb_download.argtypes = [vp, vp, i64, i64]
    L.lsb_device_ptr.argtypes = [vp, pvp]
    L.lsb_host_alloc.argtypes = [pvp, i64]
    L.lsb_host_free.argtypes = [vp]
    L.lsb_sort.argtypes = [vp, ctypes.POINTER(Stats)]
    L.lsb_pass.argtypes = [vp, ci, ctypes.POINTER(Stats)]
    L.lsb_sort_host.argtypes = [vp, vp, vp, i64, ctypes.POINTER(Stats)]
    L.lsb_sort_device.argtypes = [vp, vp, vp, vp, vp, i64, vp, ctypes.POINTER(Stats)]
    L.lsb_sort_segments_device.argtypes = [vp, vp, vp, vp, vp, i64, vp, i64, ctypes.c_uint32, vp, ctypes.POINTER(Stats)]
    L.lsb_sort_device_typed.argtypes = [vp, ctypes.c_uint32, vp, vp, vp, vp, i64, vp, ctypes.POINTER(Stats)]
    L.lsb_sort_segments_device_typed.argtypes = [vp, ctypes.c_uint32, vp, vp, vp, vp, i64, vp, i64, ctypes.c_uint32, vp,
                                                 ctypes.POINTER(Stats)]
    L.lsb_lexsort_device.argtypes = [vp, ctypes.POINTER(KeyColumn), ctypes.c_int32, vp, vp, i64, vp, ctypes.POINTER(Stats)]
    L.lsb_histogram.argtypes = [vp, ci, vp]
    L.lsb_starts.argtypes = [vp, ci, vp]
    L.lsb_num_passes.argtypes = [vp]
    L.lsb_digit_bits.argtypes = [vp, ci]
    L.lsb_checksum.argtypes = [vp, vp]
    L.lsb_verify_device.argtypes = [vp, ctypes.POINTER(Verify)]
    for name in header_symbols():
        getattr(L, name)  # every declared entry point must be exported
    _lib = L
    return L


def abi_symbols():
    L = load_library()
    return [s for s in header_symbols() if hasattr(L, s)]


def tune(key, value):
    """experiment knob for profiling sweeps (lsb_tune): applies to sorters created afterwards"""
    rc = load_library().lsb_tune(key.encode(), int(value))
    if rc:
        raise LsbError(rc, "lsb_tune", load_library().lsb_last_error(None).decode())


def comm_unique_id():
    """MPI_Init's rendezvous token: rank 0 makes it, every rank passes it to comm_init"""
    buf = ctypes.create_string_buffer(LSB_COMM_ID_BYTES)
    rc = load_library().lsb_comm_unique_id(buf)
    if rc:
        raise LsbError(rc, "lsb_comm_unique_id", load_library().lsb_last_error(None).decode())
    return buf.raw


class PinnedBuffer:
    """page-locked host array of ELT (cudaHostAlloc through the C ABI)"""

    def __init__(self, count):
        self._ptr = ctypes.c_void_p()
        rc = load_library().lsb_host_alloc(ctypes.byref(self._ptr), max(count, 1) * ELT.itemsize)
        if rc:
            raise LsbError(rc, "lsb_host_alloc")
        raw = (ctypes.c_char * (max(count, 1) * ELT.itemsize)).from_address(self._ptr.value)
        self.array = np.frombuffer(raw, dtype=ELT)[:count]

    def free(self):
        if self._ptr:
            self.array = None
            load_library().lsb_host_free(self._ptr)
            self._ptr = None


class DistributedSorter:
    """One process's view of the distributed arrays A and B (one shard of each on one GPU).

    key_dtype: None for the 8-byte key the flags name, or one of torch.uint32, int32, float32, uint16, int16, float16,
    bfloat16: sort_device / sort_segments then take keys (and keys_out) of exactly that dtype and sort them in
    ceil(W / radix_bits) passes (lsb_sort_device_typed); flags may add FLAG_DESCENDING but no 8-byte key type."""

    key_dtype = None

    def __init__(self, n, ranks=0, world_size=1, world_rank=0, device=0, radix_bits=16, seed_base=0,
                 key_mask=0xFFFFFFFFFFFFFFFF, and_draws=1, flags=0, key_dtype=None):
        if key_dtype is not None:
            torch = _torch()
            if _narrow_key_type(torch, key_dtype) is None:
                raise TypeError(f"key_dtype must be None or one of torch.{', torch.'.join(NARROW_KEY_TYPES)}, not {key_dtype}")
            if flags & (FLAG_KEY_I64 | FLAG_KEY_F64):
                raise ValueError(f"key_dtype {key_dtype} excludes the 8-byte key-type flags FLAG_KEY_I64 / FLAG_KEY_F64")
        self._L = load_library()
        self._ctx = ctypes.c_void_p()
        cfg = _Config(n=n, ranks=ranks, world_size=world_size, world_rank=world_rank, device=device,
                      radix_bits=radix_bits, and_draws=and_draws, seed_base=seed_base, key_mask=key_mask,
                      flags=flags, reserved=0)
        rc = self._L.lsb_create(ctypes.byref(self._ctx), ctypes.byref(cfg))
        if rc:
            raise LsbError(rc, "lsb_create", self._L.lsb_last_error(None).decode())
        per, here, first = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        self._L.lsb_shard_info(self._ctx, ctypes.byref(per), ctypes.byref(here), ctypes.byref(first))
        self.n, self.world_size, self.world_rank = n, world_size, world_rank
        self.per, self.here, self.first_global = per.value, here.value, first.value
        self.radix_bits = radix_bits
        self.device, self.flags = device, flags
        self.key_dtype = key_dtype

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))

    # -- plumbing -----------------------------------------------------------------------
    def _check(self, rc, what):
        if rc:
            raise LsbError(rc, what, self._L.lsb_last_error(self._ctx).decode())

    def close(self):
        if self._ctx:
            self._L.lsb_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def comm_init(self, unique_id):
            self._check(self._L.lsb_comm_init(self._ctx, unique_id), "lsb_comm_init")

    def barrier(self):
        """MPI_Barrier(MPI_COMM_WORLD): all GPUs drained their sort streams"""
        self._check(self._L.lsb_barrier(self._ctx), "lsb_barrier")

    # -- data ---------------------------------------------------------------------------
    def generate(self):
        self._check(self._L.lsb_generate(self._ctx), "lsb_generate")

    def upload(self, elts, local_off=0):
        elts = np.ascontiguousarray(elts, dtype=ELT)
        self._check(self._L.lsb_upload(self._ctx, elts.ctypes.data, local_off, len(elts)), "lsb_upload")

    def download(self, local_off=0, count=None, out=None):
        count = self.here - local_off if count is None else count
        if out is None:
            out = np.empty(count, dtype=ELT)
        self._check(self._L.lsb_download(self._ctx, out.ctypes.data, local_off, count), "lsb_download")
        return out

    def device_ptr(self):
        p = ctypes.c_void_p()
        self._check(self._L.lsb_device_ptr(self._ctx, ctypes.byref(p)), "lsb_device_ptr")
        return p.value

    # -- the hot path ---------------------------------------------------------------------
    def my_sort(self):
        """mySort(A, B): all passes; returns Stats"""
        st = Stats()
        self._check(self._L.lsb_sort(self._ctx, ctypes.byref(st)), "lsb_sort")
        return st

    def global_shuffle(self, digit):
        """globalShuffle(A, B, digit): one stable pass"""
        st = Stats()
        self._check(self._L.lsb_pass(self._ctx, digit, ctypes.byref(st)), "lsb_pass")
        return st

    def sort_host(self, host_in, host_out):
        """host buffers in, host buffers out (copies inside the call)"""
        st = Stats()
        assert host_in.dtype == ELT and host_out.dtype == ELT and len(host_in) == len(host_out)
        self._check(self._L.lsb_sort_host(self._ctx, host_in.ctypes.data, host_out.ctypes.data, len(host_in),
                                          ctypes.byref(st)), "lsb_sort_host")
        return st

    def _outputs(self, what, keys, vals, keys_out, vals_out):
        """checked keys_out / vals_out of sort_device and sort_segments: None allocates, False means none"""
        torch = _torch()
        n = self.here
        if keys_out is False and vals_out is False:
            raise ValueError(f"{what}: keys_out and vals_out cannot both be False")
        if self.key_dtype is None:
            _check_vector(torch, keys, "keys", n, self.device, key_flags=self.flags & (FLAG_KEY_I64 | FLAG_KEY_F64))
        else:
            _check_vector(torch, keys, "keys", n, self.device, dtype=self.key_dtype)
        if vals is not None:
            _check_vector(torch, vals, "vals", n, self.device)
        if keys_out is None:
            keys_out = torch.empty_like(keys)
        elif keys_out is not False:
            _check_vector(torch, keys_out, "keys_out", n, self.device, dtype=self.key_dtype)
            if keys_out.dtype != keys.dtype:
                raise TypeError(f"{what}: keys_out must have the keys' dtype {keys.dtype}, not {keys_out.dtype}")
        if vals_out is None:
            vals_out = torch.empty_like(vals) if vals is not None else torch.empty(n, dtype=torch.int64, device=keys.device)
        elif vals_out is not False:
            _check_vector(torch, vals_out, "vals_out", n, self.device)
        return keys_out, vals_out

    def sort_segments(self, keys, offsets, vals=None, keys_out=None, vals_out=None, local_index=False, stream=None):
        """Every segment of a device array sorted at once (lsb_sort_segments_device): segment s is keys[offsets[s] :
        offsets[s+1]], and the result is the stable sort by (segment, key) -- each segment in this sorter's key order,
        the segments in ascending order.  `offsets`: 1-D contiguous int64 CUDA tensor of >= 2 elements on this sorter's
        device, rising from 0 to `here` (the library checks its contents).  keys, vals, outputs and stream as in
        sort_device; without vals, vals_out receives the input index of every key, or with local_index=True its index
        within its segment (what torch.sort(dim=-1) returns for rows).  Returns (keys_out, vals_out, Stats)."""
        torch = _torch()
        if not isinstance(offsets, torch.Tensor):
            raise TypeError(f"offsets must be a torch.Tensor, not {type(offsets).__name__}")
        if offsets.dtype != torch.int64:
            raise TypeError(f"offsets must be torch.int64, not {offsets.dtype}")
        if offsets.dim() != 1 or offsets.numel() < 2:
            raise ValueError(f"offsets must be 1-D with at least 2 elements (one segment), not of shape {tuple(offsets.shape)}")
        _check_vector(torch, offsets, "offsets", None, self.device)
        keys_out, vals_out = self._outputs("sort_segments", keys, vals, keys_out, vals_out)
        if stream is None:
            stream = torch.cuda.current_stream(keys.device)
        handle = stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)
        ptr = lambda t: t.data_ptr() if t is not None and t is not False else None  # noqa: E731
        st = Stats()
        args = (ptr(keys), ptr(vals), ptr(keys_out), ptr(vals_out), self.here, offsets.data_ptr(), offsets.numel() - 1,
                SEG_LOCAL_INDEX if local_index else 0, handle, ctypes.byref(st))
        if self.key_dtype is None:
            self._check(self._L.lsb_sort_segments_device(self._ctx, *args), "lsb_sort_segments_device")
        else:
            key_type = _narrow_key_type(torch, self.key_dtype)
            self._check(self._L.lsb_sort_segments_device_typed(self._ctx, key_type, *args), "lsb_sort_segments_device_typed")
        return (keys_out if keys_out is not False else None), (vals_out if vals_out is not False else None), st

    def sort_device(self, keys, vals=None, keys_out=None, vals_out=None, stream=None):
        """CUDA tensors in, CUDA tensors out, no host copy (lsb_sort_device).  `keys`: 1-D contiguous uint64, int64 or
        float64 tensor of `here` elements on this sorter's device, of the dtype its key-type flags name (of key_dtype
        when the sorter has one: lsb_sort_device_typed); `vals`: the same
        shape with any 8-byte dtype, or None for the global input index (torch.int64: the stable argsort).  keys_out /
        vals_out: a tensor to write (may be the input itself: in place), None to allocate one, False for none (not
        both).  The library waits for the work queued on `stream` (default: the current stream) before it reads the
        inputs and returns when the outputs are written.  Returns (keys_out, vals_out, Stats of the sort itself)."""
        torch = _torch()
        n = self.here
        keys_out, vals_out = self._outputs("sort_device", keys, vals, keys_out, vals_out)
        if stream is None:
            stream = torch.cuda.current_stream(keys.device)
        handle = stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)
        ptr = lambda t: t.data_ptr() if t is not None and t is not False else None  # noqa: E731
        st = Stats()
        args = (ptr(keys), ptr(vals), ptr(keys_out), ptr(vals_out), n, handle, ctypes.byref(st))
        if self.key_dtype is None:
            self._check(self._L.lsb_sort_device(self._ctx, *args), "lsb_sort_device")
        else:
            key_type = _narrow_key_type(torch, self.key_dtype)
            self._check(self._L.lsb_sort_device_typed(self._ctx, key_type, *args), "lsb_sort_device_typed")
        return (keys_out if keys_out is not False else None), (vals_out if vals_out is not False else None), st

    def lexsort_device(self, columns, vals=None, vals_out=None, descending=False, stream=None):
        """The stable sort by several key columns (lsb_lexsort_device), np.lexsort's convention: columns[0] is the least
        significant key, columns[-1] the primary.  `columns`: a sequence of 1-D contiguous CUDA tensors of `here`
        elements on this sorter's device, each of uint64, int64, float64, uint32, int32, float32, uint16, int16, float16
        or bfloat16 (the sorter's own key_dtype and flags play no part, and it must have no key-order flags).
        `descending`: a bool for every column, or one bool per column.  Each column sorts in numpy's and torch's order:
        NaNs last (first when descending), -0.0 == +0.0; elements equal in every column keep their input order.
        `vals`: 8-byte tensor like a column, or None for the input index (torch.int64: what np.lexsort returns).
        `vals_out`: a tensor to write, or None to allocate one.  Stream as in sort_device.  Returns (vals_out, Stats)."""
        torch = _torch()
        n = self.here
        cols = _check_columns(torch, columns, n, self.device)
        desc = _check_descending(descending, len(cols))
        if vals is not None:
            _check_vector(torch, vals, "vals", n, self.device)
        if vals_out is None:
            vals_out = torch.empty_like(vals) if vals is not None else torch.empty(n, dtype=torch.int64, device=cols[0].device)
        else:
            _check_vector(torch, vals_out, "vals_out", n, self.device)
        if stream is None:
            stream = torch.cuda.current_stream(cols[0].device)
        handle = stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)
        spec = (KeyColumn * len(cols))()
        for c, (t, d) in enumerate(zip(cols, desc)):
            narrow = _narrow_key_type(torch, t.dtype)
            spec[c].keys = t.data_ptr() or None
            spec[c].key_type = narrow if narrow is not None else KEY_CONTEXT
            spec[c].flags = (0 if narrow is not None else _key_dtype_flags(torch)[t.dtype]) | (FLAG_DESCENDING if d else 0)
        st = Stats()
        ptr = lambda t: t.data_ptr() or None if t is not None else None  # noqa: E731
        self._check(self._L.lsb_lexsort_device(self._ctx, spec, len(cols), ptr(vals), ptr(vals_out), n, handle,
                                               ctypes.byref(st)), "lsb_lexsort_device")
        return vals_out, st

    # -- test hooks -----------------------------------------------------------------------
    def num_passes(self):
        return self._L.lsb_num_passes(self._ctx)

    def digit_bits(self, digit):
        return self._L.lsb_digit_bits(self._ctx, digit)

    def histogram(self, digit):
        out = np.zeros(1 << self.digit_bits(digit), dtype=np.int64)
        self._check(self._L.lsb_histogram(self._ctx, digit, out.ctypes.data), "lsb_histogram")
        return out

    def starts(self, digit):
        out = np.zeros(1 << self.digit_bits(digit), dtype=np.int64)
        self._check(self._L.lsb_starts(self._ctx, digit, out.ctypes.data), "lsb_starts")
        return out

    # -- verification ---------------------------------------------------------------------
    def checksum(self):
        out = (ctypes.c_uint64 * 4)()
        self._check(self._L.lsb_checksum(self._ctx, out), "lsb_checksum")
        return [int(x) for x in out]

    def verify(self, raise_on_failure=True):
        v = Verify()
        rc = self._L.lsb_verify_device(self._ctx, ctypes.byref(v))
        if rc and (raise_on_failure or rc != -6):
            self._check(rc, "lsb_verify_device")
        return v


def sort_pairs(keys, vals=None, descending=False, device=0):
    """Stable sort of a 1-D numpy array of uint64, int64 or float64 keys, with 8-byte `vals` (default arange(n) as int64,
    so the returned vals are the stable argsort), on one GPU through sort_host.  The order is numpy's and torch's: NaNs
    last (first when descending), -0.0 == +0.0, equal keys in input order.  Returns (keys, vals) in the input dtypes;
    the records are permuted, never rewritten (-0.0 and NaN payloads come back as they went in)."""
    keys = np.ascontiguousarray(keys)
    if keys.dtype not in KEY_DTYPE_FLAGS:
        raise TypeError(f"sort_pairs: keys must be uint64, int64 or float64, not {keys.dtype}")
    vals = np.arange(len(keys), dtype=np.int64) if vals is None else np.ascontiguousarray(vals)
    if keys.ndim != 1 or vals.shape != keys.shape:
        raise ValueError(f"sort_pairs: keys and vals must be 1-D of one length, not {keys.shape} and {vals.shape}")
    if vals.dtype.itemsize != 8:
        raise TypeError(f"sort_pairs: vals must have an 8-byte dtype, not {vals.dtype}")
    n = len(keys)
    recs = np.empty(n, dtype=ELT)
    recs["key"] = keys.view(np.uint64)
    recs["val"] = vals.view(np.uint64)
    out = np.empty(n, dtype=ELT)
    flags = KEY_DTYPE_FLAGS[keys.dtype] | (FLAG_DESCENDING if descending else 0)
    with DistributedSorter(n, ranks=1, device=device, flags=flags) as s:
        s.sort_host(recs, out)
    return out["key"].view(keys.dtype).copy(), out["val"].view(vals.dtype).copy()


def _torch():
    import torch  # only the tensor entry points need it
    return torch


def _key_dtype_flags(torch):
    return {torch.uint64: 0, torch.int64: FLAG_KEY_I64, torch.float64: FLAG_KEY_F64}


def _narrow_key_type(torch, dtype):
    """LSB_KEY_* of a narrow torch dtype, None for any other"""
    return NARROW_KEY_TYPES.get(str(dtype).replace("torch.", "")) if isinstance(dtype, torch.dtype) else None


def _check_vector(torch, t, name, n=None, device=None, key_flags=None, dtype=None):
    """TypeError / ValueError unless `t` is a 1-D contiguous CUDA tensor of 8-byte elements, or of exactly `dtype` when
    given (of n elements on `device`, and of the key dtype that `key_flags` names, when given)"""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, not {type(t).__name__}")
    if dtype is not None:
        if t.dtype != dtype:
            raise TypeError(f"{name} must be {dtype}, the sorter's key_dtype, not {t.dtype}")
    elif key_flags is not None:
        dtypes = _key_dtype_flags(torch)
        if t.dtype not in dtypes:
            raise TypeError(f"{name} must be torch.uint64, int64 or float64, not {t.dtype}")
        if dtypes[t.dtype] != key_flags:
            raise TypeError(f"{name}: dtype {t.dtype} does not match the sorter's key-type flags ({key_flags})")
    elif t.element_size() != 8:
        raise TypeError(f"{name} must have an 8-byte dtype, not {t.dtype}")
    if t.dim() != 1:
        raise ValueError(f"{name} must be 1-D, not of shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if n is not None and t.numel() != n:
        raise ValueError(f"{name} has {t.numel()} elements, the shard {n}")
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor, not on {t.device}")
    if device is not None and t.device.index != device:
        raise ValueError(f"{name} is on {t.device}, the sorter on cuda:{device}")


def sort_tensor(keys, vals=None, descending=False):
    """torch.sort(keys, stable=True, descending=descending) for a 1-D CUDA tensor of uint64, int64 or float64 keys, on
    that tensor's GPU, with no host copy: returns (sorted keys, vals permuted the same way), or (sorted keys, int64
    indices) without vals.  The order is torch's and numpy's: NaNs last (first when descending), -0.0 == +0.0, equal
    keys in input order; key bits are never rewritten.  Makes a one-GPU sorter for the call."""
    torch = _torch()
    if not isinstance(keys, torch.Tensor):
        raise TypeError(f"keys must be a torch.Tensor, not {type(keys).__name__}")
    dtypes = _key_dtype_flags(torch)
    if keys.dtype not in dtypes:
        raise TypeError(f"keys must be torch.uint64, int64 or float64, not {keys.dtype}")
    keys = keys.contiguous()
    _check_vector(torch, keys, "keys", key_flags=dtypes[keys.dtype])
    if vals is not None:
        if not isinstance(vals, torch.Tensor):
            raise TypeError(f"vals must be a torch.Tensor, not {type(vals).__name__}")
        vals = vals.contiguous()
        _check_vector(torch, vals, "vals", keys.numel(), keys.device.index)
    flags = dtypes[keys.dtype] | (FLAG_DESCENDING if descending else 0)
    with DistributedSorter(keys.numel(), ranks=1, device=keys.device.index, flags=flags) as s:
        k, v, _ = s.sort_device(keys, vals)
    return k, v


def sort_segments(keys, offsets=None, vals=None, descending=False):
    """Sort many groups of a CUDA tensor at once, on that tensor's GPU, with no host copy.  Keys are uint64, int64 or
    float64, sorted stably in numpy's and torch's order (NaNs last, first when descending; -0.0 == +0.0; equal keys in
    input order; key bits never rewritten).
      2-D keys [B, L], no offsets: every row sorted, as torch.sort(keys, dim=-1, stable=True, descending=...) does:
        returns (sorted keys [B, L], int64 indices within the row [B, L]), or vals [B, L] permuted within the rows.
      1-D keys with offsets (1-D int64 CUDA tensor of S + 1 elements rising from 0 to len(keys); empty segments
        allowed): segment s = keys[offsets[s] : offsets[s+1]] sorted, the segments in place: returns (sorted keys,
        int64 input indices), or vals permuted the same way.
    Anything else is a ValueError.  Makes a one-GPU sorter for the call."""
    torch = _torch()
    if not isinstance(keys, torch.Tensor):
        raise TypeError(f"keys must be a torch.Tensor, not {type(keys).__name__}")
    dtypes = _key_dtype_flags(torch)
    if keys.dtype not in dtypes:
        raise TypeError(f"keys must be torch.uint64, int64 or float64, not {keys.dtype}")
    if vals is not None and not isinstance(vals, torch.Tensor):
        raise TypeError(f"vals must be a torch.Tensor, not {type(vals).__name__}")
    if vals is not None and vals.shape != keys.shape:
        raise ValueError(f"vals must have the keys' shape {tuple(keys.shape)}, not {tuple(vals.shape)}")
    if keys.dim() == 2 and offsets is None:
        rows, width = keys.shape
        if not keys.is_cuda:
            raise ValueError(f"keys must be a CUDA tensor, not on {keys.device}")
        if rows == 0:
            return keys.clone(), (vals.clone() if vals is not None else torch.empty_like(keys, dtype=torch.int64))
        offsets = torch.arange(rows + 1, dtype=torch.int64, device=keys.device) * width
        k, v = _sort_segments_1d(torch, keys.reshape(-1), offsets, None if vals is None else vals.reshape(-1), descending,
                                 local_index=True)
        return k.view(rows, width), v.view(rows, width)
    if keys.dim() == 1 and offsets is not None:
        return _sort_segments_1d(torch, keys, offsets, vals, descending, local_index=False)
    raise ValueError("sort_segments takes 2-D keys without offsets (rows) or 1-D keys with offsets, not "
                     f"{keys.dim()}-D keys {'with' if offsets is not None else 'without'} offsets")


def _sort_segments_1d(torch, keys, offsets, vals, descending, local_index):
    keys = keys.contiguous()
    dtypes = _key_dtype_flags(torch)
    _check_vector(torch, keys, "keys", key_flags=dtypes[keys.dtype])
    if vals is not None:
        vals = vals.contiguous()
        _check_vector(torch, vals, "vals", keys.numel(), keys.device.index)
    flags = dtypes[keys.dtype] | (FLAG_DESCENDING if descending else 0)
    with DistributedSorter(keys.numel(), ranks=1, device=keys.device.index, flags=flags) as s:
        k, v, _ = s.sort_segments(keys, offsets, vals, local_index=local_index)
    return k, v


def _check_columns(torch, columns, n=None, device=None):
    """the key columns of a lexsort as a list: TypeError / ValueError unless `columns` is a non-empty sequence (not a
    tensor) of 1-D contiguous CUDA tensors of one of the ten key dtypes, of n elements on `device` when given"""
    if isinstance(columns, torch.Tensor) or not isinstance(columns, (list, tuple)):
        raise TypeError(f"columns must be a list or tuple of tensors, not {type(columns).__name__}")
    if not columns:
        raise ValueError("columns is empty: a lexsort needs at least one key column")
    for c, t in enumerate(columns):
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"columns[{c}] must be a torch.Tensor, not {type(t).__name__}")
        if t.dtype not in _key_dtype_flags(torch) and _narrow_key_type(torch, t.dtype) is None:
            raise TypeError(f"columns[{c}] must be torch.uint64, int64, float64, torch.{', torch.'.join(NARROW_KEY_TYPES)}, "
                            f"not {t.dtype}")
        _check_vector(torch, t, f"columns[{c}]", n, device, dtype=t.dtype)
    return list(columns)


def _check_descending(descending, k):
    """one bool per column from a bool or a sequence of k bools"""
    if isinstance(descending, bool):
        return [descending] * k
    if not isinstance(descending, (list, tuple)) or not all(isinstance(d, bool) for d in descending):
        raise TypeError(f"descending must be a bool or a list of bools, not {descending!r}")
    if len(descending) != k:
        raise ValueError(f"descending has {len(descending)} entries for {k} columns")
    return list(descending)


def lexsort(keys, descending=False, vals=None):
    """np.lexsort for CUDA tensors, on their GPU, with no host copy: the permutation that sorts stably by the last key,
    then the one before it, ..., then the first.  `keys`: a list or tuple of 1-D CUDA tensors of one length on one
    device, or a 2-D CUDA tensor whose rows are the keys; each of uint64, int64, float64, uint32, int32, float32, uint16,
    int16, float16 or bfloat16 (they may differ).  `descending`: a bool, or one bool per key.  Every key sorts in numpy's
    and torch's order (NaNs last, first when descending; -0.0 == +0.0), and elements equal in every key keep their input
    order.  Returns int64 indices, or `vals` (a tensor of 8-byte elements, one per key element) permuted.  Makes a
    one-GPU sorter for the call."""
    torch = _torch()
    if isinstance(keys, torch.Tensor):
        if keys.dim() != 2:
            raise ValueError(f"keys must be a 2-D tensor (one key per row) or a list of 1-D tensors, not {keys.dim()}-D")
        keys = list(keys.unbind(0))
    if not isinstance(keys, (list, tuple)):
        raise TypeError(f"keys must be a list or tuple of tensors or a 2-D tensor, not {type(keys).__name__}")
    if not keys:
        raise ValueError("lexsort needs at least one key")
    keys = [k.contiguous() if isinstance(k, torch.Tensor) else k for k in keys]
    _check_columns(torch, keys)
    n, dev = keys[0].numel(), keys[0].device
    for c, k in enumerate(keys):
        if k.numel() != n or k.device != dev:
            raise ValueError(f"keys[{c}] has {k.numel()} elements on {k.device}, keys[0] {n} on {dev}")
    desc = _check_descending(descending, len(keys))
    if vals is not None:
        if not isinstance(vals, torch.Tensor):
            raise TypeError(f"vals must be a torch.Tensor, not {type(vals).__name__}")
        vals = vals.contiguous()
        _check_vector(torch, vals, "vals", n, dev.index)
    with DistributedSorter(n, ranks=1, device=dev.index) as s:
        v, _ = s.lexsort_device(keys, vals, descending=desc)
    return v


def sort(input, dim=-1, descending=False, stable=False):
    """torch.sort for a CUDA tensor of uint64, int64, float64, uint32, int32, float32, uint16, int16, float16 or bfloat16
    keys, of any rank and `dim`, on that tensor's GPU: returns torch.return_types.sort(values, indices).  The result is
    always the stable sort (also a valid answer for stable=False), in numpy's and torch's order: NaNs last (first when
    descending), -0.0 == +0.0, equal keys in input order; key bits are never rewritten, and a W-bit key takes
    ceil(W / 16) passes.  One row (1-D input, or every other dimension of size 1) is one sort_device; more rows are
    sorted at once by sort_segments with `dim` moved last.  Makes a one-GPU sorter for the call."""
    torch = _torch()
    values, indices = _sort_rows(torch, input, dim, descending, keys=True)
    return torch.return_types.sort((values, indices))


def argsort(input, dim=-1, descending=False, stable=False):
    """torch.argsort: the indices of sort(input, dim, descending), without writing the sorted keys"""
    return _sort_rows(_torch(), input, dim, descending, keys=False)[1]


def _sort_rows(torch, x, dim, descending, keys):
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"input must be a torch.Tensor, not {type(x).__name__}")
    wide = _key_dtype_flags(torch)
    if x.dtype not in wide and _narrow_key_type(torch, x.dtype) is None:
        raise TypeError(f"input must be torch.uint64, int64, float64, torch.{', torch.'.join(NARROW_KEY_TYPES)}, not {x.dtype}")
    if not x.is_cuda:
        raise ValueError(f"input must be a CUDA tensor, not on {x.device}")
    nd = max(x.dim(), 1)
    if isinstance(dim, bool) or not isinstance(dim, int) or not -nd <= dim < nd:
        raise ValueError(f"dim must be an int in [{-nd}, {nd - 1}] for a {x.dim()}-D input, not {dim!r}")
    if x.dim() == 0 or x.numel() == 0:  # as torch answers: the input itself, index 0 / nothing
        return (x.clone() if keys else None), torch.zeros_like(x, dtype=torch.int64)
    d = dim % nd
    rows = x.movedim(d, -1).contiguous()
    shape, width = rows.shape, rows.shape[-1]
    flat = rows.view(-1)
    flags = wide.get(x.dtype, 0) | (FLAG_DESCENDING if descending else 0)
    key_dtype = None if x.dtype in wide else x.dtype
    with DistributedSorter(flat.numel(), ranks=1, device=x.device.index, flags=flags, key_dtype=key_dtype) as s:
        if flat.numel() == width:
            k, v, _ = s.sort_device(flat, keys_out=None if keys else False)
        else:
            offsets = torch.arange(flat.numel() // width + 1, dtype=torch.int64, device=x.device) * width
            k, v, _ = s.sort_segments(flat, offsets, keys_out=None if keys else False, local_index=True)
    back = lambda t: t.view(shape).movedim(-1, d).contiguous()  # noqa: E731
    return (back(k) if keys else None), back(v)
