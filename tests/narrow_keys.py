"""Narrow key types (LSB_KEY_U32 .. LSB_KEY_BF16 of include/lsbsort.h) for the tests: their bit patterns as numpy
unsigned arrays, special values, and the reference order -- numpy's stable argsort of the typed values, bfloat16
through its exact float32 widening -- which shares no code with order_key_narrow (csrc/lsb_keyorder.cuh).
"""
import numpy as np

from distributed_lsb_b200 import lsbsort as L

NAMES = list(L.NARROW_KEY_TYPES)  # uint32 int32 float32 uint16 int16 float16 bfloat16
KEY_TYPE = dict(L.NARROW_KEY_TYPES)
BITS = {name: 16 if name.endswith("16") else 32 for name in NAMES}
UINT = {32: np.uint32, 16: np.uint16}
SINT = {32: np.int32, 16: np.int16}
NUMPY = {"uint32": np.uint32, "int32": np.int32, "float32": np.float32, "uint16": np.uint16, "int16": np.int16,
         "float16": np.float16}

# +-0, +-inf, quiet and signalling NaNs of both signs with payloads, +- the smallest subnormal, +- the largest finite,
# +-1, and the all-ones patterns; as integers the same bits are 0, the minimum, the maximum, -1 and 1
SPECIAL = {
    32: [0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x7FC00123, 0xFFE0ABCD, 0x7F800001,
         0xFF800001, 0x7FA00042, 0x00000001, 0x80000001, 0x7F7FFFFF, 0xFF7FFFFF, 0x3F800000, 0xBF800000, 0x7FFFFFFF,
         0xFFFFFFFF],
    "float16": [0x0000, 0x8000, 0x7C00, 0xFC00, 0x7E00, 0xFE00, 0x7E12, 0xFF3D, 0x7C01, 0xFC01, 0x7D42, 0x0001, 0x8001,
                0x7BFF, 0xFBFF, 0x3C00, 0xBC00, 0x7FFF, 0xFFFF],
    "bfloat16": [0x0000, 0x8000, 0x7F80, 0xFF80, 0x7FC0, 0xFFC0, 0x7FC3, 0xFFE5, 0x7F81, 0xFF81, 0x7FA2, 0x0001, 0x8001,
                 0x7F7F, 0xFF7F, 0x3F80, 0xBF80, 0x7FFF, 0xFFFF],
}


def special_bits(name):
    w = BITS[name]
    return np.array(SPECIAL[32] if w == 32 else SPECIAL.get(name, SPECIAL["float16"]), dtype=UINT[w])


def typed(bits, name):
    """the bit patterns `bits` (numpy uint32 / uint16) as values numpy orders like the key type"""
    bits = np.ascontiguousarray(bits, dtype=UINT[BITS[name]])
    if name == "bfloat16":
        return (bits.astype(np.uint32) << np.uint32(16)).view(np.float32)  # exact: bfloat16 is float32's high half
    return bits.view(NUMPY[name])


def argsort(bits, name, descending=False, axis=-1):
    """numpy's stable argsort of the typed values along `axis`; descending: the stable ascending sort of the reversed
    array, reversed (NaNs first, equal keys in input order)"""
    x = np.moveaxis(typed(bits, name), axis, -1)
    if descending:
        w = x.shape[-1]
        p = w - 1 - np.argsort(x[..., ::-1], axis=-1, kind="stable")[..., ::-1]
    else:
        p = np.argsort(x, axis=-1, kind="stable")
    return np.moveaxis(p, -1, axis)


def special_mix(n, name, seed=0):
    """n bit patterns of the type: half special values, a quarter uniform bits, a quarter normal values (integers:
    uniform bits), shuffled"""
    w = BITS[name]
    rng = np.random.default_rng([seed, w, len(name)])
    sp = special_bits(name)
    q = n // 4
    if name.startswith("float") or name == "bfloat16":
        vals = rng.standard_normal(q).astype(np.float32)
        norm = (vals.view(np.uint32) >> np.uint32(16)).astype(np.uint16) if name == "bfloat16" else vals.astype(NUMPY[name]).view(UINT[w])
    else:
        norm = rng.integers(0, 1 << w, q, dtype=np.uint64).astype(UINT[w])
    k = np.concatenate([sp[rng.integers(0, len(sp), n - 2 * q)], rng.integers(0, 1 << w, q, dtype=np.uint64).astype(UINT[w]),
                        norm])
    return k[rng.permutation(n)]


def torch_dtype(torch, name):
    return getattr(torch, name)


def to_device(torch, bits, name):
    """numpy bit patterns -> a CUDA tensor of the key type holding the same bits"""
    w = BITS[name]
    return torch.from_numpy(np.ascontiguousarray(bits, dtype=UINT[w]).view(SINT[w])).cuda().view(torch_dtype(torch, name))


def bits_of(torch, t):
    """a tensor of a narrow type -> its bit patterns as numpy uint32 / uint16"""
    w = t.element_size() * 8
    return t.view(torch.int32 if w == 32 else torch.int16).cpu().numpy().view(UINT[w])
