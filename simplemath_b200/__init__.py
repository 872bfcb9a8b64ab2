"""simplemath_b200 -- thin Python binding of libsmb200.so.

The product is the sm_100a CUDA engine behind the C ABI in include/smb200.h and
the drop-in C++ headers in include/sm/ (the reference, alielmorsy/simpleMath, is a
header-only C++ library).  Python here is glue for tests and bench.py only: it
loads the shared library with ctypes and passes raw addresses -- numpy buffers
(host memory, staged through HBM by the library) or torch CUDA tensors
(`tensor.data_ptr()`, used in place).

There is no CPU fallback: if the library is missing or no CUDA device is
usable, the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMB200_LIB") or os.path.join(HERE, "libsmb200.so")  # SMB200_LIB: a variant build (tools/ A/B runs)

OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_POW = range(5)
F32, F64, I32 = range(3)
MEM_DEVICE, MEM_MANAGED, MEM_PINNED = range(3)
# smb_set_option keys (include/smb200.h); 2, 3 and 10..13 are retired and not reused
OPT_POW_SPECIALISE = 0
OPT_STAGE_CHUNK_BYTES = 1
OPT_FORCE_WIDE_INDEX = 4
OPT_ASYNC = 5
OPT_PDL = 6
OPT_SHARD_MIN_BYTES = 7
OPT_REPLICATE_MAX_BYTES = 8
OPT_POOL_MAX_CACHED_BYTES = 9
PLAN_CONTIGUOUS, PLAN_ROW, PLAN_GENERIC = range(3)
MAX_NDIM = 6
CHAIN_MAX = 8

OPS = {"add": OP_ADD, "sub": OP_SUB, "mul": OP_MUL, "div": OP_DIV, "pow": OP_POW}
_NP_DTYPES = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.int32): I32}
_CT = {F32: ctypes.c_float, F64: ctypes.c_double, I32: ctypes.c_int32}
ELEM_SIZE = {F32: 4, F64: 8, I32: 4}

class _ChainValue(ctypes.Union):
    _fields_ = [("f32", ctypes.c_float), ("f64", ctypes.c_double), ("i32", ctypes.c_int32)]


class ChainStep(ctypes.Structure):
    """smb_chain_step of include/smb200.h."""
    _fields_ = [("op", ctypes.c_int32), ("swap", ctypes.c_int32), ("data", ctypes.c_void_p),
                ("stride", ctypes.c_uint64 * MAX_NDIM), ("value", _ChainValue)]


# every symbol include/smb200.h declares, with its ctypes signature
_u64, _vp, _i, _u64p = ctypes.c_uint64, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_uint64)
SYMBOLS = {
    "smb_elementwise": (_i, [_i, _i, _vp, _u64p, _vp, _u64p, _u64p, _i, _u64, _vp, _vp]),
    "smb_elementwise_range": (_i, [_i, _i, _vp, _u64p, _vp, _u64p, _u64p, _i, _u64, _u64, _vp, _vp]),
    "smb_contiguous": (_i, [_i, _i, _vp, _vp, _vp, _u64, _vp]),
    "smb_array_scalar": (_i, [_i, _i, _vp, _vp, _u64, _vp, _vp]),
    "smb_dot": (_i, [_i, _vp, _vp, _u64, _vp, _vp]),
    "smb_chain": (_i, [_i, ctypes.POINTER(ChainStep), _i, _u64p, _i, _u64, _vp, _vp]),
    "smb_chain_range": (_i, [_i, ctypes.POINTER(ChainStep), _i, _u64p, _i, _u64, _u64, _vp, _vp]),
    "smb_alloc": (_vp, [ctypes.c_size_t, _i]),
    "smb_free": (_i, [_vp]),
    "smb_owns": (_i, [_vp]),
    "smb_host_written": (_i, [_vp]),
    "smb_pool_trim": (_i, []),
    "smb_pool_stats": (_i, [_u64p]),
    "smb_fill": (_i, [_i, _vp, _vp, _u64, _vp]),
    "smb_prefetch": (_i, [_vp, ctypes.c_size_t, _i, _vp]),
    "smb_device_count": (_i, []),
    "smb_set_device": (_i, [_i]),
    "smb_get_device": (_i, []),
    "smb_sync": (_i, []),
    "smb_wait_pending": (_i, []),
    "smb_set_devices": (_i, [ctypes.POINTER(_i), _i]),
    "smb_get_devices": (_i, [ctypes.POINTER(_i), _i]),
    "smb_set_option": (_i, [_i, ctypes.c_int64]),
    "smb_get_option": (ctypes.c_int64, [_i]),
    "smb_launch_count": (_u64, []),
    "smb_last_kernel": (ctypes.c_char_p, []),
    "smb_last_error": (ctypes.c_char_p, []),
    "smb_version": (ctypes.c_char_p, []),
    "smb_plan_elementwise": (_i, [_u64p, _u64p, _u64p, _i, _i, ctypes.POINTER(_i), _u64p, _u64p, _u64p]),
    "smb_plan_chain": (_i, [ctypes.POINTER(ChainStep), _i, _u64p, _i, ctypes.POINTER(_i), _u64p, _u64p]),
    "smb_plan_shards": (_i, [_u64p, _u64p, _u64p, _i, _i, _i, _u64p, _u64p, _u64p, ctypes.POINTER(_i)]),
    "smb_register_op": (_i, [ctypes.c_char_p, _i, _vp]),
    "smb_find_op": (_i, [ctypes.c_char_p]),
    "smb_pow_audit_f32": (_i, [_vp, ctypes.c_float, _vp, _u64, ctypes.c_float, _u64p, ctypes.POINTER(ctypes.c_float)]),
    "smb_fill_uniform_f32": (_i, [_vp, _u64, _u64, _u64, ctypes.c_float, ctypes.c_float, _vp]),
}

_lib = None


class SmbError(RuntimeError):
    """Raised for any non-zero status of the C ABI (the C++ headers throw
    std::runtime_error in the same places)."""


def lib() -> ctypes.CDLL:
    """Load libsmb200.so.  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SmbError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise SmbError(f"smb200 error {rc}: {lib().smb_last_error().decode()}")


def dtype_code(dt) -> int:
    try:
        return _NP_DTYPES[np.dtype(dt)]
    except KeyError:
        raise SmbError(f"unsupported element type {dt}: the hot path carries float32, float64 and int32 only "
                       "(include/math/helpers.h:23-119 of the reference)") from None


def _u64arr(v: Sequence[int]):
    return (ctypes.c_uint64 * len(v))(*[int(x) for x in v])


# --------------------------------------------------------------------------
# Host mirror of sm::broadcast (include/SMUtils.h:34-99 of the reference).
def broadcast(shape1: Sequence[int], strides1: Sequence[int], shape2: Sequence[int], strides2: Sequence[int]):
    """Right-align ranks, pad with shape 1 / stride 0, stride 0 on broadcast dims.
    Returns (result_shape, new_strides1, new_strides2, total_size); raises
    SmbError with the reference's message on incompatible dims."""
    nd = max(len(shape1), len(shape2))
    o1, o2 = nd - len(shape1), nd - len(shape2)
    rs, s1, s2, total = [], [], [], 1
    for i in range(nd):
        d1, t1 = (1, 0) if i < o1 else (int(shape1[i - o1]), int(strides1[i - o1]))
        d2, t2 = (1, 0) if i < o2 else (int(shape2[i - o2]), int(strides2[i - o2]))
        if d1 != d2 and d1 != 1 and d2 != 1:
            raise SmbError("Cannot broadcast shapes: incompatible dimensions")
        if d1 == 1 and d2 > 1:
            t1 = 0
        if d2 == 1 and d1 > 1:
            t2 = 0
        rs.append(max(d1, d2))
        s1.append(t1)
        s2.append(t2)
        total *= rs[-1]
    return rs, s1, s2, total


def row_major_strides(shape: Sequence[int]) -> list[int]:
    """SMArray::calculateStride (include/SMArray.h:357-364): strides in elements."""
    out, cur = [0] * len(shape), 1
    for i in range(len(shape) - 1, -1, -1):
        out[i] = cur
        cur *= int(shape[i])
    return out


def plan(stride_a, stride_b, shape, elem_size=4):
    """Host planner only (no GPU): returns (kind, shape, stride_a, stride_b) after
    dimension coalescing."""
    nd = len(shape)
    ond = ctypes.c_int(0)
    osh, osa, osb = _u64arr([0] * MAX_NDIM), _u64arr([0] * MAX_NDIM), _u64arr([0] * MAX_NDIM)
    kind = lib().smb_plan_elementwise(_u64arr(stride_a), _u64arr(stride_b), _u64arr(shape), nd, elem_size,
                                      ctypes.byref(ond), osh, osa, osb)
    if kind < 0:
        raise SmbError(f"smb_plan_elementwise failed ({kind})")
    m = ond.value
    return kind, list(osh[:m]), list(osa[:m]), list(osb[:m])


def plan_shards(stride_a, stride_b, shape, ndev, elem_size=4):
    """Multi-GPU planner only (no GPU): (sharded?, bounds[ndev+1], ranges_a, ranges_b, (mode_a, mode_b)) for an
    smb_elementwise call spread over ndev devices; modes: 0 in place, 1 replicated, 2 refused."""
    nd = len(shape)
    bounds, ra, rb = _u64arr([0] * (ndev + 1)), _u64arr([0] * (2 * ndev)), _u64arr([0] * (2 * ndev))
    modes = (ctypes.c_int * 2)()
    rc = lib().smb_plan_shards(_u64arr(stride_a), _u64arr(stride_b), _u64arr(shape), nd, elem_size, ndev, bounds, ra, rb, modes)
    if rc < 0:
        raise SmbError(f"smb_plan_shards failed ({rc})")
    pairs = lambda v: [(int(v[2 * g]), int(v[2 * g + 1])) for g in range(ndev)]
    return bool(rc), [int(x) for x in bounds], pairs(ra), pairs(rb), (modes[0], modes[1])


# --------------------------------------------------------------------------
# Raw-pointer entry points (what the C++ headers call).
def elementwise_ptr(op, dtype, a_ptr, stride_a, b_ptr, stride_b, shape, out_ptr, stream=0):
    n = 1
    for d in shape:
        n *= int(d)
    _check(lib().smb_elementwise(op, dtype, a_ptr, _u64arr(stride_a), b_ptr, _u64arr(stride_b), _u64arr(shape),
                                 len(shape), n, out_ptr, stream or None))


def elementwise_range_ptr(op, dtype, a_ptr, stride_a, b_ptr, stride_b, shape, lin_begin, lin_count, out_ptr, stream=0):
    _check(lib().smb_elementwise_range(op, dtype, a_ptr, _u64arr(stride_a), b_ptr, _u64arr(stride_b), _u64arr(shape),
                                       len(shape), int(lin_begin), int(lin_count), out_ptr, stream or None))


def contiguous_ptr(op, dtype, a_ptr, b_ptr, out_ptr, n, stream=0):
    _check(lib().smb_contiguous(op, dtype, a_ptr, b_ptr, out_ptr, int(n), stream or None))


def array_scalar_ptr(op, dtype, a_ptr, scalar, n, out_ptr, stream=0):
    val = _CT[dtype](scalar)
    _check(lib().smb_array_scalar(op, dtype, a_ptr, ctypes.byref(val), int(n), out_ptr, stream or None))


def fill_uniform_f32_ptr(out_ptr, first, n, seed, lo, hi, stream=0):
    _check(lib().smb_fill_uniform_f32(out_ptr, int(first), int(n), int(seed), lo, hi, stream or None))


def pow_audit_f32_ptr(x_ptr, y, got_ptr, n, bound_ulp):
    """Exhaustive device-side audit of a float pow result: (elements above bound_ulp, largest error in ulps)."""
    cnt, worst = ctypes.c_uint64(0), ctypes.c_float(0)
    _check(lib().smb_pow_audit_f32(x_ptr, y, got_ptr, int(n), bound_ulp, ctypes.byref(cnt), ctypes.byref(worst)))
    return int(cnt.value), float(worst.value)


def set_option(key: int, value: int) -> None:
    _check(lib().smb_set_option(key, int(value)))


def launch_count() -> int:
    return int(lib().smb_launch_count())


def last_kernel() -> str:
    return lib().smb_last_kernel().decode()


def sync() -> None:
    _check(lib().smb_sync())


def device_count() -> int:
    return int(lib().smb_device_count())


def set_devices(devices: Sequence[int]) -> None:
    """smb_set_devices: spread every following operator on managed arrays over these GPUs
    (flat-range shards, broadcast operands replicated); [] or one entry = single device."""
    arr = (ctypes.c_int * max(len(devices), 1))(*devices)
    _check(lib().smb_set_devices(arr, len(devices)))


def get_devices() -> list[int]:
    arr = (ctypes.c_int * 64)()
    n = lib().smb_get_devices(arr, 64)
    return list(arr[:n])


# --------------------------------------------------------------------------
# numpy convenience layer: host buffers in, host buffer out, every byte of the
# computation on the GPU (the library stages host operands through HBM).
def _elem_strides(a: np.ndarray) -> list[int]:
    es = a.dtype.itemsize
    out = []
    for d, s in zip(a.shape, a.strides):
        if s < 0 or s % es:
            raise SmbError("negative or non-element strides are not representable (strides are size_t elements, "
                           "include/SMArray.h:357-364)")
        out.append(s // es if d > 1 else (s // es))
    return out


def binary(op, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """SMArray operator + - * / (include/SMArray.h:217-305) on numpy views:
    sm::broadcast -> fresh dense result -> element_wise_op."""
    op = OPS.get(op, op)
    if a.dtype != b.dtype:
        raise SmbError("operands must share one element type")
    dt = dtype_code(a.dtype)
    if a.ndim == 0 or b.ndim == 0:
        raise SmbError("rank-0 operands: use scalar()")
    shape, sa, sb, total = broadcast(a.shape, _elem_strides(a), b.shape, _elem_strides(b))
    if len(shape) > MAX_NDIM:
        raise SmbError(f"rank {len(shape)} > MAX_NDIM {MAX_NDIM}")
    out = np.empty(shape, dtype=a.dtype)
    if total and (a.size == 0 or b.size == 0):
        # sm::broadcast lets a 0-sized dim meet a 1 (result dim max(0,1) = 1, SMUtils.h:76-80) and the reference
        # then reads element 0 of an empty block; refuse instead of reading out of bounds
        raise SmbError("empty operand cannot be broadcast to a non-empty result")
    if total:
        elementwise_ptr(op, dt, a.ctypes.data, sa, b.ctypes.data, sb, shape, out.ctypes.data)
    return out


def scalar(op, a: np.ndarray, value) -> np.ndarray:
    """SMArray operator(T) / sm::pow(arr, T): array_scalar_op over the dense
    data[0..totalSize) (include/math/calculate.h:137-169)."""
    op = OPS.get(op, op)
    dt = dtype_code(a.dtype)
    a = np.ascontiguousarray(a)
    out = np.empty_like(a)
    if a.size:
        array_scalar_ptr(op, dt, a.ctypes.data, value, a.size, out.ctypes.data)
    return out


def dot(a: np.ndarray, b: np.ndarray):
    """SMArray::operator% (include/SMArray.h:213-215): sum(a[i]*b[i]) over the dense data."""
    if a.dtype != b.dtype or a.size != b.size:
        raise SmbError("dot: operands must share element type and size")
    dt = dtype_code(a.dtype)
    a, b = np.ascontiguousarray(a).ravel(), np.ascontiguousarray(b).ravel()
    res = _CT[dt]()
    _check(lib().smb_dot(dt, a.ctypes.data, b.ctypes.data, a.size, ctypes.byref(res), None))
    return a.dtype.type(res.value)


def dot_ptr(dtype, a_ptr, b_ptr, n, stream=0):
    res = _CT[dtype]()
    _check(lib().smb_dot(dtype, a_ptr, b_ptr, int(n), ctypes.byref(res), stream or None))
    return res.value


def chain_steps(dtype: int, leaves, shape):
    """Build the smb_chain_step array.  `leaves` = [(op, swap, leaf)], leaf = (ptr, strides) for an
    array broadcast against `shape` (strides already 0 on broadcast dims) or a Python scalar."""
    arr = (ChainStep * len(leaves))()
    for st, (op, swap, leaf) in zip(arr, leaves):
        st.op = OPS.get(op, op) if op is not None else 0
        st.swap = 1 if swap else 0
        if isinstance(leaf, tuple):
            st.data = leaf[0]
            for k, v in enumerate(leaf[1]):
                st.stride[k] = int(v)
        else:
            st.data = None
            if dtype == F32:
                st.value.f32 = leaf
            elif dtype == F64:
                st.value.f64 = leaf
            else:
                st.value.i32 = int(leaf)
    return arr


def plan_chain(dtype, leaves, shape):
    """Host planner of smb_chain only (no GPU): (vectorisable, coalesced shape, per-leaf coalesced strides)."""
    arr = chain_steps(dtype, leaves, shape)
    ond = ctypes.c_int(0)
    osh, ost = _u64arr([0] * MAX_NDIM), _u64arr([0] * (MAX_NDIM * len(leaves)))
    rc = lib().smb_plan_chain(arr, len(leaves), _u64arr(shape), len(shape), ctypes.byref(ond), osh, ost)
    if rc < 0:
        raise SmbError(f"smb_plan_chain failed ({rc})")
    m = ond.value
    return bool(rc), list(osh[:m]), [list(ost[i * MAX_NDIM:i * MAX_NDIM + m]) for i in range(len(leaves))]


def chain_ptr(dtype, leaves, shape, out_ptr, stream=0, lin_range=None):
    n = 1
    for d in shape:
        n *= int(d)
    arr = chain_steps(dtype, leaves, shape)
    if lin_range is None:
        _check(lib().smb_chain(dtype, arr, len(leaves), _u64arr(shape), len(shape), n, out_ptr, stream or None))
    else:
        _check(lib().smb_chain_range(dtype, arr, len(leaves), _u64arr(shape), len(shape), int(lin_range[0]),
                                     int(lin_range[1]), out_ptr, stream or None))


def chain(first: np.ndarray, *steps) -> np.ndarray:
    """Fused left-deep chain on numpy operands: chain(a, ("add", b), ("mul", 2.0), ("rsub", c), ("pow", 2.5)).
    A leading "r" swaps the operands of that step (leaf (op) acc).  Leaves broadcast NumPy-style
    against each other exactly as a sequence of SMArray operators would."""
    dt = dtype_code(first.dtype)
    arrays = [first] + [leaf for _, leaf in steps if isinstance(leaf, np.ndarray)]
    shape = list(np.broadcast_shapes(*[x.shape for x in arrays]))
    if len(shape) > MAX_NDIM:
        raise SmbError(f"rank {len(shape)} > MAX_NDIM {MAX_NDIM}")

    def leaf_of(x):
        if not isinstance(x, np.ndarray):
            return x
        if x.dtype != first.dtype:
            raise SmbError("operands must share one element type")
        pad = len(shape) - x.ndim
        st = [0] * pad + _elem_strides(x)
        dims = [1] * pad + list(x.shape)
        st = [0 if d == 1 and r > 1 else s for d, r, s in zip(dims, shape, st)]
        return (x.ctypes.data, st)

    leaves = [(None, False, leaf_of(first))]
    for op, leaf in steps:
        swap = op.startswith("r") and op[1:] in OPS
        leaves.append((op[1:] if swap else op, swap, leaf_of(leaf)))
    out = np.empty(shape, dtype=first.dtype)
    if out.size:
        chain_ptr(dt, leaves, shape, out.ctypes.data)
    return out


def pow(a: np.ndarray, y) -> np.ndarray:  # noqa: A001 - mirrors sm::pow
    return scalar(OP_POW, a, y)


# --------------------------------------------------------------------------
# Multi-GPU sharding of the flat output range (SURVEY.md §8e): rank g of G owns
# [begin, end); boundaries are multiples of `align` elements so every shard
# starts on a vector / row boundary.  No collective on the data path.
def shard_range(n: int, rank: int, world: int, align: int = 1) -> tuple[int, int]:
    if world < 1 or not (0 <= rank < world):
        raise SmbError("bad rank / world size")
    units = (n + align - 1) // align
    base, extra = divmod(units, world)
    ub = rank * base + min(rank, extra)
    ue = ub + base + (1 if rank < extra else 0)
    return min(ub * align, n), min(ue * align, n)
