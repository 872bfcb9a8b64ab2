"""Parity tests proper (need a B200): the CUDA path, called through the C ABI,
against the oracle / golden vectors.

Bars: bit-exact for int32 and for float/double + - * /; float/double pow within
the stated ULP bound of std::pow computed in higher precision
(stated: 1 ULP; pinned here at the measured maxima plus a margin, f32 <= 0.6 ULP vs double,
f64 <= 0.65 ULP vs long double).
"""
import ctypes

import numpy as np
import pytest

import oracle
import simplemath_b200 as smb
from conftest import assert_same_bits

pytestmark = pytest.mark.gpu

# The stated contract is 1 ULP; the kernels measure <= 0.56 (f32) / <= 0.61 (f64) over the host-compiled
# sweeps (tests/test_hostcheck.py), and the GPU tests pin THAT with a small margin, so a regression
# to "just under 1 ULP" fails here.
F32_POW_ULP_BOUND = 0.6
F64_POW_ULP_BOUND = 0.65


def _pow_close(got, a, y, dtype, orc):
    if dtype == np.float32:
        yv = np.asarray(y, np.float32)
        if yv.ndim == 0:
            err = oracle.ulp_error_f32(got.ravel(), orc.pow_ref_f32(a.ravel(), float(yv)))
        else:
            with np.errstate(all="ignore"):
                ref = np.power(a.astype(np.float64), np.broadcast_to(yv, got.shape).astype(np.float64))
            err = oracle.ulp_error_f32(got.ravel(), np.broadcast_to(ref, got.shape).ravel())
        return err.max() <= F32_POW_ULP_BOUND, err.max()
    yv = np.asarray(y, np.float64)
    if yv.ndim == 0:
        hi, lo = orc.pow_ref_f64(a.ravel(), float(yv))
        err = oracle.ulp_error_f64(got.ravel(), hi, lo)
        return err.max() <= F64_POW_ULP_BOUND, err.max()
    ref = np.power(np.broadcast_to(a, got.shape).astype(np.longdouble), np.broadcast_to(yv, got.shape).astype(np.longdouble))
    err = np.abs((got.astype(np.longdouble) - ref) / np.spacing(np.abs(ref.astype(np.float64)))).astype(np.float64)
    return err.max() <= F64_POW_ULP_BOUND + 0.5, err.max()


def test_every_golden_vector_through_the_c_abi(golden, orc):
    """All committed fixtures (produced by the unmodified reference)."""
    for c in golden.cases:
        a, b = c["a"], c["b"]
        es = a.dtype.itemsize
        dt = smb.dtype_code(a.dtype)
        out = np.empty(c["out"].shape, a.dtype)
        if c["kind"] == "elementwise":
            smb.elementwise_ptr(smb.OPS[c["op"]], dt, a.ctypes.data, c["sa"], b.ctypes.data, c["sb"], c["shape"], out.ctypes.data)
        else:
            smb.array_scalar_ptr(smb.OPS[c["op"]], dt, a.ctypes.data, b[0].item(), a.size, out.ctypes.data)
        what = f"golden case {c['idx']} ({c['kind']} {c['op']} {a.dtype})"
        if c["op"] == "pow" and a.dtype.kind == "f":
            if c["kind"] == "scalar":
                ok, worst = _pow_close(out, a, b[0], a.dtype.type, orc)
            else:
                av = np.lib.stride_tricks.as_strided(a, c["shape"], [s * es for s in c["sa"]])
                bv = np.lib.stride_tricks.as_strided(b, c["shape"], [s * es for s in c["sb"]])
                ok, worst = _pow_close(out, av, bv, a.dtype.type, orc)
            assert ok, (what, worst)
        else:
            assert_same_bits(out, c["out"], what)


SHAPES = [((1,), (1,)), ((1000,), (1000,)), ((100_003,), (100_003,)), ((33, 65), (1, 65)), ((33, 65), (33, 1)),
          ((33, 1), (1, 65)), ((12, 1, 40), (1, 9, 40)), ((5, 6, 7, 3), (1, 6, 1, 3)), ((2, 3, 4, 5, 6, 7), (2, 1, 4, 1, 6, 1)),
          ((400, 300), (300,)), ((64, 1024), (64, 1024)), ((3, 1, 4, 1, 5), (2, 1, 6, 1)), ((257, 129), (257, 129))]


def _operands(rng, dtype, op, s1, s2):
    if dtype == np.int32:
        lo, hi = (-2**31, 2**31) if op in ("add", "sub", "mul") else (-1000, 1001)
        a = rng.integers(lo, hi, size=s1, dtype=np.int64).astype(np.int32)
        if op == "div":
            b = (rng.integers(1, 98, size=s2) * rng.choice([-1, 1], size=s2)).astype(np.int32)
        elif op == "pow":
            a = rng.integers(-12, 13, size=s1).astype(np.int32)
            b = rng.integers(-4, 34, size=s2).astype(np.int32)
        else:
            b = rng.integers(lo, hi, size=s2, dtype=np.int64).astype(np.int32)
        return a, b
    if op == "pow":
        return rng.uniform(0.01, 50, size=s1).astype(dtype), rng.uniform(-4, 4, size=s2).astype(dtype)
    a = (rng.standard_normal(s1) * 10.0 ** rng.integers(-30, 30, size=s1)).astype(dtype)
    b = (rng.standard_normal(s2) * 10.0 ** rng.integers(-30, 30, size=s2)).astype(dtype)
    return a, b


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32])
@pytest.mark.parametrize("op", ["add", "sub", "mul", "div", "pow"])
def test_random_broadcast_vs_oracle(orc, dtype, op):
    rng = np.random.default_rng(hash((op, np.dtype(dtype).name, 1)) % 2**32)
    for s1, s2 in SHAPES:
        a, b = _operands(rng, dtype, op, s1, s2)
        got = smb.binary(op, a, b)
        if op == "pow" and dtype != np.int32:
            ok, worst = _pow_close(got, np.broadcast_to(a, got.shape), np.broadcast_to(b, got.shape), dtype, orc)
            assert ok, (op, s1, s2, worst)
        else:
            assert_same_bits(got, orc.binary(op, a, b), f"{op} {np.dtype(dtype).name} {s1}x{s2} [{smb.last_kernel()}]")
        v = b.ravel()[0].item()
        got = smb.scalar(op, a, v)
        if op == "pow" and dtype != np.int32:
            ok, worst = _pow_close(got, a, np.asarray(v, dtype), dtype, orc)
            assert ok, (op, s1, worst)
        else:
            assert_same_bits(got, orc.array_scalar(op, a, v), f"{op} scalar {np.dtype(dtype).name} {s1}")


def test_views_interior_pointers_and_transposes(orc):
    rng = np.random.default_rng(5)
    big = rng.standard_normal((4, 30, 20, 3)).astype(np.float32)
    small = rng.standard_normal((1, 30, 1, 3)).astype(np.float32)
    for k in range(4):
        v = big[k]                                   # interior pointer, parent strides
        assert_same_bits(smb.binary("add", v, small), orc.binary("add", v, small), f"view {k}")
    m = rng.standard_normal((37, 53)).astype(np.float32)
    n = rng.standard_normal((53, 37)).astype(np.float32)
    assert_same_bits(smb.binary("mul", m.T, n), orc.binary("mul", m.T, n), "transposed operand")
    assert smb.last_kernel().startswith("k_tile")
    w = rng.standard_normal((64, 100)).astype(np.float32)
    sl = w[:, 3:67]                                  # misaligned rows: inner stride 1, odd base offset
    assert_same_bits(smb.binary("sub", sl, sl), orc.binary("sub", sl, sl), "misaligned slice")
    odd = rng.standard_normal(4099).astype(np.float32)
    assert_same_bits(smb.binary("add", odd[1:], odd[:-1]), orc.binary("add", odd[1:], odd[:-1]), "operands misaligned differently")
    assert_same_bits(smb.binary("add", odd[3:], odd[3:]), orc.binary("add", odd[3:], odd[3:]), "common misalignment (peeled head)")


def test_reference_broadcast_test_shape(orc):
    """tests/add.cpp:59-92 at full size: ones(32,224,224,3)(0, SLICE_ALL) + {1,224,1,3}."""
    big = np.ones((2, 224, 224, 3), np.float32)
    two = np.full((1, 224, 1, 3), 3, np.float32)
    got = smb.binary("add", big[0], two)
    assert got.shape == (1, 224, 224, 3)
    assert_same_bits(got, np.full((1, 224, 224, 3), 4, np.float32))


def test_reference_int_pow_tests(orc):
    """tests/pow.cpp:46-99 through the C ABI."""
    a = np.full(2_000_000, 5, np.int32)
    assert_same_bits(smb.pow(a, 3), np.full(2_000_000, 125, np.int32))
    alt = np.where(np.arange(5000) % 2 == 0, 5, -5).astype(np.int32)
    assert_same_bits(smb.pow(alt, 3), (alt.astype(np.int64) ** 3).astype(np.int32))
    assert_same_bits(smb.pow(alt, -2), np.zeros(5000, np.int32))


def test_int_pow_lane_and_tail_semantics(orc):
    bases = np.array([0, 1, -1, 2, -2, 3, -3, 5, -5, 7, 10, -10, 46340, 46341, -46341, 65536, 2**31 - 1, -2**31, 123, -77], np.int32)
    for e in (0, 1, 2, 3, 5, 13, 20, 31, 32, 33, 62, -1, -2, -31, 2**31 - 1, -2**31):
        for n in (1, 7, 8, 11, 16, 20, 1000, 1003):
            a = np.resize(bases, n).astype(np.int32)
            assert_same_bits(smb.pow(a, e), orc.array_scalar("pow", a, e), f"i32 pow e={e} n={n}")


@pytest.mark.parametrize("y", [2.0, 2.5, 0.5, -1.0, 3.0, -2.5, 1 / 3, 17.0, 100.5, -77.7, 1e-3, 0.1, 9.25, 255.0, -256.0, 256.5, 1000.0])
def test_pow_f32_ulp_general_kernel(orc, y):
    rng = np.random.default_rng(int(abs(y) * 1000) % 2**31)
    x = np.concatenate([rng.uniform(0.01, 100, 1 << 21).astype(np.float32),
                        rng.integers(1, 0x7f800000, 1 << 21, dtype=np.uint32).view(np.float32),
                        (1 + rng.uniform(-2e-2, 2e-2, 1 << 20)).astype(np.float32)])   # keeps large |y| on the fast core
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        got = smb.pow(x, y)
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)
    err = oracle.ulp_error_f32(got, orc.pow_ref_f32(x, y))
    assert err.max() <= F32_POW_ULP_BOUND, (y, err.max(), x[err.argmax()], got[err.argmax()])
    if y in (2.0, 0.5, -1.0):  # the specialised exact forms agree within the same bound
        err = oracle.ulp_error_f32(smb.pow(x, y), orc.pow_ref_f32(x, y))
        assert err.max() <= 0.5 + 1e-6, (y, err.max())


@pytest.mark.parametrize("y", [2.0, 2.5, 0.5, -1.0, 1 / 3, 17.0, -77.7, 1e-3])
def test_pow_f64_ulp_general_kernel(orc, y):
    rng = np.random.default_rng(int(abs(y) * 1000) % 2**31 + 7)
    x = np.concatenate([rng.uniform(0.01, 100, 1 << 19), rng.integers(1, 0x7ff0000000000000, 1 << 19, dtype=np.uint64).view(np.float64)])
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        got = smb.pow(x, y)
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)
    hi, lo = orc.pow_ref_f64(x, y)
    err = oracle.ulp_error_f64(got, hi, lo)
    # results comfortably inside the normal range (what the fast core takes): the pinned bound.  Results that are
    # denormal or within 2^22 of the underflow / overflow thresholds go through the double-double path, whose
    # final scaling rounds a second time there: the stated 1 ULP
    inside = (np.abs(hi) >= 2.0 ** -1000) & (np.abs(hi) <= 2.0 ** 1000)
    assert err[inside].max() <= F64_POW_ULP_BOUND, (y, err[inside].max(), x[inside][err[inside].argmax()])
    assert err.max() <= 1.0, (y, err.max(), x[err.argmax()])


def test_pow_special_case_table_on_device(orc):
    xs = np.array([0.0, -0.0, 1.0, -1.0, 2.0, -2.0, 0.5, -0.5, 3.0, -3.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 3.4e38,
                   -3.4e38, 1.17549435e-38, 0.99999994, 1.0000001], np.float32)
    ys = [0.0, -0.0, 1.0, -1.0, 2.0, -2.0, 3.0, -3.0, 0.5, -0.5, 2.5, -2.5, np.inf, -np.inf, np.nan, 1e30, -1e30, 16777216.0,
          16777217.0, 4294967296.0, 1e-30, 127.0, -149.0, 1 / 3]
    for spec in (0, 1):
        smb.set_option(smb.OPT_POW_SPECIALISE, spec)
        for y in ys:
            got = smb.pow(xs, np.float32(y))
            want64 = orc.pow_ref_f32(xs, float(np.float32(y)))
            with np.errstate(all="ignore"):
                want = want64.astype(np.float32)
            for xi, g, w, w64 in zip(xs, got, want, want64):
                if np.isnan(w):
                    assert np.isnan(g), (xi, y, g)
                elif np.isinf(w) or w == 0 or np.isinf(g) or g == 0:
                    ok = g == w and np.signbit(g) == np.signbit(w)
                    assert ok or oracle.ulp_error_f32(np.array([g]), np.array([w64]))[0] <= 1, (xi, y, g, w)
                else:
                    assert oracle.ulp_error_f32(np.array([g]), np.array([w64]))[0] <= 1, (xi, y, g, w)
    smb.set_option(smb.OPT_POW_SPECIALISE, 1)


def test_float_specials_bit_exact(orc):
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.1754942e-38, 3.4028235e38, -3.4028235e38, 1.0, -1.5,
                   5.9e-39, 1e-40], np.float32)
    A, B = [np.ascontiguousarray(v.ravel()) for v in np.meshgrid(sp, sp, indexing="ij")]
    for op in ("add", "sub", "mul", "div"):
        assert_same_bits(smb.binary(op, A, B), orc.binary(op, A, B), f"f32 specials {op}")
        assert_same_bits(smb.binary(op, A.astype(np.float64), B.astype(np.float64)),
                         orc.binary(op, A.astype(np.float64), B.astype(np.float64)), f"f64 specials {op}")


def test_empty_and_rejects():
    e = np.empty((0, 5), np.float32)
    assert smb.binary("add", e, e).shape == (0, 5)
    with pytest.raises(smb.SmbError, match="empty operand"):
        smb.binary("add", e, np.ones((1, 5), np.float32))  # the reference would read a[0] of an empty block
    assert smb.scalar("mul", np.empty(0, np.int32), 3).size == 0
    with pytest.raises(smb.SmbError, match="Cannot broadcast"):
        smb.binary("add", np.ones((2, 3), np.float32), np.ones((4, 3), np.float32))
    with pytest.raises(smb.SmbError, match="unsupported element type"):
        smb.binary("add", np.ones(4, np.int64), np.ones(4, np.int64))
    with pytest.raises(smb.SmbError):
        smb.elementwise_ptr(9, smb.F32, 0, [1], 0, [1], [4], 0)


def test_staging_pipeline_many_chunks(orc):
    """Host operands larger than the staging chunk: slabs overlap on 3 streams."""
    rng = np.random.default_rng(9)
    smb.set_option(smb.OPT_STAGE_CHUNK_BYTES, 1 << 16)
    try:
        a = rng.standard_normal((301, 1000)).astype(np.float32)
        row = rng.standard_normal((1, 1000)).astype(np.float32)
        col = rng.standard_normal((301, 1)).astype(np.float32)
        assert_same_bits(smb.binary("add", a, a[::-1].copy()), orc.binary("add", a, a[::-1].copy()), "chunked contiguous")
        assert_same_bits(smb.binary("mul", a, row), orc.binary("mul", a, row), "chunked row broadcast")
        assert_same_bits(smb.binary("sub", col, row), orc.binary("sub", col, row), "chunked outer")
        x = rng.integers(-9, 10, size=100_003).astype(np.int32)
        assert_same_bits(smb.pow(x, 5), orc.array_scalar("pow", x, 5), "chunked i32 pow keeps lane/tail split")
        ia = rng.integers(-1000, 1000, size=(40, 1, 256)).astype(np.int32)
        ib = rng.integers(1, 98, size=(1, 50, 256)).astype(np.int32)
        assert_same_bits(smb.binary("div", ia, ib), orc.binary("div", ia, ib), "chunked 3-D")
    finally:
        smb.set_option(smb.OPT_STAGE_CHUNK_BYTES, 64 << 20)


def test_reused_broadcast_operand_vector_row_kernel(orc):
    """A small reused operand (a row, a column, a 4-D view's small factor) is read through L1/L2 by
    the row kernel (k_row<vec16> for the aligned rows); same bits as the oracle."""
    rng = np.random.default_rng(21)
    a = rng.standard_normal((300, 1024)).astype(np.float32)
    row = rng.standard_normal((1, 1024)).astype(np.float32)
    assert_same_bits(smb.binary("add", a, row), orc.binary("add", a, row), "reused b")
    assert smb.last_kernel() == "k_row<vec16>"
    assert_same_bits(smb.binary("sub", row, a), orc.binary("sub", row, a), "reused a")
    assert smb.last_kernel() == "k_row<vec16>"
    big = rng.integers(-99, 99, size=(4, 64, 20, 4)).astype(np.int32)
    small = rng.integers(1, 9, size=(1, 64, 1, 4)).astype(np.int32)
    assert_same_bits(smb.binary("mul", big[2], small), orc.binary("mul", big[2], small), "4-D view, small reused operand")
    col = rng.standard_normal((300, 1)).astype(np.float32)
    assert_same_bits(smb.binary("mul", a, col), orc.binary("mul", a, col), "inner-broadcast reused operand")


def test_outer_broadcast_kernel_and_row_fallback(orc):
    """{D0,1,L} (op) {1,D1,L} (config C4's pattern) takes the register-tiled k_outer kernel:
    both operand orders, non-commutative ops, ragged tile edges, slab-aligned shards; rows that
    are not vector-aligned and ranges that are not whole slabs fall back to k_row, same bits."""
    torch = _torch()
    rng = np.random.default_rng(41)
    for d0, d1, L in ((5, 7, 40), (16, 16, 1024), (3, 130, 12), (33, 2, 2052)):
        x = rng.integers(-1000, 1001, size=(d0, 1, L)).astype(np.int32)
        y = rng.integers(1, 98, size=(1, d1, L)).astype(np.int32)
        for op in ("sub", "div", "mul"):
            assert_same_bits(smb.binary(op, x, y), orc.binary(op, x, y), f"outer {op} a-on-dim0 {d0}x{d1}x{L}")
            assert smb.last_kernel() == "k_outer<4x4>", smb.last_kernel()
            assert_same_bits(smb.binary(op, y, x + (x == 0)), orc.binary(op, y, x + (x == 0)), f"outer {op} b-on-dim0")
            assert smb.last_kernel() == "k_outer<4x4>"
        xf, yf = x.astype(np.float64), y.astype(np.float64)
        assert_same_bits(smb.binary("div", xf, yf), orc.binary("div", xf, yf), "outer f64")
    # not vector-aligned rows -> k_row; results identical
    x = rng.integers(-9, 9, size=(6, 1, 37)).astype(np.int32)
    y = rng.integers(1, 9, size=(1, 5, 37)).astype(np.int32)
    assert_same_bits(smb.binary("mul", x, y), orc.binary("mul", x, y), "odd row length")
    assert smb.last_kernel().startswith("k_row")
    # shards: slab-aligned ranges use k_outer, others k_row
    x = rng.standard_normal((8, 1, 64)).astype(np.float32)
    y = rng.standard_normal((1, 6, 64)).astype(np.float32)
    want = orc.binary("sub", x, y).ravel()
    dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    shape, sa, sb, n = smb.broadcast(x.shape, smb.row_major_strides(x.shape), y.shape, smb.row_major_strides(y.shape))
    for lo, cnt, kern in ((0, n, "k_outer"), (2 * 6 * 64, 3 * 6 * 64, "k_outer"), (100, 1000, "k_row")):
        part = torch.empty(cnt, dtype=torch.float32, device="cuda")
        smb.elementwise_range_ptr(smb.OP_SUB, smb.F32, dx.data_ptr(), sa, dy.data_ptr(), sb, shape, lo, cnt, part.data_ptr())
        assert smb.last_kernel().startswith(kern), (lo, cnt, smb.last_kernel())
        assert_same_bits(part.cpu().numpy(), want[lo:lo + cnt], f"range {lo}+{cnt}")


def test_outer_int_division_by_reciprocal_full_range(orc):
    """k_outer divides int32 by a precomputed double reciprocal (one multiply per quotient):
    bit-exact with C truncating division over the full operand range, exact multiples, +-1
    around multiples and the extreme values (b != 0, not INT_MIN / -1: undefined in the reference)."""
    rng = np.random.default_rng(43)
    L = 1024
    edge = np.array([-2**31, -2**31 + 1, 2**31 - 1, 2**31 - 2, -1, 1, 2, -2, 3, -3, 7, 65535, 65536, -65536, 46341, -46341], np.int64)
    cases = []
    a = rng.integers(-2**31, 2**31, size=(16, 1, L)); b = rng.integers(-2**31, 2**31, size=(1, 12, L)); cases.append((a, b))
    b = rng.integers(-2**16, 2**16, size=(1, 12, L)); k = rng.integers(-2**15, 2**15, size=(16, 1, L)); cases.append((k * b[:, :1, :], b))
    b = rng.integers(-1000, 1000, size=(1, 8, L)); k = rng.integers(-2**20, 2**20, size=(8, 1, L)); cases.append((k * b[:, :1, :] + rng.integers(-1, 2, size=(8, 1, L)), b))
    cases.append((np.resize(edge, (16, 1, L)), np.resize(np.roll(np.repeat(edge, 16), 3), (1, 16, L))))
    for a, b in cases:
        a = np.clip(a, -2**31 + 1, 2**31 - 1).astype(np.int32)   # keeps INT_MIN / -1 out
        b = np.where(b == 0, 3, np.clip(b, -2**31, 2**31 - 1)).astype(np.int32)
        assert_same_bits(smb.binary("div", a, b), orc.binary("div", a, b), "outer div, divisor on dim 1")
        assert smb.last_kernel() == "k_outer<4x4>", smb.last_kernel()
        bt = np.ascontiguousarray(b.transpose(1, 0, 2)); at = np.ascontiguousarray(a.transpose(1, 0, 2))
        assert_same_bits(smb.binary("div", at, bt), orc.binary("div", at, bt), "outer div, divisor on dim 0")
        assert smb.last_kernel() == "k_outer<4x4>", smb.last_kernel()
    amin = np.full((4, 1, L), -2**31, np.int32)
    bb = rng.integers(2, 2**31, size=(1, 4, L)).astype(np.int32)
    assert_same_bits(smb.binary("div", amin, bb), orc.binary("div", amin, bb), "INT_MIN / b")


def test_transposed_operands_tile_kernel(orc):
    """SMArray::transpose() views (stride 1 along an earlier dim): shared-memory tile transpose."""
    rng = np.random.default_rng(61)
    for r, c in ((37, 53), (64, 64), (1, 200), (200, 1), (129, 1025), (1000, 33)):
        m = rng.standard_normal((c, r)).astype(np.float32)      # m.T has shape {r, c}, strides {1, r}
        n = rng.standard_normal((r, c)).astype(np.float32)
        for op in ("sub", "div"):
            assert_same_bits(smb.binary(op, m.T, n), orc.binary(op, m.T, n), f"a^T {op} b {r}x{c}")
            assert_same_bits(smb.binary(op, n, m.T), orc.binary(op, n, m.T), f"a {op} b^T {r}x{c}")
            assert_same_bits(smb.binary(op, m.T, m.T * 2), orc.binary(op, m.T, m.T * 2), f"a^T {op} (2a)^T")
        if r > 1 and c > 1:
            smb.binary("add", m.T, n)
            assert smb.last_kernel() == "k_tile<transpose>", smb.last_kernel()
        row = rng.standard_normal((1, c)).astype(np.float32)
        assert_same_bits(smb.binary("mul", m.T, row), orc.binary("mul", m.T, row), "a^T * row")
        col = rng.standard_normal((r, 1)).astype(np.float32)
        assert_same_bits(smb.binary("mul", col, m.T), orc.binary("mul", col, m.T), "col * a^T")
    # 3-D full transpose (reversed dims) against a dense operand, int32 and f64
    for dt in (np.int32, np.float64):
        x = (rng.standard_normal((7, 40, 33)) * 100).astype(dt)
        y = (rng.standard_normal((33, 40, 7)) * 100).astype(dt)
        assert_same_bits(smb.binary("add", x.T, y), orc.binary("add", x.T, y), f"3-D reversed {np.dtype(dt).name}")
        assert smb.last_kernel() == "k_tile<transpose>", smb.last_kernel()
        assert_same_bits(smb.binary("sub", x.transpose(0, 2, 1), x.transpose(0, 2, 1)), orc.binary("sub", x.transpose(0, 2, 1), x.transpose(0, 2, 1)), "batched transpose")
    # a strided slice that is not a transpose stays on the generic kernel
    w = rng.standard_normal((64, 100)).astype(np.float32)
    assert_same_bits(smb.binary("add", w[:, ::2], w[:, 1::2]), orc.binary("add", w[:, ::2], w[:, 1::2]), "stride-2 columns")
    assert smb.last_kernel().startswith("k_sgather")      # {64,50} with strides {100,2} coalesces to one stride-2 dim of 3200
    assert_same_bits(smb.binary("add", w[:, ::7], w[:, 1::7]), orc.binary("add", w[:, ::7], w[:, 1::7]), "stride-7 columns")
    assert smb.last_kernel().startswith("k_generic")


def test_small_inner_strides_vector_gather_kernel(orc):
    """w[:, ::2] + w[:, 1::2] and friends: inner strides 0..4 (f64: 0..2) take k_sgather -- aligned 16-byte loads,
    elements picked in registers -- for every operand phase; anything it cannot take stays on k_generic."""
    torch = _torch()
    rng = np.random.default_rng(71)
    for dtype, tdt in ((np.float32, torch.float32), (np.int32, torch.int32), (np.float64, torch.float64)):
        epv = 16 // np.dtype(dtype).itemsize
        rows, cols = 37, 96 * epv
        hw = (rng.standard_normal(rows * cols + 16) * 100).astype(dtype)
        dw = torch.from_numpy(hw).cuda()
        es = hw.itemsize
        for s_a in range(0, epv + 1):
            for s_b in range(0, epv + 1):
                if max(s_a, s_b) < 2:
                    continue
                L = cols // max(s_a, s_b, 1)
                L -= L % epv
                for off_a in range(epv):
                    off_b = (off_a * 3 + 1) % epv
                    va = np.lib.stride_tricks.as_strided(hw[off_a:], (rows, L), (cols * es, s_a * es))
                    vb = np.lib.stride_tricks.as_strided(hw[off_b:], (rows, L), (cols * es, s_b * es))
                    want = orc.elementwise("sub", hw[off_a:], [cols, s_a], hw[off_b:], [cols, s_b], [rows, L]).reshape(rows, L)
                    assert_same_bits(want, (va - vb).astype(dtype), "oracle == numpy on the strided views")
                    out = torch.empty(rows * L, dtype=tdt, device="cuda")
                    smb.elementwise_ptr(smb.OP_SUB, smb.dtype_code(dtype), dw.data_ptr() + off_a * es, [cols, s_a],
                                        dw.data_ptr() + off_b * es, [cols, s_b], [rows, L], out.data_ptr())
                    assert smb.last_kernel() == "k_sgather", (dtype, s_a, s_b, off_a, smb.last_kernel())
                    assert_same_bits(out.cpu().numpy().reshape(rows, L), want, f"sgather {np.dtype(dtype).name} strides {s_a},{s_b} phases {off_a},{off_b}")
    # 3-D with a broadcast outer dim, flat sub-ranges (shards), and the fallbacks
    hw = rng.standard_normal(8 * 16 * 64).astype(np.float32)
    dw = torch.from_numpy(hw).cuda()
    hb = rng.standard_normal(16 * 32).astype(np.float32)
    db = torch.from_numpy(hb).cuda()
    shape, sa, sb = [8, 16, 32], [16 * 64, 64, 2], [0, 32, 1]
    want = orc.elementwise("mul", hw, sa, hb, sb, shape).ravel()
    out = torch.empty(8 * 16 * 32, dtype=torch.float32, device="cuda")
    smb.elementwise_ptr(smb.OP_MUL, smb.F32, dw.data_ptr(), sa, db.data_ptr(), sb, shape, out.data_ptr())
    assert smb.last_kernel() == "k_sgather"
    assert_same_bits(out.cpu().numpy(), want, "3-D strided x broadcast")
    part = torch.empty(1024, dtype=torch.float32, device="cuda")
    smb.elementwise_range_ptr(smb.OP_MUL, smb.F32, dw.data_ptr(), sa, db.data_ptr(), sb, shape, 512, 1024, part.data_ptr())
    assert smb.last_kernel() == "k_sgather"
    assert_same_bits(part.cpu().numpy(), want[512:1536], "strided, flat sub-range")
    smb.elementwise_range_ptr(smb.OP_MUL, smb.F32, dw.data_ptr(), sa, db.data_ptr(), sb, shape, 510, 1024, part.data_ptr())
    assert smb.last_kernel() == "k_generic"     # range not on a vector boundary
    assert_same_bits(part.cpu().numpy(), want[510:1534], "strided, ragged sub-range")
    smb.elementwise_ptr(smb.OP_MUL, smb.F32, dw.data_ptr(), [16 * 64, 64, 5], db.data_ptr(), sb, [8, 16, 12], out.data_ptr())
    assert smb.last_kernel() == "k_generic"     # stride 5 > 4
    assert_same_bits(out.cpu().numpy()[:8 * 16 * 12], orc.elementwise("mul", hw, [16 * 64, 64, 5], hb, sb, [8, 16, 12]).ravel(), "stride 5")


def test_wide_index_path_on_small_shapes(orc):
    """The 64-bit index kernels (results beyond 2^31 elements) forced on small shapes."""
    rng = np.random.default_rng(31)
    smb.set_option(smb.OPT_FORCE_WIDE_INDEX, 1)
    try:
        for s1, s2 in SHAPES:
            a, b = _operands(rng, np.int32, "mul", s1, s2)
            assert_same_bits(smb.binary("mul", a, b), orc.binary("mul", a, b), f"wide {s1}x{s2} [{smb.last_kernel()}]")
        a = rng.standard_normal((64, 256)).astype(np.float32)
        row = rng.standard_normal((1, 256)).astype(np.float32)
        smb.binary("add", a, row)
        assert smb.last_kernel() == "k_row<vec16,wide>"
        m = rng.standard_normal((37, 53)).astype(np.float64)
        n = rng.standard_normal((53, 37)).astype(np.float64)
        w2 = rng.standard_normal((64, 100))
        assert_same_bits(smb.binary("div", w2[:, ::2], w2[:, 1::2]), orc.binary("div", w2[:, ::2], w2[:, 1::2]), "wide strided")
        assert smb.last_kernel() == "k_sgather<wide>"
        w3 = rng.standard_normal((64, 99))
        assert_same_bits(smb.binary("div", w3[:, ::3], w3[:, 1::3]), orc.binary("div", w3[:, ::3], w3[:, 1::3]), "wide generic")
        assert smb.last_kernel() == "k_generic<wide>"
    finally:
        smb.set_option(smb.OPT_FORCE_WIDE_INDEX, 0)


def test_result_beyond_2_31_elements(orc):
    """A real > 2^31-element result: {3, 2^30} + {1, 2^30} int32 (12 GiB out), sampled windows
    against the oracle plus a whole-array identity on the device."""
    torch = _torch()
    L = 1 << 30
    a = torch.empty(3 * L, dtype=torch.int32, device="cuda")
    b = torch.empty(L, dtype=torch.int32, device="cuda")
    out = torch.empty(3 * L, dtype=torch.int32, device="cuda")
    # deterministic fill: reuse the f32 generator's bit patterns as int32 data
    smb.fill_uniform_f32_ptr(a.data_ptr(), 0, 3 * L, 11, 1.0, 2.0)
    smb.fill_uniform_f32_ptr(b.data_ptr(), 0, L, 12, 1.0, 2.0)
    shape, sa, sb, n = smb.broadcast((3, L), (L, 1), (1, L), (L, 1))
    assert n == 3 * L > 2**31
    smb.elementwise_ptr(smb.OP_ADD, smb.I32, a.data_ptr(), sa, b.data_ptr(), sb, shape, out.data_ptr())
    assert smb.last_kernel() == "k_row<vec16,wide>"
    for row in range(3):
        assert bool((out[row * L:(row + 1) * L] == a[row * L:(row + 1) * L] + b).all())
    w = 1 << 16
    for start in (0, 2**31 - w // 2, 3 * L - w):
        ha = orc.fill_uniform_f32(start, w, 11, 1.0, 2.0).view(np.int32)
        hb = np.concatenate([orc.fill_uniform_f32((start + k) % L, w // 2, 12, 1.0, 2.0) for k in (0, w // 2)]).view(np.int32)
        want = orc.elementwise("add", ha, [1], hb, [1], [w])
        assert_same_bits(out[start:start + w].cpu().numpy(), want, f"window at {start}")


# ---- device-resident operands (torch owns the memory; the C ABI gets raw addresses) ----
def _torch():
    import torch
    return torch


def test_device_pointers_and_flat_range_sharding(orc):
    torch = _torch()
    rng = np.random.default_rng(12)
    a = rng.standard_normal((96, 1, 64)).astype(np.float32)
    b = rng.standard_normal((1, 40, 64)).astype(np.float32)
    want = orc.binary("mul", a, b).ravel()
    da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    shape, sa, sb, n = smb.broadcast(a.shape, smb.row_major_strides(a.shape), b.shape, smb.row_major_strides(b.shape))
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.elementwise_ptr(smb.OP_MUL, smb.F32, da.data_ptr(), sa, db.data_ptr(), sb, shape, out.data_ptr())
    assert_same_bits(out.cpu().numpy(), want, "device operands")
    # the same result assembled from 1, 2, 3, 8 flat-range shards (multi-GPU unit of work)
    for world in (1, 2, 3, 8):
        parts = []
        for r in range(world):
            lo, hi = smb.shard_range(n, r, world, align=256)
            part = torch.empty(hi - lo, dtype=torch.float32, device="cuda")
            smb.elementwise_range_ptr(smb.OP_MUL, smb.F32, da.data_ptr(), sa, db.data_ptr(), sb, shape, lo, hi - lo, part.data_ptr())
            parts.append(part)
        assert_same_bits(torch.cat(parts).cpu().numpy(), want, f"{world} shards")
    # unaligned range boundaries fall back to the scalar row kernel
    part = torch.empty(1001, dtype=torch.float32, device="cuda")
    smb.elementwise_range_ptr(smb.OP_MUL, smb.F32, da.data_ptr(), sa, db.data_ptr(), sb, shape, 777, 1001, part.data_ptr())
    assert_same_bits(part.cpu().numpy(), want[777:1778], "odd range")


def test_async_stream_and_generator(orc):
    torch = _torch()
    n = 1 << 20
    s = torch.cuda.Stream()
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    y = torch.empty(n, dtype=torch.float32, device="cuda")
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.fill_uniform_f32_ptr(x.data_ptr(), 0, n, 1, -1.0, 1.0, s.cuda_stream)
    smb.fill_uniform_f32_ptr(y.data_ptr(), 0, n, 2, -1.0, 1.0, s.cuda_stream)
    smb.contiguous_ptr(smb.OP_ADD, smb.F32, x.data_ptr(), y.data_ptr(), out.data_ptr(), n, s.cuda_stream)
    s.synchronize()
    hx, hy = orc.fill_uniform_f32(0, n, 1, -1.0, 1.0), orc.fill_uniform_f32(0, n, 2, -1.0, 1.0)
    assert_same_bits(x.cpu().numpy(), hx, "generator matches the oracle's")
    assert_same_bits(out.cpu().numpy(), orc.elementwise("add", hx, [1], hy, [1], [n]), "async add")


def test_pool_allocator_and_managed_memory(orc):
    lib = smb.lib()
    stats = (ctypes.c_uint64 * 4)()
    p = lib.smb_alloc(1 << 20, smb.MEM_MANAGED)
    assert p and lib.smb_owns(p) and lib.smb_owns(p + 4096) and not lib.smb_owns(p + (4 << 20))
    n = (1 << 20) // 4
    host = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_float)), shape=(n,))
    host[:] = np.arange(n, dtype=np.float32)           # written through the host mapping
    q = lib.smb_alloc(1 << 20, smb.MEM_MANAGED)
    smb.array_scalar_ptr(smb.OP_MUL, smb.F32, p, 0.5, n, q)
    res = np.ctypeslib.as_array(ctypes.cast(q, ctypes.POINTER(ctypes.c_float)), shape=(n,))
    assert_same_bits(res.copy(), np.arange(n, dtype=np.float32) * np.float32(0.5), "managed in/out")
    # interior pointer of a managed block as an operand (what a view hands over)
    smb.array_scalar_ptr(smb.OP_ADD, smb.F32, p + 4 * 1000, 1.0, 5000, q)
    assert_same_bits(res[:5000].copy(), np.arange(1000, 6000, dtype=np.float32) + 1, "interior pointer")
    assert lib.smb_free(p) == 0 and lib.smb_free(q) == 0
    lib.smb_pool_stats(stats)
    calls = stats[2]
    p2 = lib.smb_alloc(1 << 20, smb.MEM_MANAGED)       # recycled, no driver call
    lib.smb_pool_stats(stats)
    assert p2 in (p, q) and stats[2] == calls and stats[3] >= 1
    lib.smb_free(p2)
    assert lib.smb_free(12345) != 0                    # foreign pointer refused


# ---- BASELINE.json configs at full size: oracle on samples + size-independent properties ----
def test_config_c1_million_check(orc):
    a = np.ones(1_000_000, np.float32)
    assert_same_bits(smb.binary("add", a, a), np.full(1_000_000, 2, np.float32), "C1 as in benchmark/add.cpp:21-29")
    rng = np.random.default_rng(1)
    a, b = rng.uniform(-1, 1, 1_000_000).astype(np.float32), rng.uniform(-1, 1, 1_000_000).astype(np.float32)
    assert_same_bits(smb.binary("add", a, b), orc.binary("add", a, b), "C1 random")


def test_config_c2_row_broadcast_full(orc):
    rng = np.random.default_rng(1)
    a = rng.uniform(-1, 1, (4096, 4096)).astype(np.float32)
    b = np.random.default_rng(2).uniform(-1, 1, (1, 4096)).astype(np.float32)
    got = smb.binary("add", a, b)
    assert smb.last_kernel().startswith("k_row<vec16")
    assert_same_bits(got, orc.binary("add", a, b), "C2 full")


def test_config_c4_int_3d_broadcast_full(orc):
    torch = _torch()
    rng = np.random.default_rng(4)
    a = rng.integers(-1000, 1001, size=(512, 1, 1024)).astype(np.int32)
    bm = rng.integers(-2**31, 2**31, size=(1, 512, 1024), dtype=np.int64).astype(np.int32)
    bd = rng.integers(1, 98, size=(1, 512, 1024)).astype(np.int32)
    shape, sa, sb, n = smb.broadcast(a.shape, smb.row_major_strides(a.shape), bm.shape, smb.row_major_strides(bm.shape))
    assert n == 268435456
    da = torch.from_numpy(a).cuda()
    out = torch.empty(n, dtype=torch.int32, device="cuda")
    for op, b in ((smb.OP_MUL, bm), (smb.OP_DIV, bd)):
        db = torch.from_numpy(b).cuda()
        smb.elementwise_ptr(op, smb.I32, da.data_ptr(), sa, db.data_ptr(), sb, shape, out.data_ptr())
        o3 = out.view(512, 512, 1024)
        # sampled slabs against the oracle, bit-exact
        for i in (0, 1, 255, 511):
            want = orc.binary("mul" if op == smb.OP_MUL else "div", a[i:i + 1], b)
            assert_same_bits(o3[i:i + 1].cpu().numpy(), want, f"C4 slab {i}")
        # whole-output property: torch's own integer ops on the broadcast views agree everywhere
        ta, tb = da.view(512, 1, 1024), db.view(1, 512, 1024)
        ref = ta * tb if op == smb.OP_MUL else torch.div(ta, tb, rounding_mode="trunc")
        assert bool((o3 == ref).all())
        del ref


def test_config_c3_c5_large_pow_and_add_properties(orc):
    """256M-element f32 pow (C3) and 1 Gi-element add (C5 per-GPU at N=1 is 4 GiB
    arrays): sampled windows against the oracle + linear-time whole-array
    properties."""
    torch = _torch()
    n = 268_435_456
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.fill_uniform_f32_ptr(x.data_ptr(), 0, n, 3, 0.01, 100.0)
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for y in (2.0, 2.5):
            smb.array_scalar_ptr(smb.OP_POW, smb.F32, x.data_ptr(), y, n, out.data_ptr())
            for start in (0, 123_456_789, n - (1 << 20)):
                w = orc.fill_uniform_f32(start, 1 << 20, 3, 0.01, 100.0)
                got = out[start:start + (1 << 20)].cpu().numpy()
                err = oracle.ulp_error_f32(got, orc.pow_ref_f32(w, y))
                assert err.max() <= F32_POW_ULP_BOUND, (y, start, err.max())
            # EVERY element, on the device: error against |x|^y in double (the reference-accuracy pipeline
            # before its rounding), none above the bound -- the declined-element slow path included
            over, worst = smb.pow_audit_f32_ptr(x.data_ptr(), y, out.data_ptr(), n, F32_POW_ULP_BOUND)
            assert over == 0 and worst <= F32_POW_ULP_BOUND, (y, over, worst)
            # monotone in x for y > 0: sorting inputs sorts outputs (whole array, on device)
            idx = torch.argsort(x[: 1 << 24])
            assert bool((out[: 1 << 24][idx].diff() >= 0).all())
        # the reference benchmark's own fill, arr(i, j) = i + j + 1 on {16384, 16384} (benchmark/pow.cpp:33-47), audited whole
        ij = (torch.arange(16384, device="cuda", dtype=torch.float32)[:, None] + torch.arange(16384, device="cuda", dtype=torch.float32)[None, :] + 1).reshape(-1)
        torch.cuda.synchronize()   # torch filled it on ITS stream; the library's private stream does not wait for that one
        for y in (2.0, 2.5):
            smb.array_scalar_ptr(smb.OP_POW, smb.F32, ij.data_ptr(), y, n, out.data_ptr())
            over, worst = smb.pow_audit_f32_ptr(ij.data_ptr(), y, out.data_ptr(), n, F32_POW_ULP_BOUND)
            assert over == 0, (y, over, worst)
        del ij
        # every finite positive bit pattern class in one array (denormals, huge, tiny: the slow path's share)
        bits = torch.arange(n, device="cuda", dtype=torch.int32) * 7 + 1
        xb = bits.view(torch.float32)
        torch.cuda.synchronize()
        for y in (2.5, -0.5, 31.0):
            smb.array_scalar_ptr(smb.OP_POW, smb.F32, xb.data_ptr(), y, n, out.data_ptr())
            over, worst = smb.pow_audit_f32_ptr(xb.data_ptr(), y, out.data_ptr(), n, F32_POW_ULP_BOUND)
            assert over == 0, (y, over, worst)
        del bits, xb
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)
    # pow(x, 2) specialised == x*x exactly, everywhere
    smb.array_scalar_ptr(smb.OP_POW, smb.F32, x.data_ptr(), 2.0, n, out.data_ptr())
    assert bool((out == x * x).all())
    # add: (a + b) - b' == exact torch result everywhere (same IEEE op), checksum of the whole output
    y = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.fill_uniform_f32_ptr(y.data_ptr(), 0, n, 4, -1.0, 1.0)
    smb.contiguous_ptr(smb.OP_ADD, smb.F32, x.data_ptr(), y.data_ptr(), out.data_ptr(), n)
    assert bool((out == x + y).all())
    w = orc.fill_uniform_f32(n - 4096, 4096, 3, 0.01, 100.0), orc.fill_uniform_f32(n - 4096, 4096, 4, -1.0, 1.0)
    assert_same_bits(out[n - 4096:].cpu().numpy(), orc.elementwise("add", w[0], [1], w[1], [1], [4096]), "C5 add tail window")


def test_config_c3_f64_pow_at_256m(orc):
    """C3 in double at the stated size: 268 435 456 elements (2 GiB in, 2 GiB out), y = 2 (the reference
    benchmark's exponent) and 2.5: sampled windows against powl + whole-array properties."""
    torch = _torch()
    n = 268_435_456
    xf = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.fill_uniform_f32_ptr(xf.data_ptr(), 0, n, 3, 0.01, 100.0)
    x = xf.double()
    del xf
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for y in (2.0, 2.5):
            smb.array_scalar_ptr(smb.OP_POW, smb.F64, x.data_ptr(), y, n, out.data_ptr())
            for start in (0, 123_456_789, n - (1 << 19)):
                w = orc.fill_uniform_f32(start, 1 << 19, 3, 0.01, 100.0).astype(np.float64)
                hi, lo = orc.pow_ref_f64(w, y)
                err = oracle.ulp_error_f64(out[start:start + (1 << 19)].cpu().numpy(), hi, lo)
                assert err.max() <= F64_POW_ULP_BOUND, (y, start, err.max())
            idx = torch.argsort(x[: 1 << 24])
            assert bool((out[: 1 << 24][idx].diff() >= 0).all())
            # against torch's own double pow everywhere: both are within an ulp of the truth
            ref = torch.pow(x, y)
            rel = ((out - ref).abs() / ref.abs()).max().item()
            del ref
            assert rel <= 4 * 2.2204460492503131e-16, (y, rel)
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)
    smb.array_scalar_ptr(smb.OP_POW, smb.F64, x.data_ptr(), 2.0, n, out.data_ptr())
    assert bool((out == x * x).all())


# ---- SURVEY.md §8(f) row 2: dot product (SMArray::operator%) on the device --------------------
def test_dot_int32_bit_exact(orc):
    rng = np.random.default_rng(51)
    for n in (1, 3, 4, 5, 1000, 100_003, 1 << 22):
        a = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
        b = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
        assert smb.dot(a, b) == orc.dot(a, b), n
    assert smb.last_kernel() == "k_dot"


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_dot_float_within_tolerance_and_no_worse_than_the_reference(orc, dtype):
    """float/double: the device sums pairwise, the reference in 8 (4) sequential lanes; both are
    compared with the exactly rounded sum.  Tolerance: |err| <= 8 eps * sum|a_i b_i| (a loose
    pairwise-summation bound); in practice the device is closer than the reference."""
    import math
    rng = np.random.default_rng(52)
    eps = np.finfo(dtype).eps
    for n in (1, 7, 1000, 100_003, 1 << 22):
        a, b = rng.standard_normal(n).astype(dtype), rng.standard_normal(n).astype(dtype)
        prods = a.astype(np.float64) * b.astype(np.float64) if dtype == np.float32 else None
        exact = math.fsum(prods) if dtype == np.float32 else float(np.sum(a.astype(np.longdouble) * b.astype(np.longdouble)))
        bound = 8 * eps * float(np.sum(np.abs(a.astype(np.float64) * b.astype(np.float64)))) + 1e-300
        got, refv = float(smb.dot(a, b)), float(orc.dot(a, b))
        assert abs(got - exact) <= bound, (n, got, exact, bound)
        if n >= 100_003:
            assert abs(got - exact) <= abs(refv - exact) + bound * 1e-3, (n, got, refv, exact)
    a = rng.standard_normal(1 << 20).astype(dtype)
    assert smb.dot(a, a) == smb.dot(a, a)  # deterministic


def test_dot_device_pointers_and_sharded_sum(orc):
    torch = _torch()
    n = 1 << 24
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    y = torch.empty(n, dtype=torch.float32, device="cuda")
    smb.fill_uniform_f32_ptr(x.data_ptr(), 0, n, 5, -1.0, 1.0)
    smb.fill_uniform_f32_ptr(y.data_ptr(), 0, n, 6, -1.0, 1.0)
    full = smb.dot_ptr(smb.F32, x.data_ptr(), y.data_ptr(), n)
    ref = float((x.double() * y.double()).sum().item())
    assert abs(full - ref) <= 1e-6 * n ** 0.5 + 1e-3 * abs(ref)
    parts = 0.0
    for r in range(4):  # the multi-GPU form: per-shard partial sums + one tiny all-reduce
        lo, hi = smb.shard_range(n, r, 4, align=4)
        parts += smb.dot_ptr(smb.F32, x.data_ptr() + 4 * lo, y.data_ptr() + 4 * lo, hi - lo)
    assert abs(parts - ref) <= 1e-6 * n ** 0.5 + 1e-3 * abs(ref)


# ---- randomized views of device-resident parents: the kernels see the real base alignment and strides ----
def _random_view(rng, dtype, want_shape, op_is_divisor, friendly=False):
    """A numpy view with shape `want_shape` (1 = broadcast dim) cut out of a larger parent: random start, step and
    axis order per dim, optional leading-dim drop.  `friendly`: unit inner stride, inner start and row pitch on
    16 bytes (what the vector kernels need).  Returns (parent, view)."""
    nd = len(want_shape)
    perm = rng.permutation(nd) if (rng.random() < 0.35 and not friendly) else np.arange(nd)      # memory order of the parent's axes
    steps = [int(rng.choice([1, 1, 1, 1, 2, 3])) for _ in range(nd)]
    starts = [int(rng.integers(0, 4)) for _ in range(nd)]
    pshape = [starts[k] + (want_shape[k] - 1) * steps[k] + 1 + int(rng.integers(0, 3)) for k in range(nd)]
    if friendly:
        steps[-1], starts[-1] = 1, 4 * int(rng.integers(0, 3))
        pshape[-1] = (starts[-1] + want_shape[-1] + int(rng.integers(0, 3)) + 3) // 4 * 4
    mem_shape = [pshape[perm[k]] for k in range(nd)]
    n = int(np.prod(mem_shape))
    if dtype == np.int32:
        flat = rng.integers(1, 60, size=n).astype(np.int32) * rng.choice(np.array([-1, 1], np.int32), size=n) if op_is_divisor \
            else rng.integers(-2**31, 2**31, size=n, dtype=np.int64).astype(np.int32)
    else:
        flat = (rng.uniform(0.5, 3, size=n) * rng.choice([-1, 1], size=n)).astype(dtype) if op_is_divisor \
            else (rng.standard_normal(n) * 100).astype(dtype)
    parent = flat.reshape(mem_shape)
    logical = parent.transpose(np.argsort(perm))                                # axes back in logical order
    view = logical[tuple(slice(starts[k], starts[k] + (want_shape[k] - 1) * steps[k] + 1, steps[k]) for k in range(nd))]
    assert view.shape == tuple(want_shape)
    return parent, view


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32])
def test_fuzz_random_views_of_device_arrays_vs_oracle(orc, dtype):
    """~250 random (shape, broadcast pattern, slicing step, axis order, interior offset) pairs per dtype on DEVICE-resident
    parents, every operator, bit for bit against the oracle -- whichever kernel the planner picks."""
    torch = _torch()
    rng = np.random.default_rng(20261102 + np.dtype(dtype).itemsize + (7 if dtype == np.int32 else 0))
    dims = [1, 2, 3, 4, 5, 8, 12, 16, 24, 33, 64, 100]
    dt = smb.dtype_code(np.dtype(dtype))
    kernels = {}
    for case in range(250):
        nd = int(rng.integers(1, 6))
        shape = [int(rng.choice(dims)) for _ in range(nd)]
        while int(np.prod(shape)) > 400_000:
            shape[int(rng.integers(0, nd))] = 2
        op = ["add", "sub", "mul", "div"][case % 4]
        friendly = case % 3 == 0                                               # a third of the cases qualify for the vector kernels
        if friendly:
            shape[-1] = int(rng.choice([4, 8, 16, 64, 100]))
        views = []
        for o in range(2):
            want = [1 if rng.random() < 0.25 else d for d in shape]
            drop = int(rng.integers(0, nd)) if rng.random() < 0.2 else 0      # missing leading dims (rank padding)
            want = want[drop:]
            views.append(_random_view(rng, dtype, want, op == "div" and o == 1, friendly))
        (pa, va), (pb, vb) = views
        want = orc.binary(op, va, vb)
        dpa, dpb = torch.from_numpy(pa.copy()).cuda(), torch.from_numpy(pb.copy()).cuda()
        es = np.dtype(dtype).itemsize
        a_ptr = dpa.data_ptr() + (va.__array_interface__["data"][0] - pa.__array_interface__["data"][0])
        b_ptr = dpb.data_ptr() + (vb.__array_interface__["data"][0] - pb.__array_interface__["data"][0])
        rshape, sa, sb, total = smb.broadcast(va.shape, [s // es for s in va.strides], vb.shape, [s // es for s in vb.strides])
        assert tuple(rshape) == want.shape
        pad = 0 if friendly else int(rng.integers(0, 4))                       # the result may start off a vector boundary too
        out = torch.zeros(total + pad + 3, dtype={np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32}[dtype], device="cuda")
        torch.cuda.synchronize()
        smb.elementwise_ptr(smb.OPS[op], dt, a_ptr, sa, b_ptr, sb, rshape, out.data_ptr() + pad * es)
        k = smb.last_kernel()
        kernels[k] = kernels.get(k, 0) + 1
        host = out.cpu().numpy()
        assert_same_bits(host[pad:pad + total].reshape(want.shape), want,
                         f"case {case}: {op} {va.shape}/{va.strides} x {vb.shape}/{vb.strides} [{k}]")
        assert not host[:pad].any() and not host[pad + total:].any(), f"case {case}: wrote outside the result [{k}]"
    families = {k.split("<")[0] for k in kernels}
    assert {"k_row", "k_generic", "k_stream"} <= families, kernels
    assert "k_row<vec16>" in kernels and len(kernels) >= 6, kernels
