"""GPU tests of the runtime around the kernels (need a B200; called through the C ABI):

  * the parity holes the round-1 review named: 1-D stride-0 operands (SURVEY F11), operator% on
    misaligned views, the int32 pow step of a fused chain on a broadcast intermediate;
  * multi-GPU behind the operator API (smb_set_devices, SURVEY.md §8e): every operator spread over a
    device set, bit-identical to one device.  On a one-GPU box the set lists device 0 several times
    (each entry owns a flat range), which drives the whole sharded path -- range planning, placement
    records, read-mostly duplicates of shared operands, per-range launches; with >= 2 GPUs the same tests
    also run on distinct devices;
  * asynchronous hand-off (SMB_OPT_ASYNC), programmatic dependent launch on / off;
  * the exhaustive device-side pow audit.
"""
import ctypes

import numpy as np
import pytest

import oracle
import simplemath_b200 as smb
from conftest import assert_same_bits

pytestmark = pytest.mark.gpu

_CT = {np.dtype(np.float32): ctypes.c_float, np.dtype(np.float64): ctypes.c_double, np.dtype(np.int32): ctypes.c_int32}


class Managed:
    """A managed (cudaMallocManaged, pooled) block seen as a numpy array: what sm::SMArray<T>::data is."""

    def __init__(self, arr=None, shape=None, dtype=None):
        if arr is not None:
            arr = np.ascontiguousarray(arr)
            shape, dtype = arr.shape, arr.dtype
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape)
        n = int(np.prod(self.shape)) if len(self.shape) else 1
        self.ptr = smb.lib().smb_alloc(max(n, 1) * self.dtype.itemsize, smb.MEM_MANAGED)
        assert self.ptr, smb.lib().smb_last_error()
        self.np = np.ctypeslib.as_array(ctypes.cast(self.ptr, ctypes.POINTER(_CT[self.dtype])), shape=(max(n, 1),))[:n].reshape(self.shape)
        if arr is not None:
            self.np[...] = arr
            smb.lib().smb_host_written(self.ptr)

    def free(self):
        if self.ptr:
            smb.lib().smb_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _binary_managed(op, a: np.ndarray, b: np.ndarray):
    """smb_elementwise on managed operands / result (the SMArray operator path); returns the result as numpy."""
    dt = smb.dtype_code(a.dtype)
    shape, sa, sb, total = smb.broadcast(a.shape, smb.row_major_strides(a.shape), b.shape, smb.row_major_strides(b.shape))
    ma, mb, mo = Managed(a), Managed(b), Managed(shape=shape, dtype=a.dtype)
    smb.elementwise_ptr(smb.OPS[op], dt, ma.ptr, sa, mb.ptr, sb, shape, mo.ptr)
    smb.sync()
    out = mo.np.copy()
    kern = smb.last_kernel()
    for m in (ma, mb, mo):
        m.free()
    return out, kern


def _device_sets():
    n = smb.device_count()
    sets = [[0, 0], [0, 0, 0], [0] * 8]
    if n >= 2:
        sets += [[0, 1], list(range(n))]
    return sets


@pytest.fixture
def sharded():
    """Force sharding on small results; restore single-device behaviour afterwards."""
    old = smb.lib().smb_get_option(smb.OPT_SHARD_MIN_BYTES)
    smb.set_option(smb.OPT_SHARD_MIN_BYTES, 0)
    yield
    smb.set_devices([])
    smb.set_option(smb.OPT_SHARD_MIN_BYTES, old)


# ---------------------------------------------------------------- parity holes of round 1 ----
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32])
def test_f11_one_dim_stride_zero_operands(dtype):
    """{5} + {1} and {1} + {5} (reference calculate.h:10-13 takes its contiguous loop for every 1-D
    call and reads past the one-element operand; documented divergence: the stride table is honoured)."""
    rng = np.random.default_rng(3)
    for n in (5, 1, 8, 1003, 100_003):
        a = (rng.standard_normal(n) * 50).astype(dtype)
        one = (rng.standard_normal(1) * 7 + 9).astype(dtype)
        for op, f in (("add", np.add), ("sub", np.subtract), ("mul", np.multiply)):
            with np.errstate(all="ignore"):
                assert_same_bits(smb.binary(op, a, one), f(a, one).astype(dtype), f"{{{n}}} {op} {{1}}")
                assert_same_bits(smb.binary(op, one, a), f(one, a).astype(dtype), f"{{1}} {op} {{{n}}}")
            got, _ = _binary_managed(op, a, one)
            with np.errstate(all="ignore"):
                assert_same_bits(got, f(a, one).astype(dtype), f"managed {{{n}}} {op} {{1}}")


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32])
def test_dot_on_misaligned_views(orc, dtype):
    """SMArray::operator% hands interior pointers straight to dot_product (SMArray.h:208); the reference
    reads them with loadu (product.h:26-71).  Same phase -> peeled head, different phases -> the
    element-wise kernel; int32 is bit-exact either way."""
    import torch
    rng = np.random.default_rng(8)
    es = np.dtype(dtype).itemsize
    n = 100_003
    if dtype == np.int32:
        ha = rng.integers(-2**31, 2**31, n + 8, dtype=np.int64).astype(np.int32)
        hb = rng.integers(-2**31, 2**31, n + 8, dtype=np.int64).astype(np.int32)
    else:
        ha, hb = rng.standard_normal(n + 8).astype(dtype), rng.standard_normal(n + 8).astype(dtype)
    da, db = torch.from_numpy(ha).cuda(), torch.from_numpy(hb).cuda()
    dt = smb.dtype_code(dtype)
    for oa, ob, kern in ((0, 0, "k_dot"), (1, 1, "k_dot"), (3, 3, "k_dot"), (1, 2, "k_dot<unaligned>"), (0, 1, "k_dot<unaligned>"), (5, 2, "k_dot<unaligned>")):
        if (oa * es) % 16 == (ob * es) % 16:
            kern = "k_dot"
        for m in (n, 1, 2, 7):
            got = smb.dot_ptr(dt, da.data_ptr() + oa * es, db.data_ptr() + ob * es, m)
            va, vb = ha[oa:oa + m], hb[ob:ob + m]
            if dtype == np.int32:
                assert np.int32(got) == orc.dot(va, vb), (oa, ob, m)
            else:
                exact = float(np.sum(va.astype(np.longdouble) * vb.astype(np.longdouble)))
                bound = 8 * np.finfo(dtype).eps * float(np.sum(np.abs(va.astype(np.float64) * vb.astype(np.float64)))) + 1e-300
                assert abs(float(got) - exact) <= bound, (oa, ob, m, got, exact)
        assert smb.last_kernel() == kern, (oa, ob, smb.last_kernel())
    # host views (numpy slices): staged, any offset
    assert smb.dot(ha[1:n], hb[2:n + 1]) == (orc.dot(ha[1:n], hb[2:n + 1]) if dtype == np.int32 else smb.dot(ha[1:n].copy(), hb[2:n + 1].copy()))


def test_chain_int32_pow_on_broadcast_intermediate(orc):
    """sm::pow(lazy(a{1,N}), e) + B{M,N}: the unfused reference runs array_scalar_op over the N-element
    intermediate (lane/scalar split at N - N % 8, calculate.h:139-140); the fused call evaluates that
    prefix first.  Exponents that overflow or are negative tell the two semantics apart."""
    rng = np.random.default_rng(14)
    for N, M in ((13, 3), (16, 5), (1003, 7)):
        a = rng.integers(-12, 13, size=(1, N)).astype(np.int32)
        B = rng.integers(-1000, 1000, size=(M, N)).astype(np.int32)
        col = rng.integers(-5, 6, size=(M, 1)).astype(np.int32)
        for e in (3, 13, 31, 40, -1, -2):
            want = orc.binary("add", orc.array_scalar("pow", a, e), B)
            assert_same_bits(smb.chain(a, ("pow", e), ("add", B)), want, f"pow(a{{1,{N}}}, {e}) + B{{{M},{N}}}")
            want2 = orc.binary("mul", orc.array_scalar("pow", orc.array_scalar("add", a, 1), e), col)
            assert_same_bits(smb.chain(a, ("add", 1), ("pow", e), ("mul", col)), want2, f"pow(a + 1, {e}) * col")
            # two pow steps, the first on the smaller intermediate
            want3 = orc.array_scalar("pow", orc.binary("sub", orc.array_scalar("pow", a, e), B), 2)
            assert_same_bits(smb.chain(a, ("pow", e), ("sub", B), ("pow", 2)), want3, "pow(pow(a, e) - B, 2)")


# ------------------------------------------------- multi-GPU behind the operator API (§8e) ----
def test_sharded_elementwise_bit_identical(orc, sharded):
    rng = np.random.default_rng(77)
    cases = [((40_000,), (40_000,)), ((300, 257), (1, 257)), ((300, 257), (300, 1)), ((129, 1), (1, 65)),
             ((24, 1, 256), (1, 40, 256)), ((5, 6, 7, 3), (1, 6, 1, 3)), ((64, 64), (64, 64)), ((7, 2048), (2048,))]
    for devs in _device_sets():
        smb.set_devices(devs)
        assert smb.get_devices() == devs
        for s1, s2 in cases:
            for dtype, op in ((np.float32, "add"), (np.int32, "mul"), (np.float64, "div"), (np.int32, "div")):
                if dtype == np.int32:
                    a = rng.integers(-1000, 1001, size=s1).astype(np.int32)
                    b = (rng.integers(1, 98, size=s2) * rng.choice([-1, 1], size=s2)).astype(np.int32)
                else:
                    a, b = rng.standard_normal(s1).astype(dtype), (rng.standard_normal(s2) + 3).astype(dtype)
                got, kern = _binary_managed(op, a, b)
                assert_same_bits(got, orc.binary(op, a, b), f"{len(devs)} ranges {op} {np.dtype(dtype).name} {s1}x{s2} [{kern}]")


def test_sharded_transposed_operand_falls_back_to_one_device(orc, sharded):
    """An operand every device would need most of (a transpose) and that is too large to duplicate:
    the operator runs on one device -- same bits."""
    rng = np.random.default_rng(5)
    smb.set_devices([0, 0, 0, 0])
    old = smb.lib().smb_get_option(smb.OPT_REPLICATE_MAX_BYTES)
    smb.set_option(smb.OPT_REPLICATE_MAX_BYTES, 1024)
    try:
        m = rng.standard_normal((96, 200)).astype(np.float32)
        n = rng.standard_normal((200, 96)).astype(np.float32)
        dt = smb.F32
        ma, mb, mo = Managed(m), Managed(n), Managed(shape=(200, 96), dtype=np.float32)
        smb.elementwise_ptr(smb.OP_SUB, dt, ma.ptr, [1, 200], mb.ptr, [96, 1], [200, 96], mo.ptr)
        assert smb.last_kernel() == "k_tile<transpose>"
        assert_same_bits(mo.np.copy(), orc.binary("sub", m.T, n), "transposed operand, device set active")
        sharded_ok, _, _, _, modes = smb.plan_shards([1, 200], [96, 1], [200, 96], 4)
        assert not sharded_ok and modes[0] == 2
    finally:
        smb.set_option(smb.OPT_REPLICATE_MAX_BYTES, old)


def test_sharded_scalar_pow_chain_fill_dot(orc, sharded):
    rng = np.random.default_rng(78)
    lib = smb.lib()
    for devs in _device_sets():
        smb.set_devices(devs)
        n = 100_003
        # array (op) scalar incl. the int32 pow lane / scalar-tail split at the ABSOLUTE index
        for dtype, op, v in ((np.float32, "mul", 1.5), (np.int32, "pow", 5), (np.int32, "pow", 31), (np.int32, "pow", -2), (np.float64, "sub", 0.25)):
            a = rng.integers(-9, 10, n).astype(dtype) if dtype == np.int32 else rng.standard_normal(n).astype(dtype)
            ma, mo = Managed(a), Managed(shape=(n,), dtype=dtype)
            smb.array_scalar_ptr(smb.OPS[op], smb.dtype_code(dtype), ma.ptr, v, n, mo.ptr)
            assert_same_bits(mo.np.copy(), orc.array_scalar(op, a, v), f"{len(devs)} ranges scalar {op} {np.dtype(dtype).name}")
        # float pow, general kernel: every range stages its own tables
        x = rng.uniform(0.01, 100, n).astype(np.float32)
        mx, mo = Managed(x), Managed(shape=(n,), dtype=np.float32)
        smb.set_option(smb.OPT_POW_SPECIALISE, 0)
        try:
            smb.array_scalar_ptr(smb.OP_POW, smb.F32, mx.ptr, 2.5, n, mo.ptr)
        finally:
            smb.set_option(smb.OPT_POW_SPECIALISE, 1)
        assert oracle.ulp_error_f32(mo.np.copy(), orc.pow_ref_f32(x, 2.5)).max() <= 0.6
        # fused chain with a broadcast row leaf (shared: read-mostly duplicates) and a column leaf
        a = rng.standard_normal((300, 256)).astype(np.float32)
        row = rng.standard_normal((1, 256)).astype(np.float32)
        col = rng.standard_normal((300, 1)).astype(np.float32)
        ma, mr, mc, mo = Managed(a), Managed(row), Managed(col), Managed(shape=a.shape, dtype=np.float32)
        leaves = [(None, False, (ma.ptr, [256, 1])), ("mul", False, (mr.ptr, [0, 1])), ("add", False, (mc.ptr, [1, 0])), ("sub", False, 0.5)]
        smb.chain_ptr(smb.F32, leaves, list(a.shape), mo.ptr)
        want = orc.array_scalar("sub", orc.binary("add", orc.binary("mul", a, row), col), 0.5)
        assert_same_bits(mo.np.copy(), want, f"{len(devs)} ranges chain a*row+col-0.5 [{smb.last_kernel()}]")
        # fill (sm::ones) born partitioned, then used
        mf = Managed(shape=(n,), dtype=np.float32)
        one = ctypes.c_float(1.0)
        smb._check(lib.smb_fill(smb.F32, mf.ptr, ctypes.byref(one), n, None))
        assert bool((mf.np == 1.0).all())
        # dot: per-range partials added on the host; int32 wraps exactly
        ia = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
        ib = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)
        mia, mib = Managed(ia), Managed(ib)
        assert np.int32(smb.dot_ptr(smb.I32, mia.ptr, mib.ptr, n)) == orc.dot(ia, ib)
        fa, fb = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
        mfa, mfb = Managed(fa), Managed(fb)
        exact = float(np.sum(fa.astype(np.float64) * fb.astype(np.float64)))
        assert abs(smb.dot_ptr(smb.F32, mfa.ptr, mfb.ptr, n) - exact) <= 8 * np.finfo(np.float32).eps * float(np.sum(np.abs(fa * fb)))


def test_sharded_reuses_placement_and_results_feed_the_next_operator(orc, sharded):
    """c = a + b; d = c * row; e = d - c on a device set: results are born partitioned, an operand that
    is already where its range's device wants it is not prefetched again, and the answer is the
    single-device one."""
    rng = np.random.default_rng(79)
    smb.set_devices(_device_sets()[-1])
    R, C = 2048, 2048  # 16 MiB per array: every range is at least one 2 MiB page, so operands are sharded IN PLACE
    a = rng.standard_normal((R, C)).astype(np.float32)
    b = rng.standard_normal((R, C)).astype(np.float32)
    row = rng.standard_normal((1, C)).astype(np.float32)
    ma, mb, mr = Managed(a), Managed(b), Managed(row)
    mc, md, me = (Managed(shape=a.shape, dtype=np.float32) for _ in range(3))
    full, rowst = [C, 1], [0, 1]
    assert smb.plan_shards(full, full, [R, C], len(smb.get_devices()))[4] == (0, 0)
    for _ in range(3):
        smb.elementwise_ptr(smb.OP_ADD, smb.F32, ma.ptr, full, mb.ptr, full, [R, C], mc.ptr)
        smb.elementwise_ptr(smb.OP_MUL, smb.F32, mc.ptr, full, mr.ptr, rowst, [R, C], md.ptr)
        smb.elementwise_ptr(smb.OP_SUB, smb.F32, md.ptr, full, mc.ptr, full, [R, C], me.ptr)
    c = orc.binary("add", a, b)
    d = orc.binary("mul", c, row)
    assert_same_bits(me.np.copy(), orc.binary("sub", d, c), "three chained operators on a device set")
    # the host writes an operand in place (through `data`, as the reference's tests do) and says so
    ma.np[...] = b
    smb.lib().smb_host_written(ma.ptr)
    smb.elementwise_ptr(smb.OP_ADD, smb.F32, ma.ptr, full, mb.ptr, full, [R, C], mc.ptr)
    assert_same_bits(mc.np.copy(), orc.binary("add", b, b), "operand rewritten by the host between operators")


def test_sharded_shared_operand_sees_raw_host_writes(orc, sharded):
    """A shared operand (a broadcast row every device reads) is kept as read-mostly duplicates, which the driver
    invalidates on any write: after the host rewrites the row through its pointer WITHOUT smb_host_written (as
    SMArray::data allows), the next result sees the new values on every device."""
    rng = np.random.default_rng(80)
    R, C = 4096, 2048
    a = rng.standard_normal((R, C)).astype(np.float32)
    row = rng.standard_normal((1, C)).astype(np.float32)
    ma, mr, mo = Managed(a), Managed(row), Managed(shape=a.shape, dtype=np.float32)
    full, rowst = [C, 1], [0, 1]
    for devs in _device_sets():
        smb.set_devices(devs)
        assert smb.plan_shards(full, rowst, [R, C], len(devs))[4][1] == 1  # the row: a read-mostly duplicate per device
        for _ in range(2):  # the second call finds the partition and the duplicates in place
            smb.elementwise_ptr(smb.OP_ADD, smb.F32, ma.ptr, full, mr.ptr, rowst, [R, C], mo.ptr)
        assert_same_bits(mo.np.copy(), orc.binary("add", a, row), f"{len(devs)} ranges, row as first written")
        row = rng.standard_normal((1, C)).astype(np.float32)
        mr.np[...] = row
        smb.elementwise_ptr(smb.OP_ADD, smb.F32, ma.ptr, full, mr.ptr, rowst, [R, C], mo.ptr)
        assert_same_bits(mo.np.copy(), orc.binary("add", a, row), f"{len(devs)} ranges, row rewritten raw by the host")


# ------------------------------------------------------------- async hand-off, PDL on / off ----
def test_async_mode_and_pdl_variants(orc):
    """SMB_OPT_ASYNC: stream == NULL calls return before the kernels finish; results land at
    smb_wait_pending().  The same sequences with programmatic dependent launch on and off, including
    back-to-back launches WITH a data hazard (c = a + b; d = c * c) and without one."""
    import torch
    rng = np.random.default_rng(90)
    n = 1 << 22
    ha, hb = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
    a, b = torch.from_numpy(ha).cuda(), torch.from_numpy(hb).cuda()
    c, d, e, f = (torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(4))
    want_c = orc.elementwise("add", ha, [1], hb, [1], [n])
    want_d = orc.elementwise("mul", want_c, [1], want_c, [1], [n])
    want_e = orc.elementwise("sub", ha, [1], hb, [1], [n])
    want_f = orc.array_scalar("mul", want_d, 0.5)
    torch.cuda.synchronize()
    for pdl in (2, 1, 0):
        smb.set_option(smb.OPT_PDL, pdl)
        for asyn in (0, 1):
            smb.set_option(smb.OPT_ASYNC, asyn)
            for t in (c, d, e, f):
                t.zero_()
            torch.cuda.synchronize()
            for _ in range(4):  # repeated: write-after-write and read-after-write hazards between launches
                smb.contiguous_ptr(smb.OP_ADD, smb.F32, a.data_ptr(), b.data_ptr(), c.data_ptr(), n)      # no hazard with what follows it the first time
                smb.contiguous_ptr(smb.OP_MUL, smb.F32, c.data_ptr(), c.data_ptr(), d.data_ptr(), n)      # reads c: must wait
                smb.contiguous_ptr(smb.OP_SUB, smb.F32, a.data_ptr(), b.data_ptr(), e.data_ptr(), n)      # independent: may overlap
                smb.array_scalar_ptr(smb.OP_MUL, smb.F32, d.data_ptr(), 0.5, n, f.data_ptr())             # reads d
            smb._check(smb.lib().smb_wait_pending())
            tag = f"pdl={pdl} async={asyn}"
            assert_same_bits(c.cpu().numpy(), want_c, "c " + tag)
            assert_same_bits(d.cpu().numpy(), want_d, "d " + tag)
            assert_same_bits(e.cpu().numpy(), want_e, "e " + tag)
            assert_same_bits(f.cpu().numpy(), want_f, "f " + tag)
    smb.set_option(smb.OPT_ASYNC, 0)
    smb.set_option(smb.OPT_PDL, 1)
    # in-place update chains: x = x + b, repeated (every launch depends on the one before)
    x = a.clone()
    want = ha.copy()
    smb.set_option(smb.OPT_ASYNC, 1)
    try:
        for _ in range(5):
            smb.contiguous_ptr(smb.OP_ADD, smb.F32, x.data_ptr(), b.data_ptr(), x.data_ptr(), n)
            want = orc.elementwise("add", want, [1], hb, [1], [n])
    finally:
        smb.set_option(smb.OPT_ASYNC, 0)  # waits
    assert_same_bits(x.cpu().numpy(), want, "x += b five times, async")


def test_async_mode_recycles_pool_blocks_in_stream_order(orc):
    """The operator pattern of the C++ headers in an async scope: every result is a fresh pooled block,
    temporaries are freed while their kernels may still be running, and the freed block is handed out
    again at once."""
    rng = np.random.default_rng(91)
    lib = smb.lib()
    n = 1 << 20
    ha = rng.standard_normal(n).astype(np.float32)
    ma = Managed(ha)
    smb.set_option(smb.OPT_ASYNC, 1)
    try:
        cur = lib.smb_alloc(n * 4, smb.MEM_MANAGED)
        smb.array_scalar_ptr(smb.OP_ADD, smb.F32, ma.ptr, 1.0, n, cur)
        want = orc.array_scalar("add", ha, 1.0)
        for k in range(12):
            nxt = lib.smb_alloc(n * 4, smb.MEM_MANAGED)
            smb.array_scalar_ptr(smb.OP_MUL, smb.F32, cur, 1.0009765625, n, nxt)
            lib.smb_free(cur)  # still being read by the kernel just enqueued
            cur = nxt
            want = orc.array_scalar("mul", want, 1.0009765625)
        smb._check(lib.smb_wait_pending())
        got = np.ctypeslib.as_array(ctypes.cast(cur, ctypes.POINTER(ctypes.c_float)), shape=(n,)).copy()
    finally:
        smb.set_option(smb.OPT_ASYNC, 0)
    lib.smb_free(cur)
    assert_same_bits(got, want, "twelve dependent operators on recycled blocks")


def test_staged_call_is_ordered_after_the_callers_stream(orc):
    """Host (pinned) operands with stream != NULL: the H2D copies start after the work already enqueued
    on that stream (here: the async memcpy that fills the pinned input)."""
    import torch
    n = 1 << 22
    rng = np.random.default_rng(92)
    src = torch.from_numpy(rng.standard_normal(n).astype(np.float32)).cuda()
    pin_in = torch.zeros(n, dtype=torch.float32).pin_memory()
    pin_out = torch.zeros(n, dtype=torch.float32).pin_memory()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for _ in range(8):                       # keep the stream busy so the copy below is still pending
            src.mul_(1.0)
        pin_in.copy_(src, non_blocking=True)     # produces the pinned input on stream s
    smb.array_scalar_ptr(smb.OP_MUL, smb.F32, pin_in.data_ptr(), 2.0, n, pin_out.data_ptr(), s.cuda_stream)
    assert_same_bits(pin_out.numpy(), (src.cpu().numpy() * np.float32(2.0)), "staged call after async producer")


@pytest.mark.parametrize("dtype", [np.float32, np.int32])
def test_operands_of_mixed_memory_kinds(orc, dtype):
    """One call may mix host, device and managed operands (element_wise_op takes raw pointers): host inputs are
    staged slab by slab, a device / managed result is written in place (no copy back), a host result is copied
    back -- whole results and flat sub-ranges, several slabs per call."""
    import torch
    tdt = {np.float32: torch.float32, np.int32: torch.int32}[dtype]
    rng = np.random.default_rng(97)
    rows, cols = 96, 1024
    a = (rng.standard_normal((rows, cols)) * 50).astype(dtype)
    b = (rng.standard_normal((1, cols)) * 50).astype(dtype)           # invariant along the slabs: uploaded once
    c = (rng.standard_normal((rows, cols)) * 50).astype(dtype)
    dt = smb.dtype_code(np.dtype(dtype))
    shape = [rows, cols]
    smb.set_option(smb.OPT_STAGE_CHUNK_BYTES, 1 << 16)                       # 16 rows per slab: 6 slabs over 3 slots
    try:
        for name, y, sy in (("row", b, [0, 1]), ("dense", c, [cols, 1])):
            want = orc.binary("sub", a, y)
            dy = torch.from_numpy(y).cuda()
            da = torch.from_numpy(a).cuda()
            my = Managed(y)
            # host a, host y -> DEVICE result
            out = torch.zeros(rows * cols, dtype=tdt, device="cuda")
            torch.cuda.synchronize()
            smb.elementwise_ptr(smb.OP_SUB, dt, a.ctypes.data, [cols, 1], y.ctypes.data, sy, shape, out.data_ptr())
            assert_same_bits(out.cpu().numpy().reshape(rows, cols), want, f"host,host({name}) -> device")
            # host a, DEVICE y -> host result
            got = np.zeros((rows, cols), dtype)
            smb.elementwise_ptr(smb.OP_SUB, dt, a.ctypes.data, [cols, 1], dy.data_ptr(), sy, shape, got.ctypes.data)
            assert_same_bits(got, want, f"host,device({name}) -> host")
            # DEVICE a, MANAGED y -> host result
            got = np.zeros((rows, cols), dtype)
            smb.elementwise_ptr(smb.OP_SUB, dt, da.data_ptr(), [cols, 1], my.ptr, sy, shape, got.ctypes.data)
            assert_same_bits(got, want, f"device,managed({name}) -> host")
            # host a, managed y -> MANAGED result
            mo = Managed(shape=(rows, cols), dtype=dtype)
            smb.elementwise_ptr(smb.OP_SUB, dt, a.ctypes.data, [cols, 1], my.ptr, sy, shape, mo.ptr)
            smb.sync()
            assert_same_bits(mo.np.copy(), want, f"host,managed({name}) -> managed")
            # a flat sub-range with host inputs and a device result, and with a host result
            lo, cnt = 5 * cols + 17, 40 * cols + 3
            part = torch.zeros(cnt, dtype=tdt, device="cuda")
            torch.cuda.synchronize()
            smb.elementwise_range_ptr(smb.OP_SUB, dt, a.ctypes.data, [cols, 1], y.ctypes.data, sy, shape, lo, cnt, part.data_ptr())
            assert_same_bits(part.cpu().numpy(), want.ravel()[lo:lo + cnt], f"range host,host({name}) -> device")
            hpart = np.zeros(cnt, dtype)
            smb.elementwise_range_ptr(smb.OP_SUB, dt, da.data_ptr(), [cols, 1], y.ctypes.data, sy, shape, lo, cnt, hpart.ctypes.data)
            assert_same_bits(hpart, want.ravel()[lo:lo + cnt], f"range device,host({name}) -> host")
            my.free(); mo.free()
        # array (op) scalar: host in -> device out, device in -> host out
        flat = a.ravel()
        want = orc.array_scalar("mul", flat, 3)
        out = torch.zeros(flat.size, dtype=tdt, device="cuda")
        torch.cuda.synchronize()
        smb.array_scalar_ptr(smb.OP_MUL, dt, flat.ctypes.data, 3, flat.size, out.data_ptr())
        assert_same_bits(out.cpu().numpy(), want, "scalar host -> device")
        got = np.zeros(flat.size, dtype)
        smb.array_scalar_ptr(smb.OP_MUL, dt, torch.from_numpy(flat).cuda().data_ptr(), 3, flat.size, got.ctypes.data)
        assert_same_bits(got, want, "scalar device -> host")
    finally:
        smb.set_option(smb.OPT_STAGE_CHUNK_BYTES, 64 << 20)


# -------------------------------------------------------------- exhaustive device-side audit ----
def test_pow_audit_agrees_with_the_oracle_and_catches_errors(orc):
    import torch
    rng = np.random.default_rng(93)
    n = 1 << 20
    hx = np.concatenate([rng.uniform(0.01, 100, n // 2).astype(np.float32),
                         rng.integers(1, 0x7f800000, n // 2, dtype=np.uint32).view(np.float32)])
    x = torch.from_numpy(hx).cuda()
    out = torch.empty_like(x)
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for y in (2.5, -0.75, 17.0, 300.0):
            smb.array_scalar_ptr(smb.OP_POW, smb.F32, x.data_ptr(), y, n, out.data_ptr())
            cnt, worst = smb.pow_audit_f32_ptr(x.data_ptr(), y, out.data_ptr(), n, 0.6)
            err = oracle.ulp_error_f32(out.cpu().numpy(), orc.pow_ref_f32(hx, y))
            assert cnt == 0 and abs(worst - err.max()) < 0.02, (y, cnt, worst, err.max())
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)
    # a planted 2-ulp error and a wrong special are both seen
    smb.array_scalar_ptr(smb.OP_POW, smb.F32, x.data_ptr(), 2.5, n, out.data_ptr())
    h = out.cpu().numpy()
    h[12345] = np.nextafter(np.nextafter(h[12345], np.float32(np.inf)), np.float32(np.inf))
    out.copy_(torch.from_numpy(h))
    cnt, worst = smb.pow_audit_f32_ptr(x.data_ptr(), 2.5, out.data_ptr(), n, 0.6)
    assert cnt == 1 and 1.4 < worst < 2.6, (cnt, worst)


# ------------------------------------------ sm::pow(a (op) b, y): the pow kernel with a fused pre-operator ----
def test_fused_pow_of_a_binary_operator_is_bit_identical_to_the_two_operators(orc):
    """smb_chain [a, (op) b, pow y] on dense same-shape f32 arrays runs the pow kernel itself with the operator applied to
    the loaded operands: the same bits as the operator followed by sm::pow (same DevOp rounding, same pow variant), every
    tier / sign variant, ragged sizes, both operand orders of - and /."""
    rng = np.random.default_rng(97)
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for n in (100_003, 1 << 20, 8, 3):
            a = rng.uniform(0.05, 9.0, n).astype(np.float32)
            b = rng.uniform(0.05, 9.0, n).astype(np.float32)
            sgn = np.where(rng.random(n) < 0.3, -1, 1).astype(np.float32)
            for y in (2.5, 0.5, 17.0, 300.5, 3.0, 2.0, -1.5):
                for op in ("add", "sub", "mul", "div", "rsub", "rdiv"):
                    aa = a * sgn if float(y).is_integer() else a
                    bb = b
                    if not float(y).is_integer() and op in ("sub", "rsub"):
                        aa, bb = (a + 9.5, b) if op == "sub" else (a, b + 9.5)   # keep the base positive
                    base_op = op[1:] if op.startswith("r") else op
                    mid = smb.binary(base_op, bb, aa) if op.startswith("r") else smb.binary(base_op, aa, bb)
                    want = smb.pow(mid, y)
                    got = smb.chain(aa, (op, bb), ("pow", y))
                    assert smb.last_kernel() == "k_stream<pow,fused-pre>", (n, y, op, smb.last_kernel())
                    assert_same_bits(got, want, f"pow({op}(a, b), {y}) n={n}")
            # and within the stated accuracy of std::pow in double on the exactly rounded intermediate
            mid = orc.binary("add", a, b)
            err = oracle.ulp_error_f32(smb.chain(a, ("add", b), ("pow", 2.5)), orc.pow_ref_f32(mid, 2.5))
            assert err.max() <= 0.6, err.max()
        # what does not fit (a broadcast leaf, a longer chain) stays on the chain kernel
        m = rng.uniform(0.1, 5, (64, 256)).astype(np.float32)
        row = rng.uniform(0.1, 5, (1, 256)).astype(np.float32)
        got = smb.chain(m, ("add", row), ("pow", 2.5))
        assert smb.last_kernel().startswith("k_chain")
        assert oracle.ulp_error_f32(got, orc.pow_ref_f32(orc.binary("add", m, row), 2.5)).max() <= 0.6
        got = smb.chain(m, ("mul", 2.0), ("add", 1.0), ("pow", 2.5))
        assert smb.last_kernel().startswith("k_chain")
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)


def test_fused_pow_of_an_array_and_a_constant_is_bit_identical_to_the_two_operators(orc):
    """smb_chain [a, (op) constant, pow y] on a dense f32 array: the pow kernel with a one-operand pre-operator -- the same
    bits as the scalar operator followed by sm::pow, every tier / sign variant, ragged sizes, both operand orders of -
    (the two divisions stay on the chain kernel, equally bit-identical)."""
    rng = np.random.default_rng(98)
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for n, off in ((100_003, 0), (1 << 20, 0), (4099, 1), (8, 0), (3, 0)):
            a = rng.uniform(0.05, 9.0, n + off).astype(np.float32)[off:]
            sgn = np.where(rng.random(n) < 0.3, -1, 1).astype(np.float32)
            for y in (2.5, 0.5, 17.0, 300.5, 3.0, 2.0, -1.5):
                for op, cst in (("add", 1.5), ("sub", -0.25), ("mul", 1.75), ("div", 3.0), ("rsub", 20.0), ("rdiv", 2.0)):
                    aa = (a * sgn).astype(np.float32) if float(y).is_integer() else a
                    if op.startswith("r"):
                        mid = smb.binary(op[1:], np.full(n, cst, np.float32), aa)
                    else:
                        mid = smb.scalar(op, aa, cst)
                    want = smb.pow(mid, y)
                    got = smb.chain(aa, (op, cst), ("pow", y))
                    if "div" in op:   # stays on the chain kernel (its scalar form runs the reference-accuracy pow): ULP-bounded, not bit-identical
                        if n > 8:
                            assert smb.last_kernel().startswith("k_chain"), (n, y, op, smb.last_kernel())
                        if abs(y) < 8:
                            ref = orc.pow_ref_f32(mid, y)
                            fin = np.isfinite(ref) & (np.abs(ref) > 1e-30) & (np.abs(ref) < 1e30)
                            assert oracle.ulp_error_f32(got[fin], ref[fin]).max() <= 0.6, (op, y, n)
                        continue
                    if n > 8:
                        assert smb.last_kernel() == "k_stream<pow,fused-pre1>", (n, y, op, smb.last_kernel())
                    assert_same_bits(got, want, f"pow({op}(a, {cst}), {y}) n={n} off={off}")
        # and against the oracle's accuracy contract
        a = rng.uniform(0.05, 9.0, 1 << 16).astype(np.float32)
        got = smb.chain(a, ("mul", 1.75), ("pow", 2.5))
        err = oracle.ulp_error_f32(got, orc.pow_ref_f32(orc.array_scalar("mul", a, 1.75), 2.5))
        assert err.max() <= 0.6, err.max()
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)


def test_fused_pow_in_double_is_bit_identical_to_the_two_operators(orc):
    """The two fused shapes for double -- sm::pow(a (op) b, y) and sm::pow(a (op) constant, y) -- run the f64 pow kernel with a
    pre-operator: the bits of the eager operator followed by sm::pow (small / large |y|, odd / even / non-integer y, ragged sizes)."""
    rng = np.random.default_rng(100)
    smb.set_option(smb.OPT_POW_SPECIALISE, 0)
    try:
        for n in (100_003, 1 << 19, 6, 3):
            a = rng.uniform(0.05, 9.0, n)
            b = rng.uniform(0.05, 9.0, n)
            sgn = np.where(rng.random(n) < 0.3, -1.0, 1.0)
            for y in (2.5, 0.5, 17.0, 300.5, 3.0, 2.0, -1.5):
                aa = a * sgn if float(y).is_integer() else a
                for op in ("add", "sub", "mul", "div", "rsub", "rdiv"):
                    x, z = aa, b
                    if not float(y).is_integer() and op in ("sub", "rsub"):
                        x, z = (a + 9.5, b) if op == "sub" else (a, b + 9.5)   # keep the base positive
                    base_op = op[1:] if op.startswith("r") else op
                    mid = smb.binary(base_op, z, x) if op.startswith("r") else smb.binary(base_op, x, z)
                    got = smb.chain(x, (op, z), ("pow", y))
                    if n > 8:
                        assert smb.last_kernel() == "k_stream<pow,fused-pre>", (n, y, op, smb.last_kernel())
                    assert_same_bits(got, smb.pow(mid, y), f"f64 pow({op}(a, b), {y}) n={n}")
                for op, cst in (("add", 1.5), ("sub", -0.25), ("mul", 1.75), ("rsub", 20.0)):
                    mid = smb.binary("sub", np.full(n, cst), aa) if op == "rsub" else smb.scalar(op, aa, cst)
                    got = smb.chain(aa, (op, cst), ("pow", y))
                    if n > 8:
                        assert smb.last_kernel() == "k_stream<pow,fused-pre1>", (n, y, op, smb.last_kernel())
                    assert_same_bits(got, smb.pow(mid, y), f"f64 pow({op}(a, {cst}), {y}) n={n}")
        a = rng.uniform(0.05, 9.0, 1 << 16)
        b = rng.uniform(0.05, 9.0, 1 << 16)
        hi, lo = orc.pow_ref_f64(orc.binary("add", a, b), 2.5)
        assert oracle.ulp_error_f64(smb.chain(a, ("add", b), ("pow", 2.5)), hi, lo).max() <= 0.65
    finally:
        smb.set_option(smb.OPT_POW_SPECIALISE, 1)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_specialised_exponents_inside_chains_match_the_eager_operator_bit_for_bit(orc, dtype):
    """sm::pow by 2, 0.5, -1, 1 has an exact one-operation form (SMB_OPT_POW_SPECIALISE, the default); a pow step of a chain
    takes the same form, so lazy and eager agree bit for bit there -- specials and negative bases included."""
    rng = np.random.default_rng(99)
    n = 100_003
    a = np.concatenate([rng.uniform(-9, 9, n - 8), [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-42, -1e-42, 3e38]]).astype(dtype)
    b = rng.uniform(0.5, 2.0, n).astype(dtype)
    for y in (2.0, 0.5, -1.0, 1.0):
        mid = smb.binary("mul", a, b)
        assert_same_bits(smb.chain(a, ("mul", b), ("pow", y)), smb.pow(mid, y), f"pow(a*b, {y})")
        assert smb.last_kernel().startswith("k_")
        mid = smb.scalar("add", a, 0.25)
        assert_same_bits(smb.chain(a, ("add", 0.25), ("pow", y)), smb.pow(mid, y), f"pow(a+c, {y})")
        assert_same_bits(smb.chain(a, ("pow", y), ("sub", b)), smb.binary("sub", smb.pow(a, y), b), f"pow(a, {y}) - b")
        m2 = a.reshape(-1)[: 96 * 1024].reshape(96, 1024)
        row = b[:1024].reshape(1, 1024)
        assert_same_bits(smb.chain(m2, ("add", row), ("pow", y), ("mul", row)),
                         smb.binary("mul", smb.pow(smb.binary("add", m2, row), y).reshape(96, 1024), row), f"(pow(m+row, {y}))*row")


def test_device_set_in_async_mode_keeps_order_across_devices(orc, sharded):
    """Async hand-off on a device set: dependent operators whose partitions differ (a small result feeding a large one as a
    broadcast operand, a result reused as an operand with another shape), recycled blocks, and the steady state where the
    same partition repeats and the cross-device waits are skipped."""
    rng = np.random.default_rng(101)
    lib = smb.lib()
    for devs in _device_sets():
        smb.set_devices(devs)
        R, C = 1024, 2048                                   # 8 MiB per array
        a = rng.standard_normal((R, C)).astype(np.float32)
        b = rng.standard_normal((R, C)).astype(np.float32)
        row = rng.standard_normal((1, C)).astype(np.float32)
        ma, mb, mrow = Managed(a), Managed(b), Managed(row)
        mrow2, mc, md, me = Managed(shape=(1, C), dtype=np.float32), Managed(shape=(R, C), dtype=np.float32), Managed(shape=(R, C), dtype=np.float32), Managed(shape=(R, C), dtype=np.float32)
        full, rowst = [C, 1], [0, 1]
        smb.set_option(smb.OPT_ASYNC, 1)
        try:
            for it in range(4):
                smb.array_scalar_ptr(smb.OP_MUL, smb.F32, mrow.ptr, 1.0 + it, C, mrow2.ptr)                        # small: one device
                smb.elementwise_ptr(smb.OP_ADD, smb.F32, ma.ptr, full, mb.ptr, full, [R, C], mc.ptr)                # large: every device
                smb.elementwise_ptr(smb.OP_MUL, smb.F32, mc.ptr, full, mrow2.ptr, rowst, [R, C], md.ptr)            # reads the small result on every device
                smb.elementwise_ptr(smb.OP_SUB, smb.F32, md.ptr, full, mc.ptr, full, [R, C], me.ptr)                # same partition as before: no waits
                smb.elementwise_ptr(smb.OP_ADD, smb.F32, me.ptr, full, mrow.ptr, rowst, [R, C], mc.ptr)             # overwrites c, which the previous two read
                tmp = lib.smb_alloc(R * C * 4, smb.MEM_MANAGED)                                                     # a temporary freed while in flight
                smb.elementwise_ptr(smb.OP_MUL, smb.F32, mc.ptr, full, mc.ptr, full, [R, C], tmp)
                smb.elementwise_ptr(smb.OP_ADD, smb.F32, tmp, full, mb.ptr, full, [R, C], md.ptr)
                lib.smb_free(tmp)
            smb._check(lib.smb_wait_pending())
        finally:
            smb.set_option(smb.OPT_ASYNC, 0)
        row2 = orc.array_scalar("mul", row, 4.0)
        c1 = orc.binary("add", a, b)
        d1 = orc.binary("mul", c1, row2)
        e1 = orc.binary("sub", d1, c1)
        c2 = orc.binary("add", e1, row)
        d2 = orc.binary("add", orc.binary("mul", c2, c2), b)
        assert_same_bits(me.np.copy(), e1, f"e on {devs}")
        assert_same_bits(mc.np.copy(), c2, f"c on {devs}")
        assert_same_bits(md.np.copy(), d2, f"d on {devs}")


def test_synchronous_calls_land_pending_async_work_of_other_devices_first(orc):
    """In async mode an operand may still be in flight on ANOTHER device's stream when a synchronous call needs it:
    a small array computed on one device feeding a dot product that is spread over the set (2n bytes count there), and a
    host-operand call (always synchronous) reading a result the whole set is still producing."""
    rng = np.random.default_rng(103)
    lib = smb.lib()
    n = 1 << 20
    a = rng.integers(-2**31, 2**31, size=n, dtype=np.int64).astype(np.int32)
    b = rng.integers(-2**31, 2**31, size=n, dtype=np.int64).astype(np.int32)
    h = rng.integers(-1000, 1000, size=n).astype(np.int32)
    old = lib.smb_get_option(smb.OPT_SHARD_MIN_BYTES)
    try:
        for devs in _device_sets():
            smb.set_devices(devs)
            ma, mb = Managed(a), Managed(b)
            mc, md = Managed(shape=(n,), dtype=np.int32), Managed(shape=(n,), dtype=np.int32)
            smb.set_option(smb.OPT_ASYNC, 1)
            try:
                for it in range(3):
                    # 4 MiB results stay on one device, the 8 MiB dot product is spread over the set
                    smb.set_option(smb.OPT_SHARD_MIN_BYTES, 6 << 20)
                    smb.contiguous_ptr(smb.OP_MUL, smb.I32, ma.ptr, mb.ptr, mc.ptr, n)
                    for _ in range(6):
                        smb.array_scalar_ptr(smb.OP_ADD, smb.I32, mc.ptr, 1 + it, n, mc.ptr)
                    got = smb.dot_ptr(smb.I32, mc.ptr, mb.ptr, n)
                    c = (a * b + np.int32(6 * (1 + it))).astype(np.int32)
                    want = int(np.sum(c.astype(np.int64) * b.astype(np.int64)) & 0xffffffff)
                    assert (got & 0xffffffff) == want, (devs, it)
                    # every device produces d; a host-operand call reads it right away
                    smb.set_option(smb.OPT_SHARD_MIN_BYTES, 0)
                    smb.contiguous_ptr(smb.OP_SUB, smb.I32, mc.ptr, ma.ptr, md.ptr, n)
                    out = np.zeros(n, np.int32)
                    smb.contiguous_ptr(smb.OP_ADD, smb.I32, h.ctypes.data, md.ptr, out.ctypes.data, n)
                    assert_same_bits(out, (h + (c - a)).astype(np.int32), f"host + pending sharded result on {devs}")
                    hs = np.zeros(n, np.int32)
                    smb.contiguous_ptr(smb.OP_MUL, smb.I32, md.ptr, md.ptr, mc.ptr, n)      # pending again
                    smb.array_scalar_ptr(smb.OP_SUB, smb.I32, mc.ptr, 7, n, hs.ctypes.data)  # managed in, host out
                    d = (c - a).astype(np.int32)
                    assert_same_bits(hs, (d * d - np.int32(7)).astype(np.int32), f"scalar to host on {devs}")
            finally:
                smb.set_option(smb.OPT_ASYNC, 0)
            for m in (ma, mb, mc, md):
                m.free()
    finally:
        smb.set_devices([])
        smb.set_option(smb.OPT_SHARD_MIN_BYTES, old)


def test_async_launches_queued_behind_a_long_kernel_keep_their_order(orc):
    """Python enqueues more slowly than the GPU drains 4 us kernels, so dependent launches rarely overlap in the other tests.
    Here every round starts with a long kernel: the small operators queue up behind it and become eligible back to back --
    the situation in which a launch admitted behind a WAITING launch once started before that wait was over and read what an
    earlier grid was still writing (tools/pdl_stress.py; profiles/r2_pdl_stress.jsonl: 1175 of 1800 rounds wrong before the
    fix, 0 after).  One device (producer, then two consumers of its result) and one device listed twice (two ranges)."""
    lib = smb.lib()
    rng = np.random.default_rng(104)
    nbig, n = 1 << 27, 1 << 20
    big_a, big_o = lib.smb_alloc(nbig * 4, smb.MEM_MANAGED), lib.smb_alloc(nbig * 4, smb.MEM_MANAGED)
    old = lib.smb_get_option(smb.OPT_SHARD_MIN_BYTES)
    try:
        for devs in ([], [0, 0]):
            smb.set_option(smb.OPT_SHARD_MIN_BYTES, 0 if devs else old)
            smb.set_devices(devs)
            a = rng.standard_normal(n).astype(np.float32)
            b = rng.standard_normal(n).astype(np.float32)
            ma, mb = Managed(a), Managed(b)
            mc, md, me = (Managed(shape=(n,), dtype=np.float32) for _ in range(3))
            smb.contiguous_ptr(smb.OP_ADD, smb.F32, big_a, big_a, big_o, nbig)
            smb.sync()
            smb.set_option(smb.OPT_ASYNC, 1)
            try:
                wrong = 0
                for r in range(150):
                    k = np.float32(1 + r % 7)
                    smb.contiguous_ptr(smb.OP_ADD, smb.F32, big_a, big_a, big_o, nbig)           # the queue fills behind this one
                    smb.array_scalar_ptr(smb.OP_MUL, smb.F32, ma.ptr, float(k), n, mc.ptr)          # c = a * k      (producer)
                    smb.array_scalar_ptr(smb.OP_ADD, smb.F32, mc.ptr, 2.0, n, md.ptr)               # d = c + 2      (conflicts: waits)
                    smb.contiguous_ptr(smb.OP_ADD, smb.F32, mc.ptr, mb.ptr, me.ptr, n)              # e = c + b      (no conflict with d's launch)
                    smb.sync()
                    c = a * k
                    wrong += int(not (np.array_equal(md.np, c + np.float32(2.0)) and np.array_equal(me.np, c + b)))
                assert wrong == 0, (devs, wrong)
            finally:
                smb.set_option(smb.OPT_ASYNC, 0)
            for m in (ma, mb, mc, md, me):
                m.free()
    finally:
        smb.set_devices([])
        smb.set_option(smb.OPT_SHARD_MIN_BYTES, old)
        lib.smb_free(big_a)
        lib.smb_free(big_o)


def test_random_async_programs_match_sequential_evaluation(orc):
    """Random programs of ~40 dependent operators over a handful of managed arrays -- binary / scalar / in-place / row-broadcast
    / fused-chain operators, temporaries freed while in flight and their blocks handed out again -- enqueued in async mode
    behind a long kernel (so that they really are in flight together), on one device and on device sets; every array is
    compared with a sequential numpy evaluation (single float32 operations: the same bits)."""
    lib = smb.lib()
    rng = np.random.default_rng(105)
    nbig = 1 << 28
    big_a, big_o = lib.smb_alloc(nbig * 4, smb.MEM_MANAGED), lib.smb_alloc(nbig * 4, smb.MEM_MANAGED)
    old = lib.smb_get_option(smb.OPT_SHARD_MIN_BYTES)
    R, C = 256, 2048
    n = R * C
    f32 = np.float32
    np_err = np.seterr(all="ignore")     # some programs overflow: inf / NaN are compared like everything else
    try:
        sets = [[], [0, 0]] + ([list(range(smb.device_count()))] if smb.device_count() >= 2 else [])
        for devs in sets:
            smb.set_option(smb.OPT_SHARD_MIN_BYTES, 0 if devs else old)
            smb.set_devices(devs)
            smb.contiguous_ptr(smb.OP_ADD, smb.F32, big_a, big_a, big_o, nbig)
            smb.sync()
            for prog in range(12):
                host = [rng.uniform(0.5, 1.5, n).astype(f32) for _ in range(5)]
                row = rng.uniform(0.5, 1.5, C).astype(f32)
                arrs = [Managed(h) for h in host]
                mrow = Managed(row)
                smb.set_option(smb.OPT_ASYNC, 1)
                try:
                    smb.contiguous_ptr(smb.OP_ADD, smb.F32, big_a, big_a, big_o, nbig)       # ~0.5 ms: everything below queues up
                    for step in range(40):
                        kind = int(rng.integers(0, 6))
                        i, j, k = (int(x) for x in rng.integers(0, 5, 3))
                        op = ["add", "sub", "mul"][int(rng.integers(0, 3))]
                        npop = {"add": np.add, "sub": np.subtract, "mul": np.multiply}[op]
                        if kind == 0:      # k = i (op) j, possibly in place
                            smb.contiguous_ptr(smb.OPS[op], smb.F32, arrs[i].ptr, arrs[j].ptr, arrs[k].ptr, n)
                            host[k] = npop(host[i], host[j])
                        elif kind == 1:    # k = i (op) constant
                            cst = float(f32(rng.uniform(0.75, 1.25)))
                            smb.array_scalar_ptr(smb.OPS[op], smb.F32, arrs[i].ptr, cst, n, arrs[k].ptr)
                            host[k] = npop(host[i], f32(cst))
                        elif kind == 2:    # through a temporary that is freed while in flight
                            tmp = lib.smb_alloc(n * 4, smb.MEM_MANAGED)
                            smb.contiguous_ptr(smb.OPS[op], smb.F32, arrs[i].ptr, arrs[j].ptr, tmp, n)
                            smb.contiguous_ptr(smb.OP_MUL, smb.F32, tmp, arrs[i].ptr, arrs[k].ptr, n)
                            lib.smb_free(tmp)
                            host[k] = npop(host[i], host[j]) * host[i]
                        elif kind == 3:    # row broadcast (k_row: a plain launch between the stream kernels)
                            smb.elementwise_ptr(smb.OPS[op], smb.F32, arrs[i].ptr, [C, 1], mrow.ptr, [0, 1], [R, C], arrs[k].ptr)
                            host[k] = npop(host[i].reshape(R, C), row.reshape(1, C)).reshape(-1)
                        elif kind == 4 and k != i and k != j:    # fused chain (i + j) * i -> k
                            leaves = [(None, False, (arrs[i].ptr, [1])), ("add", False, (arrs[j].ptr, [1])), ("mul", False, (arrs[i].ptr, [1]))]
                            smb.chain_ptr(smb.F32, leaves, [n], arrs[k].ptr)
                            host[k] = (host[i] + host[j]) * host[i]
                        else:              # keep the values in range
                            smb.array_scalar_ptr(smb.OP_MUL, smb.F32, arrs[k].ptr, 0.5, n, arrs[k].ptr)
                            host[k] = host[k] * f32(0.5)
                    smb._check(lib.smb_wait_pending())
                finally:
                    smb.set_option(smb.OPT_ASYNC, 0)
                for idx in range(5):
                    assert_same_bits(arrs[idx].np.copy(), host[idx], f"program {prog} on {devs}: array {idx}")
                for m in arrs + [mrow]:
                    m.free()
    finally:
        np.seterr(**np_err)
        smb.set_devices([])
        smb.set_option(smb.OPT_SHARD_MIN_BYTES, old)
        lib.smb_free(big_a)
        lib.smb_free(big_o)
