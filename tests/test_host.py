"""Host-side logic that needs no GPU: the C-ABI library loads and exports every
symbol include/smb200.h declares, the planner (dimension coalescing / kernel
choice), the Python mirror of sm::broadcast, the shard splitter, and the
no-CPU-fallback guarantee."""
import ctypes
import subprocess
import sys
import os
import re

import numpy as np
import pytest

import simplemath_b200 as smb
from conftest import ROOT


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "smb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(smb_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    assert declared == set(smb.SYMBOLS), declared ^ set(smb.SYMBOLS)
    lib = smb.lib()
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.smb_version()


def test_no_cpu_fallback_without_device():
    """On a box without a CUDA device every compute entry point must fail loudly."""
    if smb.device_count() > 0:
        pytest.skip("a CUDA device is present")
    a = np.ones(16, np.float32)
    with pytest.raises(smb.SmbError, match="no CUDA device"):
        smb.binary("add", a, a)
    with pytest.raises(smb.SmbError, match="no CPU fallback"):
        smb.pow(a, 2.0)
    assert smb.lib().smb_alloc(64, smb.MEM_DEVICE) is None


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "simplemath_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".inl", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "liboracle" not in txt and "libsmref" not in txt, f
    for dirpath, _, files in os.walk(os.path.join(ROOT, "include")):
        for f in files:
            txt = open(os.path.join(dirpath, f)).read()
            assert "liboracle" not in txt and "oracle/" not in txt.replace("oracle/oracle.c:orc_fill_uniform_f32", ""), f


def test_retired_option_keys_are_rejected():
    """Keys 2, 3 and 10..13 selected kernel variants and launch modes that measured slower and were removed:
    setting one fails like any unknown key, reading one returns -1, and the keys that remain keep their numbers."""
    lib = smb.lib()
    for key in (2, 3, 10, 11, 12, 13):
        assert lib.smb_set_option(key, 1) == 1  # SMB_ERR_INVALID
        assert b"unknown option" in lib.smb_last_error()
        with pytest.raises(smb.SmbError, match="unknown option"):
            smb.set_option(key, 0)
        assert lib.smb_get_option(key) == -1
    assert (smb.OPT_POW_SPECIALISE, smb.OPT_STAGE_CHUNK_BYTES, smb.OPT_FORCE_WIDE_INDEX, smb.OPT_ASYNC, smb.OPT_PDL,
            smb.OPT_SHARD_MIN_BYTES, smb.OPT_REPLICATE_MAX_BYTES, smb.OPT_POOL_MAX_CACHED_BYTES) == (0, 1, 4, 5, 6, 7, 8, 9)
    assert lib.smb_get_option(smb.OPT_POW_SPECIALISE) == 1


# ---- broadcast mirror ----------------------------------------------------------
CASES = [((4096, 4096), (1, 4096)), ((512, 1, 1024), (1, 512, 1024)), ((224, 224, 3), (1, 224, 1, 3)),
         ((5,), (1,)), ((3, 1, 4, 1, 5), (2, 1, 6, 1)), ((1, 1), (1, 1)), ((7,), (3, 7)), ((2, 3, 4, 5, 6, 7), (7,))]


@pytest.mark.parametrize("s1,s2", CASES)
def test_broadcast_mirror_matches_oracle(orc, ref, s1, s2):
    st1, st2 = smb.row_major_strides(s1), smb.row_major_strides(s2)
    got = smb.broadcast(s1, st1, s2, st2)
    want = orc.broadcast(s1, st1, s2, st2)
    assert tuple(got) == tuple(want)
    if ref is not None:
        assert tuple(got) == tuple(ref.broadcast(s1, st1, s2, st2))


def test_broadcast_mirror_config_tables():
    # SURVEY.md §8(a) a4: the stride tables of BASELINE configs C2 and C4
    shape, sa, sb, n = smb.broadcast((4096, 4096), (4096, 1), (1, 4096), (4096, 1))
    assert (shape, sa, sb, n) == ([4096, 4096], [4096, 1], [0, 1], 16777216)
    shape, sa, sb, n = smb.broadcast((512, 1, 1024), (1024, 1024, 1), (1, 512, 1024), (524288, 1024, 1))
    assert (shape, sa, sb, n) == ([512, 512, 1024], [1024, 0, 1], [0, 1024, 1], 268435456)


def test_broadcast_mirror_rejects():
    with pytest.raises(smb.SmbError, match="Cannot broadcast shapes: incompatible dimensions"):
        smb.broadcast((2, 3), (3, 1), (4, 3), (3, 1))


# ---- planner ---------------------------------------------------------------------
def test_plan_contiguous_collapses_to_1d():
    kind, shape, sa, sb = smb.plan([12, 4, 1], [12, 4, 1], [5, 3, 4])
    assert kind == smb.PLAN_CONTIGUOUS and shape == [60] and sa == [1] and sb == [1]


def test_plan_c2_row_broadcast():
    kind, shape, sa, sb = smb.plan([4096, 1], [0, 1], [4096, 4096])
    assert kind == smb.PLAN_ROW and shape == [4096, 4096] and sa == [4096, 1] and sb == [0, 1]


def test_plan_c4_three_dims():
    kind, shape, sa, sb = smb.plan([1024, 0, 1], [0, 1024, 1], [512, 512, 1024])
    assert kind == smb.PLAN_ROW and shape == [512, 512, 1024]


def test_plan_reference_view_case_drops_unit_dim_and_merges():
    # view {224,224,3} strides {672,3,1} padded to 4-D vs {1,224,1,3}: tests/add.cpp:59-92
    shape, sa, sb, _ = smb.broadcast((224, 224, 3), (672, 3, 1), (1, 224, 1, 3), (672, 3, 3, 1))
    assert shape == [1, 224, 224, 3] and sa == [0, 672, 3, 1] and sb == [672, 3, 0, 1]
    kind, pshape, psa, psb = smb.plan(sa, sb, shape)
    assert kind == smb.PLAN_ROW and pshape == [224, 224, 3] and psa == [672, 3, 1] and psb == [3, 0, 1]


def test_plan_transposed_operand_is_generic():
    kind, shape, sa, sb = smb.plan([1, 4], [6, 1], [4, 6])
    assert kind == smb.PLAN_GENERIC and shape == [4, 6]


def test_plan_inner_broadcast_is_row_kind():
    kind, shape, sa, sb = smb.plan([1, 0], [0, 1], [16, 24])  # {16,1} (op) {1,24}
    assert kind == smb.PLAN_ROW and sa == [1, 0] and sb == [0, 1]


def test_plan_offsets_equal_reference_formula(orc):
    """Coalescing must not change any operand offset: compare the offset of every
    flat index under the original and the coalesced tables (calculate.h:54-63)."""
    rng = np.random.default_rng(3)

    def offsets(shape, strides):
        idx = np.indices(shape).reshape(len(shape), -1)
        return (idx * np.array(strides, dtype=np.int64)[:, None]).sum(0)

    for _ in range(200):
        nd = int(rng.integers(1, 7))
        shape = [int(x) for x in rng.integers(1, 5, size=nd)]
        s1 = [d if rng.random() < 0.7 else 1 for d in shape]
        s2 = [d if rng.random() < 0.7 else 1 for d in shape]
        st1 = smb.row_major_strides(s1)
        st2 = smb.row_major_strides(s2)
        if rng.random() < 0.3:  # a view with padded parent strides
            st1 = [s * 2 for s in st1]
        rs, n1, n2, tot = smb.broadcast(s1, st1, s2, st2)
        kind, ps, pa, pb = smb.plan(n1, n2, rs)
        assert int(np.prod(ps)) == tot
        assert np.array_equal(offsets(rs, n1), offsets(ps, pa))
        assert np.array_equal(offsets(rs, n2), offsets(ps, pb))


# ---- shard splitter ----------------------------------------------------------------
@pytest.mark.parametrize("n,world,align", [(2**30, 8, 1024), (1000, 3, 8), (7, 8, 4), (0, 2, 4), (16777216, 4, 4096), (12345, 5, 1)])
def test_shard_range_partitions(n, world, align):
    prev = 0
    for r in range(world):
        b, e = smb.shard_range(n, r, world, align)
        assert b == prev and b <= e <= n
        assert b % align == 0 or b == n
        prev = e
    assert prev == n
    sizes = [smb.shard_range(n, r, world, align) for r in range(world)]
    assert max(e - b for b, e in sizes) - min(e - b for b, e in sizes) <= 2 * align


def test_pow_tables_header_is_what_the_generator_writes(tmp_path):
    """simplemath_b200/csrc/smb_pow_tables.h is generated (tools/gen_pow_tables.py, mpmath at 200 bits): the
    committed header must be exactly what the committed generator produces -- tables, fitted coefficients,
    and the exactness / two-sum assertions the generator makes along the way."""
    pytest.importorskip("mpmath")
    out = tmp_path / "smb_pow_tables.h"
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_pow_tables.py"), str(out)], check=True, capture_output=True)
    committed = open(os.path.join(ROOT, "simplemath_b200", "csrc", "smb_pow_tables.h")).read()
    assert out.read_text() == committed


# ---- multi-GPU planner (smb_plan_shards: csrc/smb_shard.h, no GPU needed) ---------------------------
def _brute_touched(shape, stride, lo, hi):
    """min / max operand offset over flat result indices [lo, hi)."""
    idx = np.unravel_index(np.arange(lo, hi), shape)
    off = sum(i.astype(np.int64) * s for i, s in zip(idx, stride))
    return int(off.min()), int(off.max()) + 1


def test_shard_planner_bounds_and_operand_ranges_match_brute_force():
    rng = np.random.default_rng(123)
    shapes = [((40_000,), (40_000,)), ((300, 257), (1, 257)), ((300, 257), (300, 1)), ((129, 1), (1, 65)), ((24, 1, 256), (1, 40, 256)),
              ((5, 6, 7, 3), (1, 6, 1, 3)), ((64, 64), (64, 64)), ((7, 2048), (2048,)), ((2, 3, 4, 5, 6, 7), (2, 1, 4, 1, 6, 1)), ((5,), (1,))]
    for s1, s2 in shapes:
        shape, sa, sb, n = smb.broadcast(s1, smb.row_major_strides(s1), s2, smb.row_major_strides(s2))
        for ndev in (1, 2, 3, 8, 64):
            ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, ndev)
            assert bounds[0] == 0 and bounds[-1] == n and all(x <= y for x, y in zip(bounds, bounds[1:])), (s1, s2, ndev, bounds)
            for g in range(ndev):
                lo, hi = bounds[g], bounds[g + 1]
                if lo == hi:
                    assert ra[g][0] == ra[g][1] and rb[g][0] == rb[g][1]
                    continue
                assert ra[g] == _brute_touched(shape, sa, lo, hi), (s1, s2, ndev, g, "a")
                assert rb[g] == _brute_touched(shape, sb, lo, hi), (s1, s2, ndev, g, "b")
    # a transposed operand: offsets are not monotone in the flat index, the hull still is exact
    for r, c in ((37, 53), (200, 96), (8, 8)):
        shape, sa, sb = [r, c], [1, r], [c, 1]
        for ndev in (2, 5):
            ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, ndev)
            for g in range(ndev):
                if bounds[g] < bounds[g + 1]:
                    assert ra[g] == _brute_touched(shape, sa, bounds[g], bounds[g + 1])
    # random strided views (every stride table a result dim could see)
    for _ in range(60):
        nd = int(rng.integers(1, 5))
        shape = [int(v) for v in rng.integers(1, 9, nd)]
        sa = [int(v) for v in rng.integers(0, 40, nd)]
        sb = [int(v) for v in rng.integers(0, 3, nd)]
        ndev = int(rng.integers(1, 6))
        ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, ndev)
        for g in range(ndev):
            if bounds[g] < bounds[g + 1]:
                assert ra[g] == _brute_touched(shape, sa, bounds[g], bounds[g + 1]), (shape, sa, ndev, g)
                assert rb[g] == _brute_touched(shape, sb, bounds[g], bounds[g + 1]), (shape, sb, ndev, g)


def test_shard_planner_on_the_baseline_configs():
    """C5 / C2 x 16 / C4 at 8 devices: page-aligned or whole-row cuts, the streaming operand split in place,
    the broadcast operand replicated; a large transposed operand refuses (one device runs it)."""
    page = (2 << 20) // 4
    ok, bounds, ra, rb, modes = smb.plan_shards([1], [1], [1 << 30], 8)
    assert ok and modes == (0, 0) and all(b % page == 0 for b in bounds) and ra == rb == list(zip(bounds, bounds[1:]))
    shape, sa, sb, n = smb.broadcast((65536, 4096), (4096, 1), (1, 4096), (4096, 1))
    ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, 8)
    assert ok and modes == (0, 1) and all(b % page == 0 and b % 4096 == 0 for b in bounds) and all(r == (0, 4096) for r in rb)
    shape, sa, sb, n = smb.broadcast((512, 1, 1024), (1024, 1024, 1), (1, 512, 1024), (512 * 1024, 1024, 1))
    ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, 8)
    assert ok and modes == (1, 1) and all(b % (512 * 1024) == 0 for b in bounds)    # whole dim-0 slabs: k_outer applies
    assert ra == [(g * 65536, (g + 1) * 65536) for g in range(8)] and all(r == (0, 524288) for r in rb)
    ok, bounds, ra, rb, modes = smb.plan_shards([1, 8192], [8192, 1], [8192, 8192], 4)
    assert not ok and modes[0] == 2 and modes[1] == 0
    # uneven: 3 devices, 10 rows
    shape, sa, sb, n = smb.broadcast((10, 1000), (1000, 1), (1, 1000), (1000, 1))
    ok, bounds, ra, rb, modes = smb.plan_shards(sa, sb, shape, 3)
    assert bounds == [0, 4000, 7000, 10000]
