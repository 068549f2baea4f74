"""The batch form of the MSM's two-level counting sort (gnark_whir_b200/csrc/msm_sort.cuh, BATCH = true: k scalar
vectors over one bases vector) compiled for the host and run CTA by CTA against a direct counting sort of the
vector-major keys (tests/host_harness/sort_batch_host.cc).  Also restates the per-call limits of a batch MSM
(msm_batch_max in msm_impl.cuh) and checks them for every window width, with and without a window table, and every
power-of-two n up to 2^26."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import bn254 as bn
from tests.test_msm_digits_cpu import msm_num_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_harness", "sort_batch_host.cc")
OUT = os.path.join(ROOT, "tests", "host_harness", "_build", "sort_batch_host.so")

SORT_POINTS = 2048   # points per CTA of the coarse count
SORT_STAGE = 10240   # entries staged per CTA of the coarse partition
MAX_BUCKETS = 1 << 23
MAX_ENTRIES = (1 << 32) - 1


@pytest.fixture(scope="module")
def harness():
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-I",
                    os.path.join(ROOT, "gnark_whir_b200", "csrc"), "-o", OUT], check=True)
    return ctypes.CDLL(OUT)


rs = np.random.Generator(np.random.PCG64(20261021))


def rand_canon(n):
    return [int(x) % bn.R for x in (int.from_bytes(rs.bytes(32), "little") for _ in range(n))]


def run(harness, rows, c, table, ld=None, ent_stride=0, ent_off=0, seed=1):
    """rows: k lists of n canonical scalars; ld > n pads every row with random scalars the sort must not read."""
    k, n = len(rows), len(rows[0])
    ld = n if ld is None else ld
    flat = []
    for r in rows:
        assert len(r) == n
        flat += list(r) + rand_canon(ld - n)
    sc = np.ascontiguousarray(bn.fr_to_mont_array(flat))
    W = msm_num_windows(c)
    assert k <= batch_max(c, table, n), "shape beyond one batch call"
    stats = (ctypes.c_uint32 * 5)()
    rc = harness.sort_batch_host(sc.ctypes.data_as(ctypes.c_void_p), ctypes.c_uint32(n), ctypes.c_uint32(k),
                                 ctypes.c_uint32(ld), ctypes.c_int(c), ctypes.c_int(W), ctypes.c_int(table),
                                 ctypes.c_uint32(ent_stride), ctypes.c_uint32(ent_off), ctypes.c_uint64(seed), stats)
    assert rc == 0, f"batch sort differs from the direct counting sort (code {rc})"
    st = dict(zip(("F", "bins", "tiles", "entries", "largest"), list(stats)))
    assert st["F"] <= 12, "a batch must count its fine passes in shared memory"
    return st


@pytest.mark.parametrize("k", [1, 2, 3, 17])
@pytest.mark.parametrize("c,table", [(16, 1), (18, 1), (11, 0), (15, 0)])
def test_uniform(harness, k, c, table):
    n = 700
    run(harness, [rand_canon(n) for _ in range(k)], c, table)


@pytest.mark.parametrize("k", [2, 3, 17])
def test_row_stride(harness, k):
    n = 900
    run(harness, [rand_canon(n) for _ in range(k)], 16, 1, ld=n + 37)
    run(harness, [rand_canon(n) for _ in range(k)], 12, 0, ld=2 * n + 1)


@pytest.mark.parametrize("n", [1, 3, SORT_POINTS - 1, SORT_POINTS + 1, 1000])
def test_vectors_straddle_ctas(harness, n):
    # k * n off the coarse count's point tile and the partition's tile, vectors crossing CTA boundaries
    for c, table in ((20, 1), (13, 0)):
        k = 5
        run(harness, [rand_canon(n) for _ in range(k)], c, table)


@pytest.mark.parametrize("c,table", [(20, 1), (15, 0)])
def test_partition_tile_edges(harness, c, table):
    P = SORT_STAGE // msm_num_windows(c)
    for n, k in ((P - 1, 3), (P + 1, 2), (P // 3 + 1, 7)):
        run(harness, [rand_canon(n) for _ in range(k)], c, table)


def test_identical_vectors_land_in_distinct_sets(harness):
    row = rand_canon(1500)
    k = 4
    st = run(harness, [row] * k, 16, 1)
    single = run(harness, [row], 16, 1)
    assert st["entries"] == k * single["entries"]
    v = rand_canon(1)[0]
    st = run(harness, [[v] * 3000] * 3, 20, 1)
    assert st["largest"] >= 3000       # every vector piles into its own bucket


def test_zero_vector(harness):
    n = 1200
    rows = [rand_canon(n), [0] * n, rand_canon(n)]
    st = run(harness, rows, 16, 1)
    two = run(harness, [rows[0], rows[2]], 16, 1)
    assert st["entries"] == two["entries"]
    st = run(harness, [[0] * n] * 3, 14, 0)
    assert st["entries"] == 0


def test_01_heavy_next_to_uniform(harness):
    n = 4000
    heavy = [int(x) for x in rs.integers(0, 2, size=n)]
    rows = [rand_canon(n), heavy, rand_canon(n), heavy]
    st = run(harness, rows, 20, 1)
    assert st["tiles"] > 0
    run(harness, rows, 15, 0)


@pytest.mark.parametrize("c,off", [(16, 0), (20, 4097)])
def test_table_sub_range(harness, c, off):
    n = 2000
    run(harness, [rand_canon(n) for _ in range(3)], c, 1, ent_stride=off + n + 11, ent_off=off)


# ---- per-call limits (msm_batch_max): restated, checked over every width / table state / size
def batch_max(c, table, n):
    W = msm_num_windows(c)
    nb = (1 if table else W) << (c - 1)
    k = MAX_BUCKETS // nb
    if n:
        k = min(k, MAX_ENTRIES // (n * W))
    return max(k, 1)


@pytest.mark.parametrize("table", [0, 1])
def test_batch_limits_every_shape(table):
    for c in range(2, 25):
        W = msm_num_windows(c)
        nbw = 1 << (c - 1)
        for lg in range(0, 27):
            n = 1 << lg
            if n * W >= 4.0e9 or (table and n * W >= 2.0e9):
                continue                      # the single MSM refuses these already
            k = batch_max(c, table, n)
            if k < 2:
                continue                      # one vector per call: the single-MSM path
            buckets = k * nbw * (1 if table else W)
            assert buckets <= MAX_BUCKETS
            assert k * n * W <= MAX_ENTRIES
            F = 0
            while (buckets + (1 << F) - 1) >> F > 2048:
                F += 1
            assert F <= 12
            # value = (w * ent_stride + ent_off + i) << 1 | neg does not depend on k: its point index stays below 2^31
            top = ((W - 1) * n + n - 1) if table else (n - 1)
            assert top < 1 << 31 and (top << 1 | 1) < 1 << 32


def pick_window(n):
    """msm_pick_window (msm_common.cu), restated"""
    return min(range(4, 18), key=lambda c: (msm_num_windows(c) * (n + 8.0 * (1 << (c - 1))), c))


def pick_table_window(n):
    """msm_pick_table_window (msm_common.cu), restated"""
    def fits(c):
        return n * msm_num_windows(c) < 2.0e9
    if n >= 1 << 24 and fits(22):
        return 22
    if n >= 3 << 17 and fits(20):
        return 20
    cands = [c for c in range(8, 18) if fits(c)]
    return min(cands, key=lambda c: (msm_num_windows(c) * n + 4.0 * (1 << (c - 1)), c)) if cands else 8


def test_batch_limits_library_widths():
    """Vectors per call at the widths the library picks for itself, 2^16 .. 2^24."""
    want_plain = {16: 341, 18: 102, 20: 30, 22: 8, 24: 8}
    want_table = {16: 512, 18: 128, 20: 16, 22: 16, 24: 4}
    for lg in want_plain:
        n = 1 << lg
        assert batch_max(pick_window(n), 0, n) == want_plain[lg], lg
        assert batch_max(pick_table_window(n), 1, n) == want_table[lg], lg
