"""The MSM's two-level counting sort (gnark_whir_b200/csrc/msm_sort.cuh) compiled for the host and run CTA by CTA
against a direct counting sort: counts, offsets, task offsets and every bucket's multiset of entries must match, and
every slot must be written exactly once.  Covers the shapes the sort has to split cleanly: uniform scalars, a
WHIR-shaped witness, equal scalars, buckets on coarse-bin edges, one bin holding almost everything, tiny n, n off the
CTA's point tile, window-table sub-ranges and the wide plain windows that place with global atomics."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import bn254 as bn
from tests.test_msm_digits_cpu import msm_num_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "host_harness", "sort_host.cc")
OUT = os.path.join(ROOT, "tests", "host_harness", "_build", "sort_host.so")

SORT_POINTS = 2048   # points per CTA of the coarse passes
SORT_TILE = 8192     # entries per tile of the fine passes


@pytest.fixture(scope="module")
def harness():
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-I",
                    os.path.join(ROOT, "gnark_whir_b200", "csrc"), "-o", OUT], check=True)
    return ctypes.CDLL(OUT)


rs = np.random.Generator(np.random.PCG64(20261020))


def rand_canon(n):
    return [int(x) % bn.R for x in (int.from_bytes(rs.bytes(32), "little") for _ in range(n))]


def run(harness, vals, c, table, ent_stride=0, ent_off=0, seed=1):
    sc = np.ascontiguousarray(bn.fr_to_mont_array(vals))
    W = msm_num_windows(c)
    stats = (ctypes.c_uint32 * 5)()
    rc = harness.sort_host(sc.ctypes.data_as(ctypes.c_void_p), ctypes.c_uint32(len(vals)), ctypes.c_int(c),
                           ctypes.c_int(W), ctypes.c_int(table), ctypes.c_uint32(ent_stride), ctypes.c_uint32(ent_off),
                           ctypes.c_uint64(seed), stats)
    assert rc == 0, f"sort differs from the direct counting sort (code {rc})"
    return dict(zip(("F", "bins", "tiles", "entries", "largest"), list(stats)))


def whir_mix(n):
    k = rs.integers(0, 10, size=n)
    out = []
    for i, v in enumerate(rand_canon(n)):
        out.append(1 if k[i] < 2 else int(k[i] & 1) if k[i] < 5 else int(v & 0xFF) if k[i] < 8 else v)
    return out


@pytest.mark.parametrize("c", [8, 16, 20, 22])
def test_uniform_table(harness, c):
    st = run(harness, rand_canon(3 * SORT_POINTS + 77), c, table=1)
    assert st["bins"] <= 2048 and st["F"] <= 12


@pytest.mark.parametrize("c", [4, 11, 16, 17])
def test_uniform_plain(harness, c):
    run(harness, rand_canon(2 * SORT_POINTS + 5), c, table=0)


@pytest.mark.parametrize("table", [0, 1])
def test_whir_mix(harness, table):
    run(harness, whir_mix(5000), 20 if table else 16, table=table)


def test_all_equal(harness):
    v = rand_canon(1)[0]
    st = run(harness, [v] * 12000, 20, table=1)
    assert st["largest"] >= 12000      # one bucket per window, several tiles of one bin
    run(harness, [v] * 3000, 12, table=0)


def test_coarse_bin_edges(harness):
    # table c = 20: F = 8, bucket = |digit| - 1, bins of 256 buckets; digits on both sides of each edge, both signs
    c = 20
    vals = []
    for b in (0, 1, 255, 256, 257, 511, 512, 1 << 18, (1 << 19) - 257, (1 << 19) - 256, (1 << 19) - 1):
        for s in (b + 1, (1 << c) - (b + 1)):           # digit +(b + 1), and -(b + 1) with a carry into window 1
            vals += [s, s << c, s << (5 * c)]
    st = run(harness, vals * 7, c, table=1)
    assert st["F"] == 8 and st["bins"] == 2048
    # plain c = 16: bins straddle window boundaries (bucket = w 2^15 + |d| - 1)
    run(harness, [v % bn.R for v in vals] * 3, 16, table=0)


def test_dominant_bin(harness):
    n = 40000
    vals = [1 if i % 200 else v for i, v in enumerate(rand_canon(n))]   # 99.5% of the scalars are 1: bucket 0
    st = run(harness, vals, 20, table=1)
    assert st["largest"] > 0.9 * st["entries"]
    assert st["tiles"] > st["largest"] // SORT_TILE


@pytest.mark.parametrize("n", [1, 2, SORT_POINTS - 1, SORT_POINTS + 1, 2 * SORT_POINTS])
def test_small_and_ragged_n(harness, n):
    run(harness, rand_canon(n), 20, table=1)
    run(harness, rand_canon(n), 15, table=0)


@pytest.mark.parametrize("c,off", [(16, 0), (20, 4097), (20, 12345)])
def test_table_sub_range(harness, c, off):
    n = 3000
    run(harness, rand_canon(n), c, table=1, ent_stride=off + n + 11, ent_off=off)


def test_wide_plain_global_fallback(harness):
    st = run(harness, rand_canon(2500), 21, table=0)     # 13 x 2^20 buckets: F = 13, global atomics
    assert st["F"] > 12
    st = run(harness, rand_canon(2500), 20, table=0)     # 13 x 2^19 buckets: F = 12, the widest shared histogram
    assert st["F"] == 12


SORT_STAGE = 10240   # entries staged per CTA of the coarse partition: its point tile is SORT_STAGE // W


@pytest.mark.parametrize("c,table", [(20, 1), (15, 0)])
@pytest.mark.parametrize("k,d", [(1, -1), (1, 1), (3, -1), (3, 1)])
def test_n_off_partition_tile(harness, c, table, k, d):
    n = k * (SORT_STAGE // msm_num_windows(c)) + d
    run(harness, rand_canon(n), c, table=table)
