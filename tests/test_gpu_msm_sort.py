"""GPU: the MSM on inputs aimed at the two-level counting sort (csrc/msm_sort.cuh) — buckets on both sides of the
coarse-bin edges, one bin holding almost every entry (many tiles of one bin), tiny n, n off the coarse passes' point
tile, window-table sub-ranges, and the wide plain windows whose fine passes use global atomics.  Expected values are
closed forms over bases k_i * G with known k_i, compared limb for limb (see tests/test_gpu_msm_edges.py); the same
shapes are checked slot by slot on the CPU in tests/test_msm_sort_host_cpu.py."""
import random

import pytest

from oracle.bn254 import R
from tests.test_gpu_msm_edges import _check

pytestmark = pytest.mark.gpu

SORT_POINTS = 2048   # points per CTA of the coarse passes


@pytest.fixture(scope="module")
def sctx():
    from gnark_whir_b200 import lib
    c = lib.Context(0)
    yield c
    c.close()


def _ks(rng, n):
    return [rng.randrange(1, R) for _ in range(n)]


def _edge_scalars(c):
    """Digits on both sides of every coarse-bin edge of a c-bit table (bins of 2^(c - 12) buckets), both signs, in
    windows 0, 1 and 5."""
    F = max(0, c - 12)
    out = []
    for b in (0, 1, (1 << F) - 1, 1 << F, (1 << F) + 1, (2 << F) - 1, 2 << F, 1 << (c - 2), (1 << (c - 1)) - (1 << F) - 1,
              (1 << (c - 1)) - (1 << F), (1 << (c - 1)) - 1):
        for s in (b + 1, (1 << c) - (b + 1)):
            out += [s, s << c, s << (5 * c)]
    return out


@pytest.mark.parametrize("group,c", [(1, 20), (1, 16), (2, 16)])
def test_coarse_bin_edges_table(sctx, group, c):
    rng = random.Random(c + 100 * group)
    ss = _edge_scalars(c) * 5
    ss += [rng.randrange(R) for _ in range(64)]
    assert _check(sctx, group, _ks(rng, len(ss)), ss, table=c) == c


@pytest.mark.parametrize("group", [1, 2])
def test_coarse_bin_edges_plain(sctx, group):
    rng = random.Random(7 + group)
    ss = [s % R for s in _edge_scalars(16)] * 3
    assert _check(sctx, group, _ks(rng, len(ss)), ss, c=16) == 16


@pytest.mark.parametrize("group,n,table", [(1, 60000, 20), (1, 60000, None), (2, 20000, 16)])
def test_dominant_bin(sctx, group, n, table):
    rng = random.Random(n + group)
    ss = [1 if i % 200 else rng.randrange(R) for i in range(n)]   # 99.5% of the entries in bucket 0
    _check(sctx, group, _ks(rng, n), ss, table=table)


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("n", [1, 2, SORT_POINTS - 1, SORT_POINTS + 1, 2 * SORT_POINTS + 3])
def test_tiny_and_ragged_n(sctx, group, n):
    rng = random.Random(n * 3 + group)
    ks, ss = _ks(rng, n), [rng.randrange(R) for _ in range(n)]
    _check(sctx, group, ks, ss)
    if group == 1 or n <= SORT_POINTS + 1:
        _check(sctx, group, ks, ss, table=0)


@pytest.mark.parametrize("group,c,offset", [(1, 20, 4097), (1, 16, 1), (2, 12, 2049)])
def test_table_sub_range(sctx, group, c, offset):
    rng = random.Random(offset + c)
    total = offset + 3000 + 17
    ks, ss = _ks(rng, total), [rng.randrange(R) for _ in range(total)]
    assert _check(sctx, group, ks, ss, table=c, offset=offset, n=3000) == c


@pytest.mark.parametrize("group,c", [(1, 20), (1, 21), (2, 20)])
def test_wide_plain(sctx, group, c):
    """c = 20 plain: 13 x 2^19 buckets, the widest shared fine histogram (2^12 keys); c = 21: global fine atomics."""
    rng = random.Random(c * 5 + group)
    n = 3000
    ss = [rng.randrange(R) for _ in range(n - 3)] + [1, R - 1, (1 << (c - 1)) - 1]
    assert _check(sctx, group, _ks(rng, n), ss, c=c) == c


SORT_STAGE = 10240   # entries staged per CTA of the coarse partition: its point tile is SORT_STAGE // W


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("k,d", [(1, -1), (1, 1), (5, 1)])
def test_n_off_partition_tile(sctx, group, k, d):
    """n next to a multiple of the coarse partition's point tile, with a c = 16 table (W = 16: 640 points per CTA)."""
    from tests.test_msm_digits_cpu import msm_num_windows
    n = k * (SORT_STAGE // msm_num_windows(16)) + d
    rng = random.Random(17 * k + d + group)
    ks, ss = _ks(rng, n), [rng.randrange(R) for _ in range(n)]
    assert _check(sctx, group, ks, ss, table=16) == 16
