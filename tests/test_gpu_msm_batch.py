"""GPU: batch MSMs (b200g16_msm_g1_batch / _g2_batch and the _dev forms): k scalar vectors over one resident bases
vector in one call.  Every row must equal the single-call MSM of that row, limb for limb, and the closed form over
bases with known discrete logs ([<k, s_j>] G, oracle C port).  Covers G1 plain and with a window table, G2, sizes
1 .. 2^20, the sub-batch boundary (2^20 with a c = 20 table: 16 vectors per call), identical / all-zero / 0-1-heavy
rows, sub-ranges, device scalars, a batch next to proves and an open asynchronous ticket, and every argument and
state error with the context usable afterwards."""
import ctypes as C

import numpy as np
import pytest

from gnark_whir_b200 import lib
from oracle import bn254 as bn
from oracle import cport
from oracle.synth import G1, G2, KnownDlogKey, check_proof, rand_fr, whir_mix

pytestmark = pytest.mark.gpu

NMAX = 1 << 20
rs = np.random.Generator(np.random.PCG64(20261021))


@pytest.fixture(scope="module")
def vecs(ctx):
    """known-discrete-log bases: G1 plain and with a table (2^20), G2 plain (2^16) and with a table (2^18)"""
    kg1, kg2 = rand_fr(rs, NMAX), rand_fr(rs, 1 << 18)
    out = {"g1": (ctx.fixed_base_mul(G1, kg1, group=1, resident=True), kg1),
           "g1t": (ctx.fixed_base_mul(G1, kg1, group=1, resident=True), kg1),
           "g2": (ctx.fixed_base_mul(G2, kg2[:1 << 16], group=2, resident=True), kg2[:1 << 16]),
           "g2t": (ctx.fixed_base_mul(G2, kg2, group=2, resident=True), kg2)}
    out["g1t"][0].precompute(0)
    out["g2t"][0].precompute(0)
    yield out
    for b, _ in out.values():
        b.free()


def closed(kind, ks, sc):
    d = cport.fr_dot(ks, sc)
    return cport.g1_gen_mul(d) if kind.startswith("g1") else cport.g2_gen_mul(d)


def check_rows(ctx, kind, b, ks, sc, got, offset=0, closed_rows=None):
    k, n = sc.shape[0], sc.shape[1]
    assert got.shape == (k, 8 if kind.startswith("g1") else 16)
    for j in range(k):
        assert np.array_equal(got[j], ctx.msm(b, sc[j], offset=offset)), f"row {j} differs from the single MSM"
    for j in (range(k) if closed_rows is None else closed_rows):
        if n:
            assert np.array_equal(got[j], closed(kind, ks[offset:offset + n], sc[j])), f"row {j} differs from the closed form"


@pytest.mark.parametrize("kind", ["g1", "g1t", "g2", "g2t"])
@pytest.mark.parametrize("n", [1, 3, 1000, 1 << 16, 1 << 20])
@pytest.mark.parametrize("k", [1, 2, 5, 64])
def test_rows_equal_single_calls(ctx, vecs, kind, n, k):
    b, ks = vecs[kind]
    if n > b.n or (n == 1 << 20 and k == 64 and kind != "g1t"):
        pytest.skip("bases shorter than n / covered by the table form")
    sc = np.stack([whir_mix(rs, n) if j % 2 else rand_fr(rs, n) for j in range(k)])
    got = ctx.msm_batch(b, sc)
    check_rows(ctx, kind, b, ks, sc, got, closed_rows=None if n * k <= 1 << 22 else [0, k - 1])


@pytest.mark.parametrize("k", [15, 16, 17])
def test_sub_batch_boundary(ctx, vecs, k):
    b, ks = vecs["g1t"]
    assert b.window() == 20
    sc = np.stack([rand_fr(rs, NMAX) for _ in range(k)])
    got = ctx.msm_batch(b, sc)
    for j in range(k):
        assert np.array_equal(got[j], closed("g1", ks, sc[j])), f"row {j}"
    assert np.array_equal(got[k - 1], ctx.msm(b, sc[k - 1]))


@pytest.mark.parametrize("kind", ["g1", "g1t", "g2"])
def test_special_rows(ctx, vecs, kind):
    b, ks = vecs[kind]
    n = 5000
    row = rand_fr(rs, n)
    zero = np.zeros((n, 4), dtype=np.uint64)
    one = bn.fr_to_mont_array([1])[0]
    heavy = np.where((rs.integers(0, 2, size=n) == 1)[:, None], one, zero)
    sc = np.stack([row, row, zero, heavy, rand_fr(rs, n), row])
    got = ctx.msm_batch(b, sc)
    check_rows(ctx, kind, b, ks, sc, got)
    assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], got[5])
    assert not got[2].any(), "an all-zero row is the point at infinity"
    # every row zero
    z = ctx.msm_batch(b, np.zeros((3, n, 4), dtype=np.uint64))
    assert not z.any()


@pytest.mark.parametrize("kind", ["g1", "g1t", "g2"])
def test_sub_range(ctx, vecs, kind):
    b, ks = vecs[kind]
    off, n = 12345, 7000
    sc = np.stack([whir_mix(rs, n) for _ in range(4)])
    got = ctx.msm_batch(b, sc, offset=off)
    check_rows(ctx, kind, b, ks, sc, got, offset=off)


@pytest.mark.parametrize("kind", ["g1t", "g2"])
def test_device_scalars(ctx, vecs, kind):
    import torch
    b, ks = vecs[kind]
    n, k = 30000, 6
    sc = np.stack([rand_fr(rs, n) for _ in range(k)])
    dev = torch.from_numpy(sc.reshape(-1, 4).view(np.int64)).cuda()
    got = ctx.msm_batch(b, dev.data_ptr(), n=n, k=k)
    assert np.array_equal(got, ctx.msm_batch(b, sc))
    check_rows(ctx, kind, b, ks, sc, got, closed_rows=[0, k - 1])


def test_batch_between_proves_and_under_an_open_ticket(ctx, vecs):
    key = KnownDlogKey(ctx, 14, seed=77)
    try:
        N = key.N
        wires, a, b_ = whir_mix(rs, N), rand_fr(rs, N - 3), rand_fr(rs, N - 3)
        c = rand_fr(rs, N - 3)
        r, s = rand_fr(rs, 1)[0], rand_fr(rs, 1)[0]
        exp, _ = key.expected(wires, a, b_, c, r, s)
        bg, kg = vecs["g1"]
        tsc = rand_fr(rs, 3000)
        ticket = ctx.msm_begin(bg, tsc)
        got1, _ = ctx.prove(key.handle, wires, a, b_, c, r, s)
        sc = np.stack([rand_fr(rs, 20000) for _ in range(3)])
        got = ctx.msm_batch(vecs["g1t"][0], sc)
        got2, _ = ctx.prove(key.handle, wires, a, b_, c, r, s)
        assert np.array_equal(ctx.msm_end(ticket), closed("g1", kg[:3000], tsc))
        assert check_proof(got1, exp) == [] and check_proof(got2, exp) == []
        for j in range(3):
            assert np.array_equal(got[j], closed("g1", vecs["g1t"][1][:20000], sc[j]))
    finally:
        key.free()


def _raw(ctx, fn, b, off, ptr, n, k, out):
    return getattr(lib.load(), fn)(ctx.h, b.handle if b is not None else None, off, ptr, n, k, out)


def test_errors_leave_the_ctx_usable(ctx, vecs):
    L = lib.load()
    b1, k1 = vecs["g1"]
    b2, _ = vecs["g2"]
    sc = rand_fr(rs, 2 * 100).reshape(2, 100, 4)
    out = np.zeros((2, 16), dtype=np.uint64)
    p, o = sc.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)
    ERR_ARG, ERR_STATE = -2, -4
    for fn in ("b200g16_msm_g1_batch", "b200g16_msm_g1_batch_dev"):
        assert _raw(ctx, fn, b1, 0, None, 100, 2, o) == ERR_ARG                  # null scalars
        assert _raw(ctx, fn, b1, 0, p, 100, 2, None) == ERR_ARG                  # null out
        assert _raw(ctx, fn, None, 0, p, 100, 2, o) == ERR_ARG                   # null bases
        assert _raw(ctx, fn, b2, 0, p, 100, 2, o) == ERR_ARG                     # wrong group
        assert _raw(ctx, fn, b1, b1.n - 50, p, 100, 2, o) == ERR_ARG             # range
        assert _raw(ctx, fn, b1, 0, p, 1 << 31, 2, o) == ERR_ARG                 # n >= 2^31 (and beyond the bases)
        assert _raw(ctx, fn, b1, 0, p, 100, (1 << 64) // 100, o) == ERR_ARG      # k x n overflows size_t
        assert _raw(ctx, fn, b1, 0, None, 100, 0, None) == 0                     # k = 0: nothing
    assert _raw(ctx, "b200g16_msm_g2_batch", b1, 0, p, 100, 2, o) == ERR_ARG
    assert not out.any(), "an error wrote results"
    # between the halves of a split prove
    key = KnownDlogKey(ctx, 12, seed=5)
    try:
        import torch
        w = torch.from_numpy(whir_mix(rs, key.N).view(np.int64)).cuda()
        ctx.prove_begin_dev(key.handle, w.data_ptr())
        assert _raw(ctx, "b200g16_msm_g1_batch", b1, 0, p, 100, 2, o) == ERR_STATE
        h = torch.zeros((key.N, 4), dtype=torch.int64, device="cuda")
        ctx.prove_end_dev(key.handle, h.data_ptr(), rand_fr(rs, 1)[0], rand_fr(rs, 1)[0])
    finally:
        key.free()
    got = ctx.msm_batch(b1, sc)
    check_rows(ctx, "g1", b1, k1, sc, got)
