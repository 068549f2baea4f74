"""GPU parity of the Fr NTT and computeH at every size the C-ABI accepts, against the C restatement (oracle.cport),
bit-exact on every output limb.

ntt.cu splits L levels into ceil(L/8) passes (uneven at many sizes: 9 -> 5+4, 17 -> 6+6+5, 25 -> 7+6+6+6) and keeps
state between calls: the twiddle table of the largest size seen so far (read with stride 2^tw_sh by smaller
transforms), and coset / fused / distributed scaling tables rebuilt when the size changes.  The contexts here are
this file's own, so which table state a transform meets is set by the test and not by the order of the suite:
  * every size 0..24, all 8 variants (forward / inverse x plain / coset x DIF / DIT), random and edge inputs, on a
    context that only grew (tw_sh = 0) and on one that ran 2^26 first (tw_sh > 0), with guard words around the data;
  * the 4-pass sizes 2^25 .. 2^28 (skipped, with the free memory in the reason, when it does not fit);
  * batched transforms (blockIdx.y), computeH through three paths at every size, size changes on one context;
  * the distributed computeH (k_ntt_cross / k_ntt_cross_h) through lib.Group at its smallest shape, with local parts
    of 1, 2 and 3 passes, size changes within one group, and through CUDA IPC at world 2, 4 and 8.
"""
import socket

import numpy as np
import pytest
import torch

from gnark_whir_b200 import lib
from oracle import bn254 as bn
from oracle import cport, synth
from oracle.bn254 import R

pytestmark = pytest.mark.gpu

VARIANTS = [(inv, cos, dec) for inv in (False, True) for cos in (False, True) for dec in (lib.DIF, lib.DIT)]
GUARD = 3                                                     # rows of 32 bytes before and after the data
SENTINEL = np.uint64(0xC0FFEE00DEADBEEF)
R_MINUS_1 = np.array([((R - 1) >> (64 * i)) & ((1 << 64) - 1) for i in range(4)], dtype=np.uint64)
SMALL = 16                                                    # edge inputs run all 8 variants up to this size
BIG_L = 26                                                    # context B runs one transform of this size first


def _vid(v):
    inv, cos, dec = v
    return ("inv" if inv else "fwd") + ("_coset" if cos else "") + ("_dit" if dec == lib.DIT else "_dif")


def _mont(vals):
    return bn.fr_to_mont_array([v % R for v in vals])


def _rand(L, seed):
    return synth.rand_fr(np.random.Generator(np.random.PCG64(seed)), 1 << L)


class Tracked:
    """A context and the twiddle-table state it is in: ensure_twiddles keeps the table of the largest size seen so
    far, and a transform of 2^L reads it with stride 2^tw_sh, tw_sh = tw_log - L."""

    def __init__(self):
        self.c = lib.Context(0)
        self.tw_log = -1

    def tw_sh(self, L):
        self.tw_log = max(self.tw_log, L)
        return self.tw_log - L

    def close(self):
        self.c.close()


def _guarded(rows):
    """(device tensor, pointer to the data): `rows` framed by GUARD sentinel rows on both sides."""
    buf = np.full((rows.shape[0] + 2 * GUARD, 4), SENTINEL, dtype=np.uint64)
    buf[GUARD:GUARD + rows.shape[0]] = rows
    t = torch.from_numpy(buf.view(np.int64)).cuda()
    torch.cuda.synchronize()
    return t, t.data_ptr() + 32 * GUARD


def _unguard(t, n):
    buf = t.cpu().numpy().view(np.uint64)
    assert (buf[:GUARD] == SENTINEL).all(), "guard words before the data were written"
    assert (buf[GUARD + n:] == SENTINEL).all(), "guard words after the data were written"
    return buf[GUARD:GUARD + n]


def _ntt_dev(tc, rows, L, inverse, coset, dec):
    t, p = _guarded(rows)
    tc.c.ntt_dev(p, L, inverse=inverse, coset=coset, decimation=dec)
    return _unguard(t, rows.shape[0])


def _edge_inputs(L):
    """name -> (rows, {variant: closed-form output}) for inputs whose transforms have closed forms (the forms hold for
    the listed variants; every variant is also compared with the C port where that runs)."""
    N = 1 << L
    out = {"zeros": (np.zeros((N, 4), np.uint64), {v: np.zeros((N, 4), np.uint64) for v in VARIANTS})}
    cv = 0x1234567890ABCDEF1234567 % R
    const = np.tile(_mont([cv]), (N, 1))
    spike = lambda x: np.concatenate([_mont([x]), np.zeros((N - 1, 4), np.uint64)])   # noqa: E731
    out["const"] = (const, {(False, False, lib.DIF): spike(cv * N), (False, False, lib.DIT): spike(cv * N),
                            (True, False, lib.DIF): spike(cv), (True, False, lib.DIT): spike(cv)})
    for p in sorted({0, min(1, N - 1), N - 1}):
        d = np.zeros((N, 4), np.uint64)
        d[p] = _mont([cv])[0]
        forms = {}
        if p == 0:       # a delta at 0 transforms to a constant (g^0 = 1 on the coset too)
            forms = {v: const for v in VARIANTS if not v[0]}
            inv_n = np.tile(_mont([cv * pow(N, -1, R)]), (N, 1))
            forms.update({(True, False, lib.DIF): inv_n, (True, False, lib.DIT): inv_n})
        out[f"delta{p}"] = (d, forms)
    alt = np.zeros((N, 4), np.uint64)
    alt[1::2] = R_MINUS_1                                     # raw limbs 0, r-1, 0, r-1, ...: add / sub wrap at every level
    out["alt0r1"] = (alt, {})
    return out


@pytest.fixture(scope="module")
def ctx_fresh():
    tc = Tracked()
    yield tc
    tc.close()


@pytest.fixture(scope="module")
def ctx_strided():
    tc = Tracked()
    z = torch.zeros((1 << BIG_L, 4), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    tc.c.ntt_dev(z.data_ptr(), BIG_L, decimation=lib.DIF)
    assert tc.tw_sh(BIG_L) == 0
    assert not z.any().item()
    del z
    yield tc
    tc.close()


@pytest.mark.parametrize("L", range(25))
def test_ntt_every_size_and_table_state(ctx_fresh, ctx_strided, L):
    """Both contexts, in ascending L: context A builds a table per size (tw_sh = 0), context B reads its 2^26 table
    with stride 2^(26 - L).  Random input through ntt_dev inside guard words, edge inputs through b200g16_ntt."""
    assert ctx_fresh.tw_sh(L) == 0
    assert ctx_strided.tw_sh(L) == BIG_L - L > 0
    a = _rand(L, 9000 + L)
    edges = _edge_inputs(L)
    for v in VARIANTS:
        inv, cos, dec = v
        want = cport.ntt(a, inv, cos, dec)
        for tc in (ctx_fresh, ctx_strided):
            got = _ntt_dev(tc, a, L, inv, cos, dec)
            assert np.array_equal(got, want), f"random input, {_vid(v)}, tw_sh {tc.tw_log - L}"
        for name, (x, forms) in edges.items():
            ref = None
            if L <= SMALL or (v not in forms and v in ((False, False, lib.DIF), (True, True, lib.DIT))):
                ref = cport.ntt(x, inv, cos, dec)
            if v in forms:
                if ref is not None:
                    assert np.array_equal(ref, forms[v]), f"closed form of {name}, {_vid(v)}"
                ref = forms[v]
            if ref is None:
                continue
            for tc in (ctx_fresh, ctx_strided):
                got = tc.c.ntt(x, inverse=inv, coset=cos, decimation=dec)
                assert np.array_equal(got, ref), f"{name}, {_vid(v)}, tw_sh {tc.tw_log - L}"


def _meminfo_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


@pytest.mark.parametrize("L", [25, 26, 27, 28])
def test_ntt_four_pass_sizes(L):
    """7+6+6+6 .. 7+7+7+7 levels.  All 8 variants at 2^25 and 2^26; forward DIF and inverse coset DIF at 2^27, 2^28."""
    vec = (1 << L) * 32
    free_dev, _ = torch.cuda.mem_get_info(0)
    free_host = _meminfo_available()
    # device: data (+1/8 slack), twiddles (N/2), coset tables (2N);  host: input, result, C port's copy and tables
    if free_dev < 4 * vec or free_host < 5 * vec:
        pytest.skip(f"2^{L}: {free_dev / 2**30:.1f} GiB free on the device (needs {4 * vec / 2**30:.0f}), "
                    f"{free_host / 2**30:.1f} GiB available on the host (needs {5 * vec / 2**30:.0f})")
    variants = VARIANTS if L <= 26 else [(False, False, lib.DIF), (True, True, lib.DIF)]
    a = _rand(L, 9000 + L)
    with lib.Context(0) as c:
        for inv, cos, dec in variants:
            got = c.ntt(a, inverse=inv, coset=cos, decimation=dec)
            want = cport.ntt(a, inv, cos, dec)
            assert np.array_equal(got, want), f"2^{L} {_vid((inv, cos, dec))}"
            del got, want


@pytest.fixture(scope="module")
def ctx_batch():
    tc = Tracked()
    yield tc
    tc.close()


@pytest.mark.parametrize("L", [1, 8, 9, 17])
@pytest.mark.parametrize("batch", [2, 3, 5])
@pytest.mark.parametrize("inverse,coset", [(False, False), (False, True), (True, False), (True, True)])
def test_ntt_batched(ctx_batch, L, batch, inverse, coset):
    """b200g16_ntt_dev over `batch` consecutive vectors (grid.y): each equals its own single-vector transform, and
    nothing past the last vector is written."""
    N = 1 << L
    vecs = [_rand(L, 500 * L + 10 * batch + i) for i in range(batch)]
    ctx_batch.tw_sh(L)
    for dec in (lib.DIF, lib.DIT):
        t, p = _guarded(np.concatenate(vecs))
        ctx_batch.c.ntt_dev(p, L, batch=batch, inverse=inverse, coset=coset, decimation=dec)
        got = _unguard(t, batch * N)
        for i, v in enumerate(vecs):
            assert np.array_equal(got[i * N:(i + 1) * N], cport.ntt(v, inverse, coset, dec)), f"vector {i}, dec {dec}"


def _abc(L, n, seed):
    rs = np.random.Generator(np.random.PCG64(seed))
    a, b = synth.rand_fr(rs, n), synth.rand_fr(rs, n)
    c = synth.rand_fr(rs, n)
    c[::2] = bn.fr_to_mont_array([x * y % R for x, y in zip(bn.fr_from_mont_array(a[::2]), bn.fr_from_mont_array(b[::2]))])
    return a, b, c


def _pad(v, N):
    out = np.zeros((N, 4), np.uint64)
    out[:v.shape[0]] = v
    return out


def _compute_h_three_ways(c, a, b, cc, L):
    """b200g16_compute_h (host), b200g16_compute_h_dev, and the staged sequence of sharded.py."""
    N = 1 << L
    out = {"host": c.compute_h(a, b, cc, L)}
    ts = [torch.from_numpy(_pad(v, N).view(np.int64)).cuda() for v in (a, b, cc)]
    torch.cuda.synchronize()
    c.compute_h_dev(*[t.data_ptr() for t in ts], L)
    out["dev"] = ts[0].cpu().numpy().view(np.uint64).copy()
    ts = [torch.from_numpy(_pad(v, N).view(np.int64)).cuda() for v in (a, b, cc)]
    torch.cuda.synchronize()
    for t in ts:
        c.ntt_dev(t.data_ptr(), L, inverse=True, decimation=lib.DIF)
        c.ntt_dev(t.data_ptr(), L, coset=True, decimation=lib.DIT)
    c.h_pointwise_dev(*[t.data_ptr() for t in ts], L)
    c.ntt_dev(ts[0].data_ptr(), L, inverse=True, coset=True, decimation=lib.DIF)
    out["staged"] = ts[0].cpu().numpy().view(np.uint64).copy()
    return out


def _h_sizes():
    out = []
    for L in list(range(23)) + [24, 26]:
        N = 1 << L
        ns = [N, N - 1, N // 2 + 1, 1, 0] if L <= 24 else [N - 1, 0]   # 2^26: one C-port computeH takes minutes
        out += [(L, n) for n in dict.fromkeys(ns)]
    return out


@pytest.fixture(scope="module")
def ctx_h():
    tc = Tracked()
    yield tc
    tc.close()


@pytest.mark.parametrize("L,n_constraints", _h_sizes())
def test_compute_h_every_size(ctx_h, L, n_constraints):
    a, b, c = _abc(L, n_constraints, 7000 + L)
    want = cport.compute_h(a, b, c, L) if n_constraints else np.zeros((1 << L, 4), np.uint64)
    ctx_h.tw_sh(L)
    for path, got in _compute_h_three_ways(ctx_h.c, a, b, c, L).items():
        assert np.array_equal(got, want), f"{path} path, 2^{L}, {n_constraints} constraints"


def test_size_changes_on_one_context():
    """computeH and coset transforms alternating over sizes on ONE context: each size change rebuilds the coset and
    fused tables (and a smaller size reads the larger twiddle table with a stride)."""
    cache = {}
    with lib.Context(0) as c:
        for L in (20, 9, 20, 12, 9):
            N = 1 << L
            if L not in cache:
                a, b, cc = _abc(L, N - 3, 300 + L)
                x = _rand(L, 400 + L)
                cache[L] = (a, b, cc, x, cport.compute_h(a, b, cc, L),
                            {v: cport.ntt(x, *v) for v in VARIANTS if v[1]})
            a, b, cc, x, h_want, ntt_want = cache[L]
            assert np.array_equal(c.compute_h(a, b, cc, L), h_want), f"computeH 2^{L}"
            for v, want in ntt_want.items():
                assert np.array_equal(c.ntt(x, inverse=v[0], coset=True, decimation=v[2]), want), f"2^{L} {_vid(v)}"
            assert np.array_equal(_compute_h_three_ways(c, a, b, cc, L)["staged"], h_want), f"staged computeH 2^{L}"


# ---- distributed computeH through lib.Group ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx_keys():
    with lib.Context(0) as c:
        yield c


def _group_key(c, L, seed):
    """Whole proving key over points with known discrete logs (as test_gpu_group.py's 2^18 test builds it)."""
    N = 1 << L
    rs = np.random.Generator(np.random.PCG64(seed))
    ks = {"a": synth.rand_fr(rs, N), "b": synth.rand_fr(rs, N), "k": synth.rand_fr(rs, N - 1), "z": synth.rand_fr(rs, N - 1),
          "b2": synth.rand_fr(rs, N)}
    small = synth.rand_fr(rs, 5)
    pts = {n: c.fixed_base_mul(synth.G1, ks[n], group=1) for n in ("a", "b", "k", "z")}
    pts["b2"] = c.fixed_base_mul(synth.G2, ks["b2"], group=2)
    g1s, g2s = c.fixed_base_mul(synth.G1, small[:3], group=1), c.fixed_base_mul(synth.G2, small[3:], group=2)
    k_skip = np.zeros(N, np.uint8)
    k_skip[0] = 1
    key = synth.KnownDlogKey.__new__(synth.KnownDlogKey)
    key.L, key.N, key.k, key.small = L, N, ks, small
    args = (L, N, pts["a"], pts["b"], pts["k"], pts["z"], pts["b2"], g1s[0], g1s[1], g1s[2], g2s[0], g2s[1],
            np.zeros(N, np.uint8), np.zeros(N, np.uint8), k_skip)
    return key, args


def _group_devices():
    out = [[0] * 2, [0] * 4, [0] * 8]
    n = torch.cuda.device_count()
    out += [list(range(k)) for k in (2, 4, 8) if n >= k]
    return out


@pytest.mark.parametrize("devices", _group_devices(), ids=lambda d: "dev" + "_".join(map(str, d)))
def test_group_dist_h_every_shape_and_size_change(ctx_keys, devices):
    """ONE group proves keys of several sizes in turn: L = 2g (the owner path), then split over the devices with
    local parts of >= 17, <= 8 and 9..16 levels (3, 1 and 2 passes), 2g + 1 (the smallest split: 2 offsets per
    device in the cross kernels) and the first split size again.  h and every proof output against the closed forms,
    with ragged constraint counts; one count leaves every slice but the first all zero padding.  The split sizes
    first shrink, so tables kept from a larger size are only ever read within their bounds."""
    G = len(devices)
    g = G.bit_length() - 1
    sizes = [2 * g, g + 17, g + 8, g + 13, 2 * g + 1, g + 17]
    rs = np.random.Generator(np.random.PCG64(60 + G))
    keys = {}
    with lib.Group(devices) as grp:
        for step, L in enumerate(sizes):
            N, M = 1 << L, (1 << L) >> g
            if L not in keys:
                keys[L] = _group_key(ctx_keys, L, 1000 * g + L)
            key, args = keys[L]
            n_c = [N - 1, N, M // 2 + 1, N // 2 + 1, N - 1, N - 5][step]
            wires = synth.whir_mix(rs, N)
            a, b, c = synth.rand_fr(rs, n_c), synth.rand_fr(rs, n_c), synth.rand_fr(rs, n_c)
            r, s = synth.rand_fr(rs, 1)[0], synth.rand_fr(rs, 1)[0]
            exp, h_exp = key.expected(wires, a, b, c, r, s)
            pk = grp.pk_upload(*args)
            try:
                got, h = grp.prove(pk, wires, a, b, c, r, s, want_h=True, log2_domain=L)
            finally:
                grp.pk_free(pk)
            assert np.array_equal(h, h_exp), f"h, step {step}: 2^{L} over {G} devices, {n_c} constraints"
            assert synth.check_proof(got, exp) == [], f"proof, step {step}: 2^{L} over {G} devices"


# ---- distributed computeH through CUDA IPC, one process per rank ---------------------------------------------------
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("shape", ["smallest", "3pass"])
def test_distributed_h_over_cuda_ipc(world, shape):
    import torch.multiprocessing as mp

    from tests.test_gpu_group import _dist_h_worker
    g = world.bit_length() - 1
    L = 2 * g + 1 if shape == "smallest" else 17 + g
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mctx = mp.get_context("spawn")
    q = mctx.Queue()
    procs = [mctx.Process(target=_dist_h_worker, args=(r, world, port, L, q)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        res = sorted(q.get(timeout=900) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.terminate()
                p.join()
    assert res == [(r, True) for r in range(world)], f"2^{L} over {world} ranks"
