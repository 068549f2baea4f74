"""CPU model of the NTT's index algebra (csrc/ntt.cu), restated line for line with the kernel's names.

* `schedule` is the pass split of `ntt_device_impl` (npass, ks, b0s, logc, tiles, smem, tfast).  For every size
  L = 1..28 and both decimations: every index bit belongs to exactly one pass (top-down for DIF, bottom-up for DIT),
  k <= NTT_MAX_K, the dynamic shared memory fits the limit set by cudaFuncSetAttribute, tiles * 2^(k + logc) = 2^L
  and the grid fits.
* `tile_index` is the load / store map (tile, x) -> i of `k_ntt_pass`; in numpy for L <= 22 it is a bijection onto
  [0, 2^L) in both shared-memory layouts (TFAST and not), and every twiddle index e << tw_sh stays inside the
  tw_half + 1 entries of the table, for tw_sh = 0 and 28 - L.
* `k_ntt_pass` / `ntt_device_impl` run the passes on Python ints (shared tile, the inverse's sign folding through
  tw[tw_half - idx], the pre / post scaling tables with their bit reversal) and equal oracle.ntt.Domain for all
  8 variants at tw_sh = 0 and 2.
* `compute_h_dist` restates `compute_h_dist_phase` (slices, `cross_levels`, `k_ntt_cross`, `k_ntt_cross_h`, the
  compact tables of `ensure_dist_tables` read at bitrev(o)) and equals oracle.ntt.compute_h for G = 2, 4, 8.
"""
import os
import random
import re

import numpy as np
import pytest

from oracle import ntt as ont
from oracle.bn254 import R

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gnark_whir_b200", "csrc", "ntt.cu")
FR_BYTES = 32
COSET_GEN = 5


def _constexpr(name):
    with open(SRC) as f:
        m = re.search(rf"constexpr int {name} = (\d+);", f.read())
    assert m, name
    return int(m.group(1))


NTT_MAX_K = _constexpr("NTT_MAX_K")
NTT_LOGC = _constexpr("NTT_LOGC")
with open(SRC) as _f:
    _m = re.search(r"const int logc_pref = (\d+);", _f.read())
LOGC_PREF = int(_m.group(1))
SMEM_ATTR = (1 << (NTT_MAX_K + NTT_LOGC)) * FR_BYTES      # cudaFuncAttributeMaxDynamicSharedMemorySize of k_ntt_pass
GRID_X_MAX = (1 << 31) - 1


def bitrev(i, bits):
    return ont.bitrev(i, bits)


def root(L):
    """domain_params(L).w: the 2^L-th root of unity, the 2^28-th root squared 28 - L times."""
    return pow(ont.ROOT_2_28, 1 << (28 - L), R)


# ---- ntt_device_impl: the pass split
class Pass:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def schedule(L, dit):
    npass = (L + NTT_MAX_K - 1) // NTT_MAX_K
    ks = [L // npass + (1 if p < L % npass else 0) for p in range(npass)]
    b0s = []
    if dit:
        b = 0
        for p in range(npass):
            b0s.append(b)
            b += ks[p]
    else:
        b = L
        for p in range(npass):
            b -= ks[p]
            b0s.append(b)
    n = 1 << L
    out = []
    for p in range(npass):
        k, b0 = ks[p], b0s[p]
        logc = L - k if L - k < LOGC_PREF else LOGC_PREF
        tiles = n >> (k + logc)
        smem = (1 << (k + logc)) * FR_BYTES
        out.append(Pass(k=k, b0=b0, logc=logc, tiles=tiles, smem=smem, tfast=(b0 == 0)))
    return out


@pytest.mark.parametrize("dit", [False, True], ids=["dif", "dit"])
@pytest.mark.parametrize("L", range(1, 29))
def test_pass_split_and_launch_bounds(L, dit):
    ps = schedule(L, dit)
    assert len(ps) == -(-L // NTT_MAX_K)
    owned = []
    for p in ps:
        assert 1 <= p.k <= NTT_MAX_K
        assert 0 <= p.logc <= LOGC_PREF
        assert p.smem <= SMEM_ATTR <= 227 * 1024
        assert p.tiles * (1 << (p.k + p.logc)) == 1 << L
        assert 1 <= p.tiles <= GRID_X_MAX
        assert p.tfast == (p.b0 == 0)
        owned.append(list(range(p.b0, p.b0 + p.k)))
    flat = [b for bits in owned for b in bits]
    assert sorted(flat) == list(range(L)), "every index bit belongs to exactly one pass"
    assert flat == (list(range(L)) if dit else [b for p in ps for b in range(p.b0, p.b0 + p.k)])
    b0s = [p.b0 for p in ps]
    assert b0s == (sorted(b0s) if dit else sorted(b0s, reverse=True))   # DIT bottom-up, DIF top-down
    assert max(p.k for p in ps) - min(p.k for p in ps) <= 1             # as even as possible
    assert sum(1 for p in ps if p.tfast) == 1                           # exactly one pass holds the low bits


# ---- k_ntt_pass: index maps
def tile_index(tile, x, k, b0, logc, tfast):
    """(tile, x) -> element index i of the load and store loops (numpy arrays or ints)."""
    rows = 1 << k
    lowmask = (1 << b0) - 1
    if tfast:
        t, c = x & (rows - 1), x >> k
    else:
        c, t = x & ((1 << logc) - 1), x >> logc
    u = (tile << logc) + c
    return ((u >> b0) << (b0 + k)) | (t << b0) | (u & lowmask)


def butterfly_twiddle_exponents(tile, q, step, k, b0, logc, L, tfast, dit):
    """e of the butterfly (tile, q) at `step` (0 where the level has no twiddles: pb == 0)."""
    rows = 1 << k
    lb = step if dit else k - 1 - step
    pb = b0 + lb
    lbmask = (1 << lb) - 1
    lowmask = (1 << b0) - 1
    if tfast:
        r, c = q & ((rows >> 1) - 1), q >> (k - 1)
    else:
        c, r = q & ((1 << logc) - 1), q >> logc
    t0 = ((r >> lb) << (lb + 1)) | (r & lbmask)
    if pb == 0:
        return t0 * 0
    u = (tile << logc) + c
    j = ((t0 & lbmask) << b0) | (u & lowmask)
    return j << (L - 1 - pb)


@pytest.mark.parametrize("L", range(1, 23))
def test_index_maps_bijective_and_twiddles_in_table(L):
    n = 1 << L
    for dit in (False, True):
        for p in schedule(L, dit):
            T = 1 << (p.k + p.logc)
            tile = np.repeat(np.arange(p.tiles, dtype=np.int64), T)
            x = np.tile(np.arange(T, dtype=np.int64), p.tiles)
            for tfast in (False, True):
                i = tile_index(tile, x, p.k, p.b0, p.logc, tfast)
                assert i.min() == 0 and i.max() == n - 1
                assert np.unique(i).size == n, f"2^{L} b0={p.b0} k={p.k} tfast={tfast}: load/store map not a bijection"
            tq = np.repeat(np.arange(p.tiles, dtype=np.int64), T // 2)
            q = np.tile(np.arange(T // 2, dtype=np.int64), p.tiles)
            for step in range(p.k):
                e = butterfly_twiddle_exponents(tq, q, step, p.k, p.b0, p.logc, L, p.tfast, dit)
                for tw_sh in {0, 28 - L}:
                    tw_half = ((1 << (L + tw_sh)) >> 1)
                    idx = e << tw_sh
                    assert idx.min() >= 0 and idx.max() < tw_half      # tw[idx] and tw[tw_half - idx] in range


# ---- k_ntt_pass / ntt_device_impl on Python ints
class Args:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def twiddle_table(tw_log):
    """ensure_twiddles: w^e for e <= N_table / 2 (one entry more than N/2: w^(N/2) = -1)."""
    half = (1 << tw_log) >> 1
    w = root(tw_log)
    out = [1] * (half + 1)
    for e in range(1, half + 1):
        out[e] = out[e - 1] * w % R
    return out


def geometric(count, first, ratio):
    """build_geometric: t[i] = first * ratio^i."""
    out = [first % R] * count
    for i in range(1, count):
        out[i] = out[i - 1] * ratio % R
    return out


def k_ntt_pass(vecs, A, DIT, TFAST, INV):
    k, L, b0, logc = A.k, A.L, A.b0, A.logc
    rows = 1 << k
    T = rows << logc
    lowmask = (1 << b0) - 1
    for y, data in enumerate(vecs):
        post = A.post_vec[y] if (A.post_mode == 2 and A.nvecs) else A.post
        for tile in range(A.tiles):
            sm = [0] * T
            for x in range(T):
                i = tile_index(tile, x, k, b0, logc, TFAST)
                v = data[i]
                if A.pre:
                    v = v * A.pre[bitrev(i, L) if A.pre_bitrev else i] % R
                sm[x] = v
            nbf = T >> 1
            for step in range(k):
                lb = step if DIT else k - 1 - step
                pb = b0 + lb
                lbmask = (1 << lb) - 1
                for q in range(nbf):
                    if TFAST:
                        r, c = q & ((rows >> 1) - 1), q >> (k - 1)
                    else:
                        c, r = q & ((1 << logc) - 1), q >> logc
                    t0 = ((r >> lb) << (lb + 1)) | (r & lbmask)
                    t1 = t0 | (1 << lb)
                    s0 = ((c << k) | t0) if TFAST else ((t0 << logc) | c)
                    s1 = ((c << k) | t1) if TFAST else ((t1 << logc) | c)
                    xv, yv = sm[s0], sm[s1]
                    if pb == 0:
                        sm[s0], sm[s1] = (xv + yv) % R, (xv - yv) % R
                        continue
                    u = (tile << logc) + c
                    j = ((t0 & lbmask) << b0) | (u & lowmask)
                    e = j << (L - 1 - pb)
                    idx = e << A.tw_sh
                    w = A.tw[A.tw_half - idx if INV else idx]
                    if DIT:
                        yv = yv * w % R
                        if not INV:
                            sm[s0], sm[s1] = (xv + yv) % R, (xv - yv) % R
                        else:
                            sm[s0], sm[s1] = (xv - yv) % R, (xv + yv) % R
                    else:
                        sm[s0] = (xv + yv) % R
                        sm[s1] = ((yv - xv) if INV else (xv - yv)) * w % R
            for x in range(T):
                i = tile_index(tile, x, k, b0, logc, TFAST)
                v = sm[x]
                if A.post_mode == 1:
                    v = v * A.post_const % R
                elif A.post_mode == 2:
                    v = v * post[bitrev(i, L) if A.post_bitrev else i] % R
                data[i] = v


class Workspace:
    """NttWorkspace: the tables a context keeps (tw_log only grows)."""

    def __init__(self, tw_log=-1):
        self.tw_log = tw_log
        self.tw = twiddle_table(tw_log) if tw_log >= 0 else None

    def ensure_twiddles(self, L):
        if self.tw_log >= L:
            return
        self.tw_log = L
        self.tw = twiddle_table(L)


def coset_tables(L):
    """ensure_coset: fwd[i] = g^i, inv[i] = g^-i / N."""
    n = 1 << L
    return geometric(n, 1, COSET_GEN), geometric(n, pow(n, -1, R), pow(COSET_GEN, -1, R))


def ntt_device_impl(ws, vecs, L, inverse, coset, dit, fused_post=None, skip_pre=False, vec_list=False):
    """vec_list: the vectors come as a pointer list (NttPassArgs.nvecs > 0), else one buffer of consecutive vectors."""
    ws.ensure_twiddles(L)
    n = 1 << L
    cos_fwd, cos_inv = coset_tables(L) if coset else (None, None)
    A = Args(nvecs=len(vecs) if vec_list else 0, tw=ws.tw, tw_sh=ws.tw_log - L, tw_half=(1 << ws.tw_log) >> 1, L=L,
             post_const=pow(n, -1, R), post_vec=[None] * 3)
    pre = cos_fwd if (coset and not inverse and not skip_pre) else None
    pre_bitrev = 1 if dit else 0
    post_mode, post = 0, None
    if inverse:
        if coset:
            post_mode, post = 2, cos_inv
        else:
            post_mode = 1
    if fused_post:
        assert inverse and not coset and vec_list
        post_mode = 2
        A.post_vec = list(fused_post)
    post_bitrev = 0 if dit else 1
    if L == 0:
        return
    ps = schedule(L, dit)
    for p_i, p in enumerate(ps):
        A.k, A.b0, A.logc, A.tiles = p.k, p.b0, p.logc, p.tiles
        A.pre = pre if p_i == 0 else None
        A.pre_bitrev = pre_bitrev
        A.post_mode = post_mode if p_i == len(ps) - 1 else 0
        A.post = post
        A.post_bitrev = post_bitrev
        k_ntt_pass(vecs, A, dit, p.tfast, inverse)


@pytest.mark.parametrize("tw_sh", [0, 2])
@pytest.mark.parametrize("L", range(0, 11))
def test_pass_model_equals_domain(L, tw_sh):
    rng = random.Random(31 * L + tw_sh)
    n = 1 << L
    a = [rng.randrange(R) for _ in range(n)]
    ws = Workspace(L + tw_sh)                  # a table built for a larger size: read with stride 2^tw_sh
    d = ont.Domain(n)
    for inverse in (False, True):
        for coset in (False, True):
            for dit in (False, True):
                got = list(a)
                ntt_device_impl(ws, [got], L, inverse, coset, dit)
                exp = list(a)
                (d.fft_inverse if inverse else d.fft)(exp, ont.DIT if dit else ont.DIF, coset=coset)
                assert got == exp, f"2^{L} tw_sh={tw_sh} inverse={inverse} coset={coset} dit={dit}"


# ---- compute_h_dist_phase over G = 2^g devices
def twiddle(tw, e, sh, half, inverse):
    idx = e << sh
    if not inverse or idx == 0:
        return tw[idx]
    return -tw[half - idx] % R


def cross_levels(x, GLOG, DIT, o, tw, tw_sh, tw_half, L, inverse):
    G = 1 << GLOG
    M = 1 << (L - GLOG)
    for step in range(GLOG):
        q = GLOG - 1 - step if DIT else step
        bit = GLOG - 1 - q
        for d0 in range(G):
            if d0 & (1 << bit):
                continue
            d1 = d0 | (1 << bit)
            j = (d0 & ((1 << bit) - 1)) * M + o
            e = j << q
            a, b = x[d0], x[d1]
            if e == 0 and not inverse:
                x[d0], x[d1] = (a + b) % R, (a - b) % R
                continue
            w = twiddle(tw, e, tw_sh, tw_half, inverse)
            if DIT:
                b = b * w % R
                x[d0], x[d1] = (a + b) % R, (a - b) % R
            else:
                x[d0], x[d1] = (a + b) % R, (a - b) * w % R


def cross_args(ws, L):
    ws.ensure_twiddles(L)
    return ws.tw, ws.tw_log - L, (1 << ws.tw_log) >> 1


def k_ntt_cross(buf, GLOG, DIT, me, L, ws, inverse):
    tw, tw_sh, tw_half = cross_args(ws, L)
    G = 1 << GLOG
    share = (1 << (L - GLOG)) >> GLOG
    for vec in buf:
        for t in range(share):
            o = me * share + t
            x = [vec[d][o] for d in range(G)]
            cross_levels(x, GLOG, DIT, o, tw, tw_sh, tw_half, L, inverse)
            for d in range(G):
                vec[d][o] = x[d]


def k_ntt_cross_h(buf, GLOG, me, L, ws):
    tw, tw_sh, tw_half = cross_args(ws, L)
    G = 1 << GLOG
    share = (1 << (L - GLOG)) >> GLOG
    for t in range(share):
        o = me * share + t
        acc = [buf[0][d][o] for d in range(G)]
        cross_levels(acc, GLOG, True, o, tw, tw_sh, tw_half, L, False)
        x = [buf[1][d][o] for d in range(G)]
        cross_levels(x, GLOG, True, o, tw, tw_sh, tw_half, L, False)
        acc = [u * v % R for u, v in zip(acc, x)]
        x = [buf[2][d][o] for d in range(G)]
        cross_levels(x, GLOG, True, o, tw, tw_sh, tw_half, L, False)
        acc = [(u - v) % R for u, v in zip(acc, x)]
        cross_levels(acc, GLOG, False, o, tw, tw_sh, tw_half, L, True)
        for d in range(G):
            buf[0][d][o] = acc[d]


def ensure_dist_tables(L, g, me):
    """t1[k] = g^(k G + br) / N, t2 = t1 / (g^N - 1), ti[k] = g^-(k G + br) / N, br = bitrev_g(me)."""
    M = 1 << (L - g)
    G = 1 << g
    n_inv = pow(1 << L, -1, R)
    br = bitrev(me, g)
    den_inv = pow((pow(COSET_GEN, 1 << L, R) - 1) % R, -1, R)
    first = n_inv * pow(COSET_GEN, br, R) % R
    gi = pow(COSET_GEN, -1, R)
    t1 = geometric(M, first, pow(COSET_GEN, G, R))
    t2 = geometric(M, first * den_inv, pow(COSET_GEN, G, R))
    ti = geometric(M, n_inv * pow(gi, br, R), pow(gi, G, R))
    return t1 + t2 + ti


def compute_h_dist_phase(buf, wss, g, me, L, phase):
    Lm = L - g
    M = 1 << Lm
    if phase in (0, 2):
        if phase == 0:
            k_ntt_cross(buf, g, False, me, L, wss[me], True)
        else:
            k_ntt_cross_h(buf, g, me, L, wss[me])
        return
    wss[me].ensure_twiddles(L)              # the size-N table also serves the size-M passes (stride 2^g)
    t = ensure_dist_tables(L, g, me)
    if phase == 1:
        v = [buf[0][me], buf[1][me], buf[2][me]]
        post = [t[M:2 * M], t[:M], t[M:2 * M]]  # a and c carry 1 / (g^N - 1)
        ntt_device_impl(wss[me], v, Lm, True, False, False, fused_post=post, vec_list=True)
        ntt_device_impl(wss[me], v, Lm, False, True, True, skip_pre=True, vec_list=True)
        return
    ntt_device_impl(wss[me], [buf[0][me]], Lm, True, False, False, fused_post=[t[2 * M:3 * M]], vec_list=True)


def compute_h_dist(a, b, c, L, g, extra_tw=0):
    G = 1 << g
    M = (1 << L) >> g
    buf = [[list(v[d * M:(d + 1) * M]) for d in range(G)] for v in (a, b, c)]
    wss = [Workspace(L + extra_tw) for _ in range(G)]
    for phase in range(4):
        for me in range(G):                 # every device runs the phase; barriers in between
            compute_h_dist_phase(buf, wss, g, me, L, phase)
    return [x for d in range(G) for x in buf[0][d]]


@pytest.mark.parametrize("g,L", [(g, L) for g in (1, 2, 3) for L in range(2 * g + 1, 13)])
def test_dist_compute_h_model_equals_oracle(g, L):
    rng = random.Random(1000 * g + L)
    n = 1 << L
    n_c = [n, n - 1, n // 2 + 1, 1][L % 4]
    a = [rng.randrange(R) for _ in range(n_c)]
    b = [rng.randrange(R) for _ in range(n_c)]
    c = [rng.randrange(R) for _ in range(n_c)]
    pad = lambda v: v + [0] * (n - len(v))     # noqa: E731
    want = ont.compute_h(a, b, c, ont.Domain(n))
    assert compute_h_dist(pad(a), pad(b), pad(c), L, g) == want
    if L <= 8:                                 # a context whose twiddle table is larger than 2^L
        assert compute_h_dist(pad(a), pad(b), pad(c), L, g, extra_tw=3) == want

