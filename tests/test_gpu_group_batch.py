"""GPU: batch Groth16 prove over a device group (b200g16_bases_copy, b200g16_group_pk_replicate,
b200g16_group_prove_batch, groth16.GroupProvingKey / GroupBatchProve).  Every field of every proof must equal the
closed form over a known-discrete-log key (oracle/synth.py) and one-ctx b200g16_prove_batch with the same r, s; real
circuits (oracle.groth16 synthetic_r1cs, with and without a BSB22 commitment) must give BatchProve's proofs, pass
Verify and BatchVerify.  A group may name a device more than once, so the split, the replication rule and the
per-member gather lists run on a single-GPU box too; with >= 2 GPUs the same tests also run on distinct devices
(where the vectors really are copied device to device)."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import cport, synth
from oracle import groth16 as og
from oracle.bn254 import R
from oracle.synth import KnownDlogKey, check_proof, rand_fr, whir_mix

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -2, -4
N_GPUS = torch.cuda.device_count()


def _device_lists():
    out = [[0], [0, 0], [0, 0, 0], [0] * 4, [0] * 8]
    if N_GPUS >= 2:
        out.append([0, 1])
    if N_GPUS >= 4:
        out.append([0, 1, 2, 3])
    if N_GPUS >= 8:
        out.append(list(range(8)))
    return out


DEVICE_LISTS = _device_lists()
dev_id = lambda d: "dev" + "_".join(map(str, d))
rs = np.random.Generator(np.random.PCG64(20261023))


def inputs(key, k, ncons):
    wires = np.stack([whir_mix(rs, key.N) for _ in range(k)])
    a, b, c = [np.stack([rand_fr(rs, ncons) for _ in range(k)]) for _ in range(3)]
    r, s = rand_fr(rs, k), rand_fr(rs, k)
    return wires, a, b, c, r, s


def ranges(k, n):
    base, rem = divmod(k, n)
    out, lo = [], 0
    for i in range(n):
        hi = lo + base + (1 if i < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def check_batch(ctx, g, gpk, key, k, ncons=None, closed_form=True):
    """One group batch of k proofs: closed forms, one-ctx prove_batch, the members' timings."""
    ncons = key.N - 1 - 5 * k if ncons is None else ncons
    wires, a, b, c, r, s = inputs(key, k, ncons)
    got = g.prove_batch(gpk, wires, a, b, c, r, s)
    assert len(got) == k
    for i, (lo, hi) in enumerate(ranges(k, len(g))):
        if hi > lo:
            assert len(g.ctx(i).last_timings()) == 8, f"member {i}"
    one = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    for j in range(k):
        for f in one[j]:
            assert np.array_equal(got[j][f], one[j][f]), f"proof {j} field {f}"
        if closed_form:
            exp, _ = key.expected(wires[j], a[j], b[j], c[j], r[j], s[j])
            assert check_proof(got[j], exp) == [], f"proof {j}"
    return got


@pytest.fixture(scope="module")
def key16(ctx):
    k = KnownDlogKey(ctx, 16, seed=1616, precompute=True)
    yield k
    k.free()


# ---- b200g16_bases_copy
@pytest.mark.parametrize("n", [1, 1000, (1 << 16) + 3])
@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("group", [1, 2])
def test_bases_copy(ctx, group, table, n):
    gen = synth.G1 if group == 1 else synth.G2
    ks = rand_fr(rs, n)
    sc = whir_mix(rs, n)
    closed = (cport.g1_gen_mul if group == 1 else cport.g2_gen_mul)(cport.fr_dot(ks, sc))
    src = ctx.fixed_base_mul(gen, ks, group=group, resident=True)
    if table:
        src.precompute(0)
    pts = src.download()
    win = src.window()
    assert (win > 0) == table
    want = ctx.msm(src, sc)
    assert np.array_equal(want, closed)
    others = [lib.Context(1)] if N_GPUS >= 2 else []
    try:
        copies = [ctx.bases_copy(src)] + [o.bases_copy(src) for o in others]
        src.free()                                  # the copies do not depend on the source
        for cp in copies:
            assert (cp.group, len(cp)) == (group, n)
            assert cp.window() == win
            assert np.array_equal(cp.download(), pts)
            assert np.array_equal(cp.ctx.msm(cp, sc), closed)
        # a copy of a copy, back onto device 0
        again = ctx.bases_copy(copies[-1])
        copies[-1].free()
        assert np.array_equal(ctx.msm(again, sc), closed)
        assert again.window() == win
        for cp in [again] + copies[:-1]:
            cp.free()
    finally:
        for o in others:
            o.close()


# ---- group batch prove over known-dlog keys
@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=dev_id)
def test_group_batch_2p16_closed_form_and_one_ctx(ctx, key16, devices):
    n = len(devices)
    with lib.Group(devices) as g:
        gpk = g.pk_replicate(key16.handle)
        try:
            for k in sorted({1, max(n - 1, 1), n, n + 1, 3 * n + 2}):
                check_batch(ctx, g, gpk, key16, k)
        finally:
            g.pk_free(gpk)


@pytest.mark.parametrize("devices,ks", [([0, 0], [35]), ([0, 0, 0], [1, 2, 3, 4, 11])]
                         + ([([0, 1], [1, 3, 35])] if N_GPUS >= 2 else []), ids=lambda v: str(v))
def test_group_batch_2p20(ctx, devices, ks):
    """2^20 with window tables; [0, 0] with k = 35 gives each member more proofs than one sub-batch holds (16 at
    2^20 with a c = 20 table), so sub-batching runs inside a device."""
    key = KnownDlogKey(ctx, 20, seed=2020, precompute=True)
    try:
        with lib.Group(devices) as g:
            gpk = g.pk_replicate(key.handle)
            try:
                for k in ks:
                    check_batch(ctx, g, gpk, key, k, ncons=key.N - 3)
            finally:
                g.pk_free(gpk)
    finally:
        key.free()


# ---- key sources and lifetime
def _host_arrays(key):
    return {n: key.vec[n].download() for n in ("a", "b", "k", "z", "b2")}


@pytest.mark.parametrize("devices", [[0, 0, 0]] + ([[1, 0]] if N_GPUS >= 2 else []), ids=dev_id)
def test_host_uploaded_source_and_freeing_the_replica(ctx, key16, devices):
    h = _host_arrays(key16)
    p = key16.points
    src = ctx.pk_upload(16, key16.N, h["a"], h["b"], h["k"], h["z"], h["b2"], p["alpha"], p["beta"], p["delta"],
                        p["beta2"], p["delta2"], key16.zeros, key16.zeros, key16.k_skip, precompute=True)
    try:
        wires, a, b, c, r, s = inputs(key16, 7, key16.N - 1)
        with lib.Group(devices) as g:
            gpk = g.pk_replicate(src)
            got = g.prove_batch(gpk, wires, a, b, c, r, s)
            g.pk_free(gpk)
        after = ctx.prove_batch(src, wires, a, b, c, r, s)           # the source outlives its replica unchanged
        for j in range(7):
            exp, _ = key16.expected(wires[j], a[j], b[j], c[j], r[j], s[j])
            assert check_proof(got[j], exp) == [], f"proof {j}"
            for f in got[j]:
                assert np.array_equal(after[j][f], got[j][f])
    finally:
        ctx.pk_free(src)


def test_alternating_key_sizes_on_one_group(ctx, key16):
    key18 = KnownDlogKey(ctx, 18, seed=1818, precompute=False)
    try:
        with lib.Group([0, 0, 0]) as g:
            g16k, g18k = g.pk_replicate(key16.handle), g.pk_replicate(key18.handle)
            try:
                for key, gpk, k in ((key16, g16k, 4), (key18, g18k, 5), (key16, g16k, 2), (key18, g18k, 3)):
                    check_batch(ctx, g, gpk, key, k)
            finally:
                g.pk_free(g16k)
                g.pk_free(g18k)
    finally:
        key18.free()


def test_sharded_prove_interleaved_with_replicated_batch(ctx, key16):
    h = _host_arrays(key16)
    p = key16.points
    wires, a, b, c, r, s = inputs(key16, 5, key16.N - 11)
    with lib.Group([0, 0, 0, 0]) as g:
        sharded = g.pk_upload(16, key16.N, h["a"], h["b"], h["k"], h["z"], h["b2"], p["alpha"], p["beta"], p["delta"],
                              p["beta2"], p["delta2"], key16.zeros, key16.zeros, key16.k_skip, precompute=True)
        rep = g.pk_replicate(key16.handle)
        try:
            alone_single, _ = g.prove(sharded, wires[0], a[0], b[0], c[0], r[0], s[0])
            alone_batch = g.prove_batch(rep, wires, a, b, c, r, s)
            for it in range(2):
                batch = g.prove_batch(rep, wires, a, b, c, r, s)
                single, _ = g.prove(sharded, wires[0], a[0], b[0], c[0], r[0], s[0])
                for f in single:
                    assert np.array_equal(single[f], alone_single[f]), f"pass {it} single {f}"
                for j in range(5):
                    for f in batch[j]:
                        assert np.array_equal(batch[j][f], alone_batch[j][f]), f"pass {it} proof {j} {f}"
            exp, _ = key16.expected(wires[0], a[0], b[0], c[0], r[0], s[0])
            assert check_proof(alone_single, exp) == []
            assert check_proof(alone_batch[0], exp) == []
        finally:
            g.pk_free(sharded)
            g.pk_free(rep)


# ---- real circuits through GroupProvingKey / GroupBatchProve
def _another_witness(r1cs, w0, nb_public, rng):
    w = list(w0)
    for i in range(1, nb_public):
        w[i] = rng.randrange(256)
    for i in range(nb_public, nb_public + 4):
        w[i] = rng.randrange(R)
    for L, Rr, O in r1cs.constraints:
        w[O[0][0]] = og.lc_eval(L, w) * og.lc_eval(Rr, w) % R
    return w


@pytest.mark.parametrize("devices", [[0, 0, 0]] + ([[0, 1]] if N_GPUS >= 2 else []), ids=dev_id)
@pytest.mark.parametrize("source", ["host", "device_setup"])
@pytest.mark.parametrize("nb_constraints,nb_public,with_commitment", [(24, 3, False), (100, 5, True)])
def test_group_batch_prove_real_circuits(ctx, nb_constraints, nb_public, with_commitment, source, devices):
    rng = random.Random(nb_constraints * 37 + len(devices))
    r1cs, w0 = og.synthetic_r1cs(nb_constraints, nb_public, rng, with_commitment=with_commitment)
    tw = g16.ToxicWaste(*[rng.randrange(1, R) for _ in range(5)], sigma=rng.randrange(1, R))
    if source == "host":
        pk, vk = g16.Setup(ctx, r1cs, tw)
    else:
        pk, vk = g16.DeviceSetup(ctx, r1cs, tw, precompute=True)
    k = 5
    ws = [list(w0)] + [_another_witness(r1cs, w0, nb_public, rng) for _ in range(k - 1)]

    def resolve(wit):
        L, Rr, O = r1cs.constraints[-1]
        wit[O[0][0]] = og.lc_eval(L, wit) * og.lc_eval(Rr, wit) % R
    res = resolve if with_commitment else None
    rr = [rng.randrange(R) for _ in range(k)]
    ss = [rng.randrange(R) for _ in range(k)]
    try:
        with lib.Group(devices) as g:
            gpk = g16.GroupProvingKey(g, pk, ctx=ctx)
            try:
                proofs = g16.GroupBatchProve(g, r1cs, gpk, ws, rs=rr, ss=ss, resolve=res)
            finally:
                gpk.free()
        want = g16.BatchProve(ctx, r1cs, pk, ws, rs=rr, ss=ss, resolve=res)
        pubs = []
        for p, q in zip(proofs, want):
            assert np.array_equal(p.Ar, q.Ar) and np.array_equal(p.Bs, q.Bs) and np.array_equal(p.Krs, q.Krs)
            if with_commitment:
                assert np.array_equal(p.Commitments[0], q.Commitments[0])
                assert np.array_equal(p.CommitmentPok, q.CommitmentPok)
            pub = p.debug["witness"][1:r1cs.nb_public]
            g16.Verify(ctx, p, vk, pub)
            pubs.append(pub)
        assert all(g16.BatchVerify(ctx, proofs, vk, pubs))
    finally:
        pk.free()


# ---- errors
def test_errors_leave_every_ctx_usable(ctx, key16):
    L = lib.load()
    N = key16.N
    P = lambda x: x.ctypes.data_as(C.c_void_p)
    wires, a, b, c, r, s = inputs(key16, 3, N - 1)
    out = (lib.ProofOut * 3)()
    h = _host_arrays(key16)
    p = key16.points
    with lib.Group([0, 0]) as g, lib.Group([0, 0]) as other:
        gpk = g.pk_replicate(key16.handle)
        foreign = other.pk_replicate(key16.handle)
        sharded = g.pk_upload(16, N, h["a"], h["b"], h["k"], h["z"], h["b2"], p["alpha"], p["beta"], p["delta"],
                              p["beta2"], p["delta2"], key16.zeros, key16.zeros, key16.k_skip)
        shard = KnownDlogKey(ctx, 12, seed=9, precompute=False,
                             lo_hi={"a": (0, 100), "b": (0, 100), "k": (0, 100), "z": (0, 100)})
        wz, az = whir_mix(rs, 1 << 12), rand_fr(rs, 1 << 12)

        def usable():
            check_batch(ctx, g, gpk, key16, 3, closed_form=False)
            for i in range(len(g)):
                single, _ = g.ctx(i).prove(key16.handle, wires[1], a[1], b[1], c[1], r[1], s[1])
                exp, _ = key16.expected(wires[1], a[1], b[1], c[1], r[1], s[1])
                assert check_proof(single, exp) == [], f"member {i}"

        gb = lambda pk, k=3, w=P(wires), nw=N, nc=N - 1, rr=P(r): L.b200g16_group_prove_batch(
            g.h, pk, k, w, nw, P(a), P(b), P(c), nc, rr, P(s), out)
        try:
            refusals = [
                ("null wires", lambda: gb(gpk, w=None), ERR_ARG),
                ("null r", lambda: gb(gpk, rr=None), ERR_ARG),
                ("n_wires", lambda: gb(gpk, nw=N - 1), ERR_ARG),
                ("n_constraints", lambda: gb(gpk, nc=N + 1), ERR_ARG),
                ("overflow", lambda: gb(gpk, k=1 << 62), ERR_ARG),
                ("sharded key", lambda: gb(sharded), ERR_ARG),
                ("another group", lambda: gb(foreign), ERR_STATE),
                ("replicated key to group_prove", lambda: L.b200g16_group_prove(
                    g.h, gpk, P(wires), N, P(a), P(b), P(c), N - 1, P(r), P(s), out, None), ERR_ARG),
                ("partial source", lambda: L.b200g16_group_pk_replicate(g.h, shard.handle, C.byref(lib._vp())),
                 ERR_ARG),
                ("null source", lambda: L.b200g16_group_pk_replicate(g.h, None, C.byref(lib._vp())), ERR_ARG),
                ("null copy source", lambda: L.b200g16_bases_copy(ctx.h, None, C.byref(lib._vp())), ERR_ARG),
            ]
            for what, call, code in refusals:
                assert call() == code, what
                assert lib.load().b200g16_last_error().decode(), what
                usable()
            # k = 0: nothing is written
            marker = (lib.ProofOut * 1)()
            C.memset(C.addressof(marker), 0x5A, C.sizeof(marker))
            before = bytes(marker)
            assert L.b200g16_group_prove_batch(g.h, gpk, 0, None, N, None, None, None, 0, None, None, marker) == 0
            assert bytes(marker) == before
            # one member refuses (a prove is open on its ctx): the error names its device, the other members finish,
            # and every ctx stays usable
            dw = torch.from_numpy(wires[0].view(np.int64)).cuda()
            g.ctx(1).prove_begin_dev(key16.handle, dw.data_ptr())
            assert gb(gpk) == ERR_STATE
            assert "device 0" in lib.load().b200g16_last_error().decode()
            hz = torch.zeros((N, 4), dtype=torch.int64, device="cuda")
            g.ctx(1).prove_end_dev(key16.handle, hz.data_ptr(), r[0], s[0])
            usable()
        finally:
            shard.free()
            g.pk_free(sharded)
            other.pk_free(foreign)
            g.pk_free(gpk)
