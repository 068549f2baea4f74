"""GPU: batch Groth16 prove (b200g16_prove_batch / _dev, groth16.BatchProve).  Every field of every proof must equal
the closed form over a known-discrete-log key (oracle/synth.py) and the single prove with the same r, s; the h rows
the device path leaves behind must equal the C restatement of computeH.  Real circuits (oracle.groth16
synthetic_r1cs, with and without a BSB22 commitment) go through Setup and BatchProve and must equal Prove, pass Verify
and pass BatchVerify.  Errors leave the context usable."""
import ctypes as C
import random

import numpy as np
import pytest

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import cport
from oracle import groth16 as og
from oracle.bn254 import R
from oracle.synth import KnownDlogKey, check_proof, rand_fr, whir_mix

pytestmark = pytest.mark.gpu

rs = np.random.Generator(np.random.PCG64(20261022))


def inputs(key, k, ncons):
    wires = np.stack([whir_mix(rs, key.N) for _ in range(k)])
    a, b, c = [np.stack([rand_fr(rs, ncons) for _ in range(k)]) for _ in range(3)]
    r, s = rand_fr(rs, k), rand_fr(rs, k)
    return wires, a, b, c, r, s


@pytest.fixture(scope="module")
def keys(ctx):
    out = {16: KnownDlogKey(ctx, 16, seed=1616), 20: KnownDlogKey(ctx, 20, seed=2020)}
    yield out
    for v in out.values():
        v.free()


@pytest.mark.parametrize("log2n,k", [(16, 1), (16, 3), (16, 8), (16, 17), (20, 3), (20, 17)])
def test_host_path_closed_form_and_single_prove(ctx, keys, log2n, k):
    key = keys[log2n]
    ncons = key.N - 1 - 7 * k                     # ragged: zero padding up to N
    wires, a, b, c, r, s = inputs(key, k, ncons)
    got = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    assert len(got) == k
    assert len(ctx.last_timings()) == 8          # a single prove's phases, summed over the sub-batches
    for j in range(k):
        exp, _ = key.expected(wires[j], a[j], b[j], c[j], r[j], s[j])
        assert check_proof(got[j], exp) == [], f"proof {j}"
    for j in sorted({0, k - 1}):
        single, _ = ctx.prove(key.handle, wires[j], a[j], b[j], c[j], r[j], s[j])
        for f in single:
            assert np.array_equal(got[j][f], single[f]), f"proof {j} field {f}"


@pytest.mark.parametrize("log2n,k", [(16, 1), (16, 8), (16, 17), (20, 17)])
def test_device_path_and_h(ctx, keys, log2n, k):
    import torch
    key = keys[log2n]
    N = key.N
    ncons = N - 3
    wires, a, b, c, r, s = inputs(key, k, ncons)
    pad = lambda x: np.concatenate([x, np.zeros((k, N - ncons, 4), dtype=np.uint64)], axis=1)
    dw = torch.from_numpy(wires.reshape(-1, 4).view(np.int64)).cuda()
    da, db, dc = [torch.from_numpy(pad(x).reshape(-1, 4).view(np.int64)).cuda() for x in (a, b, c)]
    got = ctx.prove_batch_dev(key.handle, k, dw.data_ptr(), da.data_ptr(), db.data_ptr(), dc.data_ptr(), r, s)
    hs = da.cpu().numpy().view(np.uint64).reshape(k, N, 4)
    for j in range(k):
        exp, h = key.expected(wires[j], a[j], b[j], c[j], r[j], s[j])
        assert check_proof(got[j], exp) == [], f"proof {j}"
        assert np.array_equal(hs[j], h), f"h of proof {j}"
    host = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    for j in range(k):
        for f in host[j]:
            assert np.array_equal(got[j][f], host[j][f])


def _another_witness(r1cs, w0, nb_public, rng):
    """A second satisfying assignment of the same synthetic circuit: new public and seed wires, every constraint's
    output wire re-solved in order (the commitment wire is filled later, by BatchProve)."""
    w = list(w0)
    for i in range(1, nb_public):
        w[i] = rng.randrange(256)
    for i in range(nb_public, nb_public + 4):
        w[i] = rng.randrange(R)
    for L, Rr, O in r1cs.constraints:
        w[O[0][0]] = og.lc_eval(L, w) * og.lc_eval(Rr, w) % R
    return w


@pytest.mark.parametrize("nb_constraints,nb_public,with_commitment", [(24, 3, False), (100, 5, True), (257, 9, False)])
@pytest.mark.parametrize("k", [1, 4])
def test_batch_prove_real_circuits(ctx, nb_constraints, nb_public, with_commitment, k):
    rng = random.Random(nb_constraints * 31 + k)
    r1cs, w0 = og.synthetic_r1cs(nb_constraints, nb_public, rng, with_commitment=with_commitment)
    tw = og.ToxicWaste(*[rng.randrange(1, R) for _ in range(5)], sigma=rng.randrange(1, R))
    pk, vk = g16.Setup(ctx, r1cs, g16.ToxicWaste(tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma))
    try:
        ws = [list(w0)] + [_another_witness(r1cs, w0, nb_public, rng) for _ in range(k - 1)]

        def resolve(wit):
            L, Rr, O = r1cs.constraints[-1]
            wit[O[0][0]] = og.lc_eval(L, wit) * og.lc_eval(Rr, wit) % R
        rr = [rng.randrange(R) for _ in range(k)]
        ss = [rng.randrange(R) for _ in range(k)]
        res = resolve if with_commitment else None
        proofs = g16.BatchProve(ctx, r1cs, pk, ws, rs=rr, ss=ss, resolve=res)
        pubs = []
        for j, p in enumerate(proofs):
            single = g16.Prove(ctx, r1cs, pk, ws[j], r=rr[j], s=ss[j], resolve=res)
            assert np.array_equal(p.Ar, single.Ar) and np.array_equal(p.Bs, single.Bs) and np.array_equal(p.Krs, single.Krs)
            if with_commitment:
                assert np.array_equal(p.Commitments[0], single.Commitments[0])
                assert np.array_equal(p.CommitmentPok, single.CommitmentPok)
            pub = p.debug["witness"][1:r1cs.nb_public]
            g16.Verify(ctx, p, vk, pub)
            pubs.append(pub)
        assert all(g16.BatchVerify(ctx, proofs, vk, pubs))
    finally:
        pk.free()


def test_batch_single_and_msm_back_to_back(ctx, keys):
    key = keys[16]
    wires, a, b, c, r, s = inputs(key, 5, key.N - 1)
    got = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    single, _ = ctx.prove(key.handle, wires[2], a[2], b[2], c[2], r[2], s[2])
    sc = np.stack([rand_fr(rs, 4000) for _ in range(3)])
    mb = ctx.msm_batch(key.vec["a"], sc)
    again = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    for f in single:
        assert np.array_equal(got[2][f], single[f])
    for j in range(5):
        for f in got[j]:
            assert np.array_equal(got[j][f], again[j][f])
    for j in range(3):
        assert np.array_equal(mb[j], cport.g1_gen_mul(cport.fr_dot(key.k["a"][:4000], sc[j])))


def test_errors_leave_the_ctx_usable(ctx, keys):
    import torch
    L = lib.load()
    key = keys[16]
    N = key.N
    wires, a, b, c, r, s = inputs(key, 2, N - 1)
    out = (lib.ProofOut * 2)()
    P = lambda x: x.ctypes.data_as(C.c_void_p)
    ERR_ARG, ERR_STATE = -2, -4
    assert L.b200g16_prove_batch(ctx.h, key.handle, 2, P(wires), N - 1, P(a), P(b), P(c), N - 1, P(r), P(s), out) == ERR_ARG
    assert L.b200g16_prove_batch(ctx.h, key.handle, 2, P(wires), N, P(a), P(b), P(c), N + 1, P(r), P(s), out) == ERR_ARG
    assert L.b200g16_prove_batch(ctx.h, key.handle, 2, None, N, P(a), P(b), P(c), N - 1, P(r), P(s), out) == ERR_ARG
    assert L.b200g16_prove_batch(ctx.h, key.handle, 1 << 62, P(wires), N, P(a), P(b), P(c), N - 1, P(r), P(s), out) == ERR_ARG
    assert L.b200g16_prove_batch(ctx.h, key.handle, 0, None, N, None, None, None, 0, None, None, None) == 0
    shard = KnownDlogKey(ctx, 12, seed=9, precompute=False, lo_hi={"a": (0, 100), "b": (0, 100), "k": (0, 100), "z": (0, 100)})
    try:
        wz = whir_mix(rs, shard.N)
        az = rand_fr(rs, shard.N)
        assert L.b200g16_prove_batch(ctx.h, shard.handle, 1, P(wz), shard.N, P(az), P(az), P(az), shard.N, P(r), P(s),
                                     out) == ERR_ARG
    finally:
        shard.free()
    dw = torch.from_numpy(wires[0].view(np.int64)).cuda()
    ctx.prove_begin_dev(key.handle, dw.data_ptr())
    assert L.b200g16_prove_batch(ctx.h, key.handle, 2, P(wires), N, P(a), P(b), P(c), N - 1, P(r), P(s), out) == ERR_STATE
    h = torch.zeros((N, 4), dtype=torch.int64, device="cuda")
    ctx.prove_end_dev(key.handle, h.data_ptr(), r[0], s[0])
    got = ctx.prove_batch(key.handle, wires, a, b, c, r, s)
    for j in range(2):
        exp, _ = key.expected(wires[j], a[j], b[j], c[j], r[j], s[j])
        assert check_proof(got[j], exp) == []
