"""Groth16 setup on the GPU (b200g16_setup / _setup_wire_polys, groth16.DeviceSetup) against the C restatement of
gnark's setupABC, the host-loop groth16.Setup and the python oracle: same scalars, same points, same key bytes, same
proofs."""
import random

import numpy as np
import pytest

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import bn254 as bn
from oracle import cport
from oracle import groth16 as og
from oracle import setup_port as sp
from oracle.bn254 import R
from oracle.ntt import bitrev

pytestmark = pytest.mark.gpu

G1 = bn.g1_to_array([bn.G1_GEN])[0]
G2 = bn.g2_to_array([bn.G2_GEN])[0]


def _mont(v):
    return bn.fr_to_mont_array([v % R])[0]


def _ints(a):
    return bn.fr_from_mont_array(np.asarray(a, dtype=np.uint64).reshape(-1, 4))


def _check_wire_polys(ctx, d, seed):
    tau = _mont(random.Random(seed).randrange(2, R))
    got = ctx.setup_wire_polys(d, tau)
    exp = sp.setup_abc(d, tau)
    for k in range(3):
        assert np.array_equal(got[k], exp[k]), "ABC"[k]
    return got


@pytest.mark.parametrize("m", [1, 2, 3, 64, 65, 1 << 16, 1 << 20])
def test_wire_polys_match_c_oracle(ctx, m):
    _check_wire_polys(ctx, sp.synthetic_csr(m, m), m)
    assert len(ctx.last_timings()) == 5


@pytest.mark.parametrize("shape", ["stress", "hot_wire", "edges"])
def test_wire_polys_stress_shapes(ctx, shape):
    if shape == "stress":      # a 2^16-term row, empty O rows, repeated wires, zero coefficients, unused wires
        d = sp.synthetic_csr(1 << 17, 3, stress=True, unused_wires=1000)
    elif shape == "hot_wire":  # wire 1 in all 2^20 L rows, wire 0 in ~30% of the R rows
        d = sp.synthetic_csr(1 << 20, 4, hot_wire_rows=True)
    else:                      # a handful of rows, several empty, over many unused wires
        d = sp.synthetic_csr(5, 5, n_inputs=3, stress=True, unused_wires=300)
        d["l_row"] = np.array([0, 0, 0, d["l_row"][1], d["l_row"][1], d["l_row"][1]], dtype=np.uint64)
    got = _check_wire_polys(ctx, d, 77)
    if shape == "stress":
        assert not got[0][-1000:].any()


CIRCUITS = [(1, 1, False), (7, 2, False), (24, 3, False), (24, 3, True), (100, 5, True), (257, 9, False)]


def _case(nb_constraints, nb_public, with_commitment):
    rng = random.Random(nb_constraints * 7 + nb_public)
    r1cs, w = og.synthetic_r1cs(nb_constraints, nb_public, rng, with_commitment=with_commitment)
    tw = og.ToxicWaste(*[rng.randrange(1, R) for _ in range(5)], sigma=rng.randrange(1, R))
    return r1cs, w, tw, rng


def _resolve(r1cs):
    def f(wit):
        L, Rr, O = r1cs.constraints[-1]
        wit[O[0][0]] = og.lc_eval(L, wit) * og.lc_eval(Rr, wit) % R
    return f if r1cs.commitment_wire >= 0 else None


def _host(v):
    return v.download() if hasattr(v, "download") else np.asarray(v, dtype=np.uint64)


@pytest.mark.parametrize("nb_constraints,nb_public,with_commitment", CIRCUITS)
def test_device_setup_equals_setup_and_oracle(ctx, nb_constraints, nb_public, with_commitment):
    r1cs, w, tw, rng = _case(nb_constraints, nb_public, with_commitment)
    gtw = g16.ToxicWaste(tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma)
    ref_pk, ref_vk = g16.Setup(ctx, r1cs, gtw)
    pk, vk = g16.DeviceSetup(ctx, r1cs, gtw)
    try:
        assert pk.log2_domain == ref_pk.log2_domain
        for name in ("G1_A", "G1_B", "G1_Z", "G1_K", "G2_B", "G1_Alpha", "G1_Beta", "G1_Delta", "G2_Beta", "G2_Delta"):
            assert np.array_equal(_host(getattr(pk, name)).reshape(-1), _host(getattr(ref_pk, name)).reshape(-1)), name
        for name in ("InfinityA", "InfinityB", "k_skip"):
            assert np.array_equal(getattr(pk, name), getattr(ref_pk, name)), name
        for name in ("G1_Alpha", "G1_K", "G2_Beta", "G2_Gamma", "G2_Delta", "G1_Beta", "G1_Delta"):
            assert np.array_equal(np.asarray(getattr(vk, name)).reshape(-1), np.asarray(getattr(ref_vk, name)).reshape(-1)), name
        assert vk.has_commitment == ref_vk.has_commitment
        if with_commitment:
            ck, rck = pk.CommitmentKeys[0], ref_pk.CommitmentKeys[0]
            assert np.array_equal(_host(ck.Basis), rck.Basis) and np.array_equal(_host(ck.BasisExpSigma), rck.BasisExpSigma)
            assert np.array_equal(vk.PedersenG, ref_vk.PedersenG)
            assert np.array_equal(vk.PedersenGSigmaNeg, ref_vk.PedersenGSigmaNeg)
            assert vk.PublicAndCommitmentCommitted == ref_vk.PublicAndCommitmentCommitted
        assert g16.pk_write_to(ctx, pk) == g16.pk_write_to(ctx, ref_pk)
        assert g16.vk_write_to(ctx, vk) == g16.vk_write_to(ctx, ref_vk)
        # the python oracle's key (independent group arithmetic)
        opk, ovk = og.setup(r1cs, tw)
        assert np.array_equal(_host(pk.G1_A), bn.g1_to_array(opk.A)) and np.array_equal(_host(pk.G2_B), bn.g2_to_array(opk.B2))
        assert np.array_equal(_host(pk.G1_K), bn.g1_to_array(opk.K)) and np.array_equal(_host(pk.G1_Z), bn.g1_to_array(opk.Z))
        assert np.array_equal(vk.G1_K, bn.g1_to_array(ovk.K))
        assert list(pk.InfinityA.astype(bool)) == opk.infinity_a and list(pk.InfinityB.astype(bool)) == opk.infinity_b
        if with_commitment:
            assert np.array_equal(_host(pk.CommitmentKeys[0].Basis), bn.g1_to_array(opk.ped_basis))
            assert np.array_equal(vk.PedersenGSigmaNeg, bn.g2_to_array([ovk.ped_g_sigma_neg])[0])

        # proofs with the two keys, same r, s
        rs_ = [rng.randrange(R) for _ in range(4)]
        res = _resolve(r1cs)
        p_dev = g16.Prove(ctx, r1cs, pk, w, r=rs_[0], s=rs_[1], resolve=res, want_h=True)
        p_ref = g16.Prove(ctx, r1cs, ref_pk, w, r=rs_[0], s=rs_[1], resolve=res)
        for f in ("Ar", "Bs", "Krs"):
            assert np.array_equal(getattr(p_dev, f), getattr(p_ref, f)), f
        assert len(p_dev.Commitments) == len(p_ref.Commitments)
        if with_commitment:
            assert np.array_equal(p_dev.Commitments[0], p_ref.Commitments[0])
            assert np.array_equal(p_dev.CommitmentPok, p_ref.CommitmentPok)
        wit = p_dev.debug["witness"]
        pub = wit[1:r1cs.nb_public]
        g16.Verify(ctx, p_dev, vk, pub)
        ar, bs, krs = og.closed_form_proof(r1cs, tw, wit, rs_[0], rs_[1], _ints(p_dev.debug["h"]))
        assert np.array_equal(p_dev.Ar, bn.g1_to_array([ar])[0])
        assert np.array_equal(p_dev.Bs, bn.g2_to_array([bs])[0])
        assert np.array_equal(p_dev.Krs, bn.g1_to_array([krs])[0])
        batch = g16.BatchProve(ctx, r1cs, pk, [w, w], rs=rs_[:3:2], ss=rs_[1:4:2], resolve=res)
        batch_ref = g16.BatchProve(ctx, r1cs, ref_pk, [w, w], rs=rs_[:3:2], ss=rs_[1:4:2], resolve=res)
        for a, b in zip(batch, batch_ref):
            for f in ("Ar", "Bs", "Krs"):
                assert np.array_equal(getattr(a, f), getattr(b, f)), f
        for f in ("Ar", "Bs", "Krs"):
            assert np.array_equal(getattr(batch[0], f), getattr(p_dev, f)), f
        assert g16.BatchVerify(ctx, batch, vk, [b.debug["witness"][1:r1cs.nb_public] for b in batch]) == [True, True]
    finally:
        pk.free()
        ref_pk.free()


def test_device_setup_generated_circuit_end_to_end(ctx):
    d = sp.synthetic_csr(1 << 16, 21)
    sys_ = g16.SparseR1CS(**d)
    rng = random.Random(21)
    tw = g16.ToxicWaste(*[rng.randrange(1, R) for _ in range(6)])
    pk, vk = g16.DeviceSetup(ctx, sys_, tw, precompute=True)
    try:
        w = sp.csr_witness(d, 5)
        r, s = rng.randrange(R), rng.randrange(R)
        proof = g16.Prove(ctx, sys_, pk, w, r=r, s=s, want_h=True)
        g16.Verify(ctx, proof, vk, w[1:sys_.nb_public])
        # closed form from the C oracle's wire polynomials
        A, B, Cc = [_ints(x) for x in sp.setup_abc(d, _mont(tw.tau))]
        L = pk.log2_domain
        n = 1 << L
        h = _ints(proof.debug["h"])
        sa = sum(a * x for a, x in zip(A, w)) % R
        sb = sum(b * x for b, x in zip(B, w)) % R
        sk = sum((tw.beta * A[i] + tw.alpha * B[i] + Cc[i]) * w[i] for i in range(sys_.nb_public, sys_.nb_wires)) % R
        ht = sum(h[bitrev(i, L)] * pow(tw.tau, i, R) for i in range(n - 1)) % R
        di = pow(tw.delta, -1, R)
        ar = (tw.alpha + sa + r * tw.delta) % R
        bs = (tw.beta + sb + s * tw.delta) % R
        krs = (sk * di + ht * (pow(tw.tau, n, R) - 1) * di + s * ar + r * bs - r * s * tw.delta) % R
        assert np.array_equal(proof.Ar, cport.g1_gen_mul(_mont(ar)))
        assert np.array_equal(proof.Bs, cport.g2_gen_mul(_mont(bs)))
        assert np.array_equal(proof.Krs, cport.g1_gen_mul(_mont(krs)))
    finally:
        pk.free()


@pytest.mark.parametrize("log2m", [22])
def test_large_key_scalars_and_points(ctx, log2m):
    d = sp.synthetic_csr(1 << log2m, 100 + log2m)
    rng = random.Random(log2m)
    t = [rng.randrange(1, R) for _ in range(6)]
    tau, alpha, beta, gamma, delta, sigma = t
    A, B, Cc = _check_wire_polys_tau(ctx, d, tau)
    o = ctx.setup(d, *[_mont(v) for v in t])
    try:
        nw, npub, L = d["nb_wires"], d["nb_public"], o["log2_domain"]
        Ai, Bi = _ints(A), _ints(B)
        nz_a = [i for i in range(nw) if Ai[i]]
        nz_b = [i for i in range(nw) if Bi[i]]
        assert np.array_equal(o["infinity_a"], (~np.asarray([bool(x) for x in Ai])).astype(np.uint8))
        assert len(o["a"]) == len(nz_a) and len(o["b"]) == len(o["b2"]) == len(nz_b) and len(o["z"]) == (1 << L) - 1
        assert len(o["k"]) == nw - npub and o["ped_basis"] is None
        rs = np.random.Generator(np.random.PCG64(log2m))
        di = pow(delta, -1, R)
        zc = (pow(tau, 1 << L, R) - 1) * di % R
        for j in rs.integers(0, len(nz_a), size=16).tolist():
            assert np.array_equal(o["a"].download(j, 1)[0], lib.g1_scalar_mul(G1, A[nz_a[j]]))
        for j in rs.integers(0, len(nz_b), size=8).tolist():
            assert np.array_equal(o["b2"].download(j, 1)[0], lib.g2_scalar_mul(G2, B[nz_b[j]]))
        Ci = _ints(Cc)
        for j in rs.integers(0, len(o["k"]), size=16).tolist():
            i = npub + j
            k = (beta * Ai[i] + alpha * Bi[i] + Ci[i]) * di % R
            assert np.array_equal(o["k"].download(j, 1)[0], lib.g1_scalar_mul(G1, _mont(k)))
        for j in rs.integers(0, len(o["z"]), size=16).tolist():
            assert np.array_equal(o["z"].download(j, 1)[0], lib.g1_scalar_mul(G1, _mont(zc * pow(tau, bitrev(j, L), R))))
        # MSM(pk.A, x) == [sum x_i A_i(tau)] G
        x = sp.synthetic_csr(1, 0)["coeffs"]   # a few Montgomery scalars, tiled
        xs = np.ascontiguousarray(np.resize(x, (len(nz_a), 4)))
        exp = cport.g1_gen_mul(cport.fr_dot(A[nz_a], xs))
        assert np.array_equal(ctx.msm(o["a"], xs), exp)
    finally:
        for name in lib.SETUP_VECTORS:
            if o[name] is not None:
                o[name].free()


def _check_wire_polys_tau(ctx, d, tau):
    got = ctx.setup_wire_polys(d, _mont(tau))
    exp = sp.setup_abc(d, _mont(tau))
    for k in range(3):
        assert np.array_equal(got[k], exp[k]), "ABC"[k]
    return got


def _bad_cases():
    def base():
        r1cs, _ = og.synthetic_r1cs(24, 3, random.Random(9), with_commitment=True)
        return g16.SparseR1CS.from_r1cs(r1cs)
    out = []

    def case(name, fn):
        s = base()
        fn(s)
        out.append((name, s))
    case("no constraints", lambda s: setattr(s, "l_row", s.l_row[:1]) or setattr(s, "r_row", s.r_row[:1])
         or setattr(s, "o_row", s.o_row[:1]))
    case("row[0] != 0", lambda s: s.l_row.__setitem__(0, 1))
    case("row decreases", lambda s: s.r_row.__setitem__(5, s.r_row[6] + 1))
    case("wire out of range", lambda s: s.o_wire.__setitem__(3, s.nb_wires))
    case("coefficient id out of range", lambda s: s.l_coeff.__setitem__(0, len(s.coeffs)))
    case("n_public = 0", lambda s: setattr(s, "nb_public", 0))
    case("committed not increasing", lambda s: setattr(s, "private_committed", s.private_committed[::-1].copy()))
    case("committed public wire", lambda s: s.private_committed.__setitem__(0, 1))
    case("commitment wire public", lambda s: setattr(s, "commitment_wire", 1))
    case("commitment wire committed", lambda s: setattr(s, "commitment_wire", int(s.private_committed[0])))
    case("commitment wire out of range", lambda s: setattr(s, "commitment_wire", s.nb_wires))
    case("committed without commitment", lambda s: setattr(s, "commitment_wire", -1))
    return out


@pytest.mark.parametrize("name,sys_", _bad_cases(), ids=[c[0] for c in _bad_cases()])
def test_setup_arg_errors_leave_ctx_usable(ctx, name, sys_):
    t = [_mont(v) for v in (5, 6, 7, 8, 9, 10)]
    with pytest.raises(lib.B200Error, match="error -2"):
        ctx.setup(sys_, *t)
    with pytest.raises(lib.B200Error, match="error -2"):
        ctx.setup_wire_polys(sys_, t[0])
    _valid_setup_and_prove(ctx)


@pytest.mark.parametrize("which", ["domain_over_2p28", "nnz_over_limit", "n_wires_2p32"])
def test_setup_size_limits(ctx, which):
    """Shapes past the limits, refused on the host before any array is read past its first and last row entries."""
    import ctypes
    row = np.array([0, 1], dtype=np.uint64)
    one = np.zeros(1, dtype=np.uint32)
    coeffs = g16.fr_array([1])
    d = lib.R1csDesc()
    d.n_constraints, d.n_wires, d.n_public, d.n_coeffs, d.commitment_wire = 1, 4, 1, 1, -1
    d.coeffs = coeffs.ctypes.data_as(ctypes.c_void_p)
    big = np.array([0, 0xf0000001], dtype=np.uint64)
    for p in "lro":
        r = big if (which == "nnz_over_limit" and p == "r") else row
        setattr(d, p + "_row", r.ctypes.data_as(ctypes.c_void_p))
        setattr(d, p + "_wire", one.ctypes.data_as(ctypes.c_void_p))
        setattr(d, p + "_coeff", one.ctypes.data_as(ctypes.c_void_p))
    if which == "domain_over_2p28":
        d.n_constraints = (1 << 28) + 1        # the row arrays are never read
    elif which == "n_wires_2p32":
        d.n_wires = 1 << 32
    t = lib.Toxic()
    for name, v in zip(("tau", "alpha", "beta", "gamma", "delta", "sigma"), g16.fr_array([5, 6, 7, 8, 9, 10])):
        getattr(t, name)[:] = [int(x) for x in v]
    flags = np.zeros((3, 4), dtype=np.uint8)
    out = lib.SetupOut()
    L = lib.load()
    st = L.b200g16_setup(ctx.h, ctypes.byref(d), ctypes.byref(t), *[f.ctypes.data_as(ctypes.c_void_p) for f in flags],
                         ctypes.byref(out))
    assert st == -2, L.b200g16_last_error()
    a = np.zeros((4, 4), dtype=np.uint64)
    assert L.b200g16_setup_wire_polys(ctx.h, ctypes.byref(d), g16.fr_array([5]).ctypes.data_as(ctypes.c_void_p),
                                      a.ctypes.data_as(ctypes.c_void_p), None, None) == -2
    _valid_setup_and_prove(ctx)


@pytest.mark.parametrize("which", ["gamma", "delta", "tau_in_domain"])
def test_setup_toxic_errors(ctx, which):
    r1cs, _, _, _ = _case(24, 3, True)
    sys_ = g16.SparseR1CS.from_r1cs(r1cs)
    t = [5, 6, 7, 8, 9, 10]
    if which == "gamma":
        t[3] = 0
    elif which == "delta":
        t[4] = 0
    else:
        from oracle.ntt import Domain
        t[0] = pow(Domain(24).gen, 5, R)
    with pytest.raises(lib.B200Error, match="error -2"):
        ctx.setup(sys_, *[_mont(v) for v in t])
    _valid_setup_and_prove(ctx)


def test_setup_refused_during_split_prove(ctx):
    import torch
    r1cs, w, tw, _ = _case(24, 3, False)
    gtw = g16.ToxicWaste(tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma)
    pk, _ = g16.DeviceSetup(ctx, r1cs, gtw)
    try:
        wires = torch.from_numpy(g16.fr_array(w).view(np.int64)).cuda()
        h = torch.zeros((1 << pk.log2_domain, 4), dtype=torch.int64, device="cuda")
        ctx.prove_begin_dev(pk.device_handle(ctx), wires.data_ptr())
        sys_ = g16.SparseR1CS.from_r1cs(r1cs)
        with pytest.raises(lib.B200Error, match="error -4"):
            ctx.setup(sys_, *g16.fr_array([5, 6, 7, 8, 9, 10]))
        with pytest.raises(lib.B200Error, match="error -4"):
            ctx.setup_wire_polys(sys_, g16.fr_array([5])[0])
        ctx.prove_end_dev(pk.device_handle(ctx), h.data_ptr(), g16.fr_array([1])[0], g16.fr_array([2])[0])
    finally:
        pk.free()
    _valid_setup_and_prove(ctx)


def _valid_setup_and_prove(ctx):
    r1cs, w, tw, rng = _case(24, 3, True)
    pk, vk = g16.DeviceSetup(ctx, r1cs, g16.ToxicWaste(tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma))
    try:
        proof = g16.Prove(ctx, r1cs, pk, w, r=rng.randrange(R), s=rng.randrange(R), resolve=_resolve(r1cs))
        g16.Verify(ctx, proof, vk, proof.debug["witness"][1:r1cs.nb_public])
    finally:
        pk.free()
