"""GPU: batch Groth16 verification (b200g16_verify_batch, Context.verify_batch, groth16.BatchVerify) on real proofs
from Setup / Prove, on simulated proofs minted from a verifying key with known discrete logs, on tampered batches
(the per-proof answers must name exactly the bad proofs), on malformed calls, and on the context afterwards."""
import random

import numpy as np
import pytest

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import bn254 as bn
from oracle import cport
from oracle import groth16 as og
from oracle.bn254 import R
from tests.test_pairing_cpu import _f2_sqrt

pytestmark = pytest.mark.gpu

G1 = g16.g1_point(g16.G1_GEN)
G2 = g16.g2_point(g16.G2_GEN)


class SimBatch:
    """k valid proofs for a verifying key whose alpha, beta, gamma, delta, K_j and sigma have known discrete logs:
    A = a G, B = b H, C = c G with c = (ab - alpha beta - gamma l) / delta, where l is the discrete log of
    L = K_0 + sum_j x_j K_j (+ D), the commitment challenge's K term included; D = d G and PoK = sigma D.
    n_public counts b200g16_verify's public inputs, so with a commitment the public witness has n_public - 1."""

    def __init__(self, ctx, k, n_public, with_commitment, seed):
        rng = random.Random(seed)
        alpha, beta, gamma, delta, sigma = [rng.randrange(1, R) for _ in range(5)]
        kd = [rng.randrange(1, R) for _ in range(n_public + 1)]
        g1s = ctx.fixed_base_mul(G1, g16.fr_array(kd + [alpha]), group=1)
        g2s = ctx.fixed_base_mul(G2, g16.fr_array([beta, gamma, delta, (-sigma) % R]), group=2)
        n_wit = n_public - 1 if with_commitment else n_public
        self.vk = g16.VerifyingKey(g1s[-1], g1s[:-1].copy(), g2s[0], g2s[1], g2s[2])
        if with_commitment:
            self.vk.PedersenG, self.vk.PedersenGSigmaNeg = G2.copy(), g2s[3]
            self.vk.PublicAndCommitmentCommitted = [1] if n_wit else []
            self.vk.has_commitment = True
        self.witnesses = [[rng.randrange(R) if rng.random() < 0.5 else rng.randrange(256) for _ in range(n_wit)]
                          for _ in range(k)]
        ls = [(kd[0] + sum(x * kj for x, kj in zip(w, kd[1:]))) % R for w in self.witnesses]
        coms, poks = [None] * k, [None] * k
        if with_commitment:
            ds = [rng.randrange(1, R) for _ in range(k)]
            coms = list(ctx.fixed_base_mul(G1, g16.fr_array(ds), group=1))
            poks = list(ctx.fixed_base_mul(G1, g16.fr_array([sigma * d % R for d in ds]), group=1))
            for i, w in enumerate(self.witnesses):
                ch = g16.commitment_challenge(coms[i], [1 if j == 0 else w[j - 1] for j in self.vk.PublicAndCommitmentCommitted])
                ls[i] = (ls[i] + ch * kd[-1] + ds[i]) % R
        a = [rng.randrange(1, R) for _ in range(k)]
        b = [rng.randrange(1, R) for _ in range(k)]
        di = pow(delta, -1, R)
        c = [(ai * bi - alpha * beta - gamma * li) * di % R for ai, bi, li in zip(a, b, ls)]
        A = ctx.fixed_base_mul(G1, g16.fr_array(a + c), group=1)
        B = ctx.fixed_base_mul(G2, g16.fr_array(b), group=2)
        self.proofs = [g16.Proof(A[i], A[k + i], B[i], [coms[i]] if with_commitment else [], poks[i]) for i in range(k)]

    def arrays(self):
        """(ar, bs, krs, public inputs (k, n_public, 4), commitments, poks) as b200g16_verify_batch takes them"""
        ins = [g16._verify_inputs(p, self.vk, w) for p, w in zip(self.proofs, self.witnesses)]
        n_pub = len(self.vk.G1_K) - 1
        pubs = np.stack([g16.fr_array(pub) if pub else np.zeros((0, 4), np.uint64) for pub, _, _ in ins]) if ins \
            else np.zeros((0, n_pub, 4), np.uint64)
        st = lambda xs, w: np.array(xs, dtype=np.uint64).reshape(len(xs), w)
        com = st([c for _, c, _ in ins], 8) if self.vk.has_commitment else None
        pok = st([p for _, _, p in ins], 8) if self.vk.has_commitment else None
        return (st([p.Ar for p in self.proofs], 8), st([p.Bs for p in self.proofs], 16),
                st([p.Krs for p in self.proofs], 8), pubs, com, pok)

    def verify_batch(self, ctx, coeffs, **kw):
        ar, bs, krs, pubs, com, pok = self.arrays()
        v = self.vk
        return ctx.verify_batch(v.G1_Alpha, v.G2_Beta, v.G2_Gamma, v.G2_Delta, v.G1_K, ar, bs, krs, pubs, coeffs,
                                commitments=com, poks=pok, ped_g=v.PedersenG if v.has_commitment else None,
                                ped_g_sigma_neg=v.PedersenGSigmaNeg if v.has_commitment else None, **kw)


def _coeff_words(rng, n):
    c = [rng.randrange(1, 1 << 128) for _ in range(n)]
    return np.array([(x & (2**64 - 1), x >> 64) for x in c], dtype=np.uint64).reshape(n, 2)


def _verify_one(ctx, proof, vk, w):
    try:
        g16.Verify(ctx, proof, vk, w)
        return True
    except ValueError:
        return False


# ------------------------------------------------------------------------------------------------ real proofs
@pytest.mark.parametrize("nb_constraints,nb_public,with_commitment", [(7, 1, False), (24, 3, False), (40, 4, True)])
def test_batch_accepts_setup_prove_proofs(ctx, nb_constraints, nb_public, with_commitment):
    rng = random.Random(100 + nb_constraints)
    r1cs, w = og.synthetic_r1cs(nb_constraints, nb_public, rng, with_commitment=with_commitment)
    pk, vk = g16.Setup(ctx, r1cs)
    try:
        def resolve(wit):
            L, Rr, O = r1cs.constraints[-1]
            wit[O[0][0]] = og.lc_eval(L, wit) * og.lc_eval(Rr, wit) % R
        proofs = [g16.Prove(ctx, r1cs, pk, w, r=rng.randrange(R), s=rng.randrange(R),
                            resolve=resolve if with_commitment else None) for _ in range(5)]
        publics = [p.debug["witness"][1:r1cs.nb_public] for p in proofs]
        assert len({bytes(p.Ar.tobytes()) for p in proofs}) == 5
        got = g16.BatchVerify(ctx, proofs, vk, publics)
        assert got == [True] * 5
        assert got == [_verify_one(ctx, p, vk, pw) for p, pw in zip(proofs, publics)]
    finally:
        pk.free()


# ------------------------------------------------------------------------------------------------ simulated proofs
# the per-proof kernels run 64-thread CTAs, the public-input fold 256-thread CTAs, the product tree 64 values per CTA
SIM_K = [1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 16384]
SIM_SHAPES = [(False, 0), (False, 1), (False, 5), (True, 1), (True, 5)]


@pytest.mark.parametrize("with_commitment,n_public", SIM_SHAPES)
@pytest.mark.parametrize("k", SIM_K)
def test_batch_accepts_simulated_proofs(ctx, k, with_commitment, n_public):
    sim = SimBatch(ctx, k, n_public, with_commitment, seed=k * 10 + n_public + with_commitment)
    got = g16.BatchVerify(ctx, sim.proofs, sim.vk, sim.witnesses)
    assert got == [True] * k
    phases = ctx.last_timings()
    assert len(phases) == 5 and all(t >= 0 for t in phases)
    if k <= 2:
        assert all(_verify_one(ctx, p, sim.vk, w) for p, w in zip(sim.proofs, sim.witnesses))


# ------------------------------------------------------------------------------------------------ tampering
N_TAMPER = 129


@pytest.fixture(scope="module")
def sim129(ctx):
    return SimBatch(ctx, N_TAMPER, 5, True, seed=129)


def _twist_point_outside_torsion():
    x = (5, 1)
    while True:
        y = _f2_sqrt(bn.f2_add(bn.f2_mul(bn.f2_sqr(x), x), bn.B2))
        if y is not None:
            return bn.g2_to_array([(x, y)])[0]
        x = (x[0] + 1, x[1])


def _fr1(v):
    return g16.fr_array([v])[0]


def _tamper(proofs, wits, cls, p, ctx):
    """copies of proofs / witnesses with tampering class `cls` applied at position p, and the indexes that must fail"""
    proofs = [g16.Proof(q.Ar, q.Krs, q.Bs, list(q.Commitments), q.CommitmentPok) for q in proofs]
    wits = [list(w) for w in wits]
    q = p + 1 if p + 1 < len(proofs) else p - 1
    pr = proofs[p]
    if cls == "ar_double":
        pr.Ar = lib.g1_scalar_mul(pr.Ar, _fr1(2))
    elif cls == "krs_plus_g":
        pr.Krs = lib.g1_add(pr.Krs, G1)
    elif cls == "bs_other":
        pr.Bs = lib.g2_scalar_mul(pr.Bs, _fr1(3))
    elif cls == "bs_outside_torsion":
        pr.Bs = _twist_point_outside_torsion()
    elif cls == "ar_off_curve":
        x, y = bn.g1_from_array(pr.Ar.reshape(1, 8))[0]
        pr.Ar = bn.g1_to_array([(x, (y + 1) % bn.P)])[0]
    elif cls == "public_plus_one":
        wits[p][0] = (wits[p][0] + 1) % R
    elif cls == "publics_swapped":
        wits[p], wits[q] = wits[q], wits[p]
        return proofs, wits, {p, q}
    elif cls == "commitment_changed":
        pr.Commitments = [lib.g1_add(pr.Commitments[0], G1)]
    elif cls == "pok_times_3":
        pr.CommitmentPok = lib.g1_scalar_mul(pr.CommitmentPok, _fr1(3))
    elif cls == "cancelling_pair":
        E = ctx.fixed_base_mul(G1, g16.fr_array([12345]), group=1)[0]
        nE = ctx.fixed_base_mul(G1, g16.fr_array([R - 12345]), group=1)[0]
        pr.Krs = lib.g1_add(pr.Krs, E)
        proofs[q].Krs = lib.g1_add(proofs[q].Krs, nE)
        return proofs, wits, {p, q}
    return proofs, wits, {p}


TAMPER = ["ar_double", "krs_plus_g", "bs_other", "bs_outside_torsion", "ar_off_curve", "public_plus_one",
          "publics_swapped", "commitment_changed", "pok_times_3", "cancelling_pair"]


@pytest.mark.parametrize("cls", TAMPER)
def test_batch_rejects_and_names_tampered_proofs(ctx, sim129, cls):
    for p in (0, N_TAMPER // 2, N_TAMPER - 1):
        proofs, wits, bad = _tamper(sim129.proofs, sim129.witnesses, cls, p, ctx)
        got = g16.BatchVerify(ctx, proofs, sim129.vk, wits)
        assert [i for i, ok in enumerate(got) if not ok] == sorted(bad), (cls, p)
        assert len(ctx.last_timings()) == 6          # the per-proof pass ran


def test_ok_each_equals_single_verify_on_mixed_batch(ctx):
    sim = SimBatch(ctx, 12, 5, True, seed=12)
    proofs, wits = sim.proofs, sim.witnesses
    for cls, p in (("ar_double", 1), ("pok_times_3", 5), ("bs_outside_torsion", 8), ("public_plus_one", 10)):
        proofs, wits, _ = _tamper(proofs, wits, cls, p, ctx)
    got = g16.BatchVerify(ctx, proofs, sim.vk, wits)
    assert got == [_verify_one(ctx, pr, sim.vk, w) for pr, w in zip(proofs, wits)]
    assert [i for i, ok in enumerate(got) if not ok] == [1, 5, 8, 10]


# ------------------------------------------------------------------------------------------------ errors, edges
def test_batch_errors_and_edge_cases(ctx):
    rng = random.Random(7)
    sim = SimBatch(ctx, 4, 5, True, seed=7)
    co = _coeff_words(rng, 8)
    ok, each = sim.verify_batch(ctx, co)
    assert ok and each.all()
    ok2, none = sim.verify_batch(ctx, co, want_each=False)    # ok_each = NULL
    assert ok2 and none is None
    zero = co.copy()
    zero[6] = 0                                               # a zero tau
    with pytest.raises(lib.B200Error):
        sim.verify_batch(ctx, zero)
    ar, bs, krs, pubs, com, pok = sim.arrays()
    v = sim.vk
    call = lambda **kw: ctx.verify_batch(v.G1_Alpha, v.G2_Beta, v.G2_Gamma, v.G2_Delta, v.G1_K, **kw)
    base = dict(ar=ar, bs=bs, krs=krs, public_inputs=pubs, coeffs=co, commitments=com, poks=pok, ped_g=v.PedersenG,
                ped_g_sigma_neg=v.PedersenGSigmaNeg)
    with pytest.raises(lib.B200Error):                        # n_public + 1 != n_k
        call(**{**base, "public_inputs": pubs[:, :4]})
    with pytest.raises(lib.B200Error):                        # commitments without poks
        call(**{**base, "poks": None})
    with pytest.raises(lib.B200Error):                        # commitments without the pedersen key
        call(**{**base, "ped_g": None, "ped_g_sigma_neg": None})
    # k = 0 accepts
    ok, each = call(ar=np.zeros((0, 8), np.uint64), bs=np.zeros((0, 16), np.uint64), krs=np.zeros((0, 8), np.uint64),
                    public_inputs=np.zeros((0, 5, 4), np.uint64), coeffs=np.zeros((0, 2), np.uint64),
                    commitments=np.zeros((0, 8), np.uint64), poks=np.zeros((0, 8), np.uint64), ped_g=v.PedersenG,
                    ped_g_sigma_neg=v.PedersenGSigmaNeg)
    assert ok and each.shape == (0,)
    assert g16.BatchVerify(ctx, [], sim.vk, []) == []


def test_fixed_coefficients_are_deterministic(ctx, sim129):
    proofs, wits, bad = _tamper(sim129.proofs, sim129.witnesses, "cancelling_pair", 40, ctx)
    rng = random.Random(8)
    coeffs = [rng.randrange(1, 1 << 128) for _ in range(2 * N_TAMPER)]
    first = g16.BatchVerify(ctx, proofs, sim129.vk, wits, coeffs=coeffs)
    assert first == g16.BatchVerify(ctx, proofs, sim129.vk, wits, coeffs=coeffs)
    assert [i for i, ok in enumerate(first) if not ok] == sorted(bad)
    # equal coefficients on the cancelling pair let it through: the coefficients are what catches it
    coeffs[41] = coeffs[40]
    assert g16.BatchVerify(ctx, proofs, sim129.vk, wits, coeffs=coeffs) == [True] * N_TAMPER


# ------------------------------------------------------------------------------------------------ ctx reuse
def test_ctx_usable_after_batches(ctx):
    rng = random.Random(9)
    sim = SimBatch(ctx, 300, 5, True, seed=9)
    proofs, wits, _ = _tamper(sim.proofs, sim.witnesses, "krs_plus_g", 3, ctx)
    assert g16.BatchVerify(ctx, proofs, sim.vk, wits).count(False) == 1     # the fallback ran too
    # an MSM on the same ctx against its closed form
    rs = np.random.Generator(np.random.PCG64(9))
    ks = rs.integers(0, 1 << 62, size=(3000, 4), dtype=np.uint64)
    sc = rs.integers(0, 1 << 62, size=(3000, 4), dtype=np.uint64)
    bases = ctx.fixed_base_mul(G1, ks, group=1, resident=True)
    try:
        assert np.array_equal(ctx.msm(bases, sc), cport.g1_gen_mul(cport.fr_dot(ks, sc)))
    finally:
        bases.free()
    # a small prove on the same ctx against the closed form
    r1cs, w = og.synthetic_r1cs(24, 3, rng)
    tw = og.ToxicWaste(*[rng.randrange(1, R) for _ in range(5)], sigma=rng.randrange(1, R))
    r, s = rng.randrange(R), rng.randrange(R)
    pk, vk = g16.Setup(ctx, r1cs, g16.ToxicWaste(tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma))
    try:
        proof = g16.Prove(ctx, r1cs, pk, w, r=r, s=s, want_h=True)
        h = bn.fr_from_mont_array(proof.debug["h"])
        ar, bs, krs = og.closed_form_proof(r1cs, tw, w, r, s, h)
        assert np.array_equal(proof.Ar, bn.g1_to_array([ar])[0])
        assert np.array_equal(proof.Bs, bn.g2_to_array([bs])[0])
        assert np.array_equal(proof.Krs, bn.g1_to_array([krs])[0])
        assert g16.BatchVerify(ctx, [proof], vk, [w[1:r1cs.nb_public]]) == [True]
    finally:
        pk.free()
