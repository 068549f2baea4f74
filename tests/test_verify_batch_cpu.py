"""Batch Groth16 verification on the CPU: a restatement of the small-exponent batch test on the oracle's pairing
(batch_verify below), checked on real proofs from the oracle's setup / prove, and a pin of the scalar
multiplication the batch verifier's kernels run (gnark_whir_b200/csrc/verify_batch.cuh, compiled for the host by
tests/host_harness/verify_batch_host.cc) against oracle/bn254.py.

The restatement lives here, beside its tests, so that the oracle package itself stays untouched; the GPU tests
(tests/test_gpu_verify_batch.py) share its proof fixtures."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bn254 as bn
from oracle import groth16 as og
from oracle.bn254 import R

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_harness", "verify_batch_host.cc")
OUT = os.path.join(HERE, "host_harness", "_build", "verify_batch_host.so")
CSRC = os.path.join(HERE, "..", "gnark_whir_b200", "csrc")


def g2_in_subgroup(q):
    return q is None or (bn.g2_on_curve(q) and bn._mul(bn._F2, q, R, mod=R + 1) is None)


def batch_verify(proofs, vk, publics, rho, tau=None):
    """The batch test b200g16_verify_batch runs, on the oracle's pairing.  publics[i]: proof i's public wires
    INCLUDING wire 0 (as og.verify takes them); rho: k coefficients, tau: k more with a commitment."""
    com = vk.has_commitment
    pubs = []
    for p, pw in zip(proofs, publics):
        pub = list(pw)
        if com:
            pub.append(og.commitment_challenge(p.commitments[0], [pw[i] for i in vk.public_committed]))
        if len(pub) != len(vk.K):
            return False
        pubs.append(pub)
    pts1 = [p.Ar for p in proofs] + [p.Krs for p in proofs]
    if com:
        pts1 += [p.commitments[0] for p in proofs] + [p.commitment_pok for p in proofs]
    if not all(q is None or bn.g1_on_curve(q) for q in pts1) or not all(g2_in_subgroup(p.Bs) for p in proofs):
        return False
    # wire 0 is the constant one, so y_0 = sum_i rho_i = S and K_0 takes S
    y = [sum(r * pub[j] for r, pub in zip(rho, pubs)) % R for j in range(len(vk.K))]
    lsum = bn.g1_sum([bn.g1_msm(vk.K, y)] + ([bn.g1_mul(p.commitments[0], r) for p, r in zip(proofs, rho)] if com else []))
    pairs = [(bn.g1_mul(p.Ar, r), p.Bs) for p, r in zip(proofs, rho)]
    pairs += [(bn.g1_neg(bn.g1_mul(vk.alpha1, sum(rho) % R)), vk.beta2),
              (bn.g1_neg(lsum), vk.gamma2),
              (bn.g1_neg(bn.g1_sum([bn.g1_mul(p.Krs, r) for p, r in zip(proofs, rho)])), vk.delta2)]
    if com:
        pairs += [(bn.g1_sum([bn.g1_mul(p.commitments[0], t) for p, t in zip(proofs, tau)]), vk.ped_g_sigma_neg),
                  (bn.g1_sum([bn.g1_mul(p.commitment_pok, t) for p, t in zip(proofs, tau)]), vk.ped_g)]
    return bn.pairing_check(pairs)


def resolve_witness(r1cs, w, publics, seeds):
    """Another satisfying witness of a synthetic_r1cs circuit: new public inputs and seed wires, every constraint
    output recomputed in order (the commitment wire is filled afterwards by og.finalize_witness)."""
    w = list(w)
    w[1:r1cs.nb_public] = publics
    w[r1cs.nb_public:r1cs.nb_public + len(seeds)] = seeds
    for L, Rr, O in r1cs.constraints:
        w[O[0][0]] = og.lc_eval(L, w) * og.lc_eval(Rr, w) % R
    return w


def oracle_proofs(k, nb_public, with_commitment, seed):
    """k proofs of one synthetic circuit over different witnesses -> (tw, vk, proofs, public wires incl. wire 0)"""
    rng = random.Random(seed)
    r1cs, w = og.synthetic_r1cs(6, nb_public, rng, with_commitment=with_commitment)
    tw = og.ToxicWaste(*[rng.randrange(1, R) for _ in range(5)], sigma=rng.randrange(1, R))
    pk, vk = og.setup(r1cs, tw)
    proofs, publics = [], []
    for _ in range(k):
        wi = resolve_witness(r1cs, w, [rng.randrange(1000) for _ in range(nb_public - 1)],
                             [rng.randrange(R) for _ in range(4)])
        com = og.finalize_witness(r1cs, pk, wi)
        assert og.is_satisfied(r1cs, wi)
        proof, _ = og.prove(r1cs, pk, wi, rng.randrange(R), rng.randrange(R), commitment=com)
        proofs.append(proof)
        publics.append(wi[:r1cs.nb_public])
    return tw, vk, proofs, publics


def _coeffs(rng, k):
    return [rng.randrange(1, 1 << 128) for _ in range(k)]


@pytest.fixture(scope="module")
def plain():
    return oracle_proofs(3, 3, False, 71)


@pytest.fixture(scope="module")
def committed():
    return oracle_proofs(2, 3, True, 72)


def test_batch_accepts_valid_proofs(plain, committed):
    rng = random.Random(1)
    _, vk, proofs, publics = plain
    assert all(og.verify(p, vk, pw) for p, pw in zip(proofs, publics))
    assert batch_verify(proofs, vk, publics, _coeffs(rng, 3))
    _, vk, proofs, publics = committed
    assert batch_verify(proofs, vk, publics, _coeffs(rng, 2), _coeffs(rng, 2))


def test_batch_rejects_changed_krs_and_swapped_publics(plain):
    rng = random.Random(2)
    _, vk, proofs, publics = plain
    bad = list(proofs)
    bad[1] = og.Proof(bad[1].Ar, bad[1].Bs, bn.g1_add(bad[1].Krs, bn.G1_GEN))
    assert not batch_verify(bad, vk, publics, _coeffs(rng, 3))
    assert publics[0] != publics[2]
    swapped = [publics[2], publics[1], publics[0]]
    assert not batch_verify(proofs, vk, swapped, _coeffs(rng, 3))


def test_cancelling_pair_needs_distinct_coefficients(plain):
    """Krs_1 + E and Krs_2 - E cancel in the sum of the Krs: distinct rho expose them, equal rho do not."""
    rng = random.Random(3)
    _, vk, proofs, publics = plain
    E = bn.g1_mul(bn.G1_GEN, rng.randrange(1, R))
    bad = [og.Proof(proofs[0].Ar, proofs[0].Bs, bn.g1_add(proofs[0].Krs, E)),
           og.Proof(proofs[1].Ar, proofs[1].Bs, bn.g1_add(proofs[1].Krs, bn.g1_neg(E))), proofs[2]]
    assert not og.verify(bad[0], vk, publics[0]) and not og.verify(bad[1], vk, publics[1])
    rho = _coeffs(rng, 3)
    assert not batch_verify(bad, vk, publics, rho)
    assert batch_verify(bad, vk, publics, [rho[0], rho[0], rho[2]])


def test_pok_error_cannot_offset_a_main_error_under_independent_tau(committed):
    """Krs_0 + E breaks the main equation by e(G, H)^(-rho_0 e delta); PoK_0 + delta E breaks the proof of knowledge
    by e(G, H)^(tau_0 e delta).  With tau = rho the two cancel, with independent tau they do not."""
    rng = random.Random(4)
    tw, vk, proofs, publics = committed
    E = bn.g1_mul(bn.G1_GEN, rng.randrange(1, R))
    p0 = proofs[0]
    bad0 = og.Proof(p0.Ar, p0.Bs, bn.g1_add(p0.Krs, E), p0.commitments,
                    bn.g1_add(p0.commitment_pok, bn.g1_mul(E, tw.delta)))
    bad = [bad0, proofs[1]]
    assert not og.verify(bad0, vk, publics[0])
    rho, tau = _coeffs(rng, 2), _coeffs(rng, 2)
    assert not batch_verify(bad, vk, publics, rho, tau)
    assert batch_verify(bad, vk, publics, rho, rho)


# ---------------------------------------------------------------------------- host pin of the scalar multiplication
@pytest.fixture(scope="module")
def H():
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-I", CSRC, "-o", OUT], check=True)
    return C.CDLL(OUT)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _words(x, n):
    return np.array([(x >> (64 * i)) & ((1 << 64) - 1) for i in range(n)], dtype=np.uint64)


def test_coefficient_scalar_mul_matches_oracle(H):
    rng = random.Random(5)
    out = np.zeros(8, dtype=np.uint64)
    pts = [bn.G1_GEN, bn.g1_mul(bn.G1_GEN, rng.randrange(1, R))]
    for pt in pts:
        for c in [1, 2, 3, (1 << 128) - 1, 1 << 127, (1 << 64) - 1, 1 << 64] + _coeffs(rng, 4):
            H.host_g1_mul_coeff(_ptr(bn.g1_to_array([pt])[0]), _ptr(_words(c, 2)), _ptr(out))
            assert bn.g1_from_array(out.reshape(1, 8))[0] == bn.g1_mul(pt, c), hex(c)
    # the point at infinity stays there; a zero coefficient (rejected by the ABI) would give infinity
    inf = np.zeros(8, dtype=np.uint64)
    H.host_g1_mul_coeff(_ptr(inf), _ptr(_words((1 << 128) - 1, 2)), _ptr(out))
    assert not out.any()
    H.host_g1_mul_coeff(_ptr(bn.g1_to_array([pts[1]])[0]), _ptr(_words(0, 2)), _ptr(out))
    assert not out.any()


def test_full_width_scalar_mul_matches_oracle(H):
    """S * alpha in k_fixed_pairs: S is a canonical Fr element, 254 bits."""
    rng = random.Random(6)
    out = np.zeros(8, dtype=np.uint64)
    pt = bn.g1_mul(bn.G1_GEN, rng.randrange(1, R))
    for s in [1, R - 1, (1 << 253) + 5] + [rng.randrange(R) for _ in range(3)]:
        H.host_g1_mul_bits(_ptr(bn.g1_to_array([pt])[0]), _ptr(_words(s, 4)), 254, _ptr(out))
        assert bn.g1_from_array(out.reshape(1, 8))[0] == bn.g1_mul(pt, s)
