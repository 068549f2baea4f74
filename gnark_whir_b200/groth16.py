"""Host-side mirror of gnark's groth16 API for BN254, on top of libb200g16.

Same entry points, argument meaning and flow as the calls the reference makes at
/root/reference/mt.go:448 (groth16.Setup), mt.go:496 (groth16.Prove) and mt.go:497
(groth16.Verify); gnark v0.11.0 backend/groth16/bn254/{setup,prove}.go is the behaviour
restated.  What runs where:

  Setup   host: toxic waste, per-wire A_i(tau), B_i(tau), C_i(tau), K_i, Z_i scalars (python ints)
          GPU : every group element, through b200g16_fixed_base_mul_g1/g2
  DeviceSetup  the same key, all of it on the GPU (b200g16_setup), point vectors left resident
  Prove   host: the constraint "solver" (here: L.w, R.w, O.w from a full assignment), the BSB22
                challenge hash, sampling r, s
          GPU : Pedersen commit + PoK (b200g16_msm_g1), computeH, the five MSMs, via b200g16_prove
  Verify  host: the BSB22 challenge hash
          GPU : public-input MSM, Pedersen PoK check and the pairing product, via b200g16_verify
  BatchVerify  k proofs of one circuit in one b200g16_verify_batch call (small-exponent batch test)
  wire formats (gnark / gnark-crypto marshal.go): Proof, VerifyingKey, ProvingKey, fft.Domain; the point encodings run
          batched on the GPU (b200g16_g1/g2_encode / _decode)

The host language would be Go (a cgo shim, INTEGRATION.md) if a Go toolchain existed in this
image; this module is the same marshalling in Python over ctypes.  There is no CPU fallback:
every group operation below goes through the CUDA library.
"""
from __future__ import annotations

import functools
import hashlib
import secrets
from dataclasses import dataclass, field

import numpy as np

from . import lib

R_MOD = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
P_MOD = 0x30644e72e131a029b85045b68181585d97816a916871ca8d3c208c16d87cfd47
_ROOT_2_28 = 19103219067921713944291392827692070036145651957329286315305642004821462161904
_MONT = 1 << 256
_M64 = (1 << 64) - 1

G1_GEN = (1, 2)
G2_GEN = ((10857046999023057135944570762232829481370756359578518086990519993285655852781,
           11559732032986387107991004021392285783925812861821192530917403151452391805634),
          (8495653923123431417604973247489272438418190587263600148770280649306958101930,
           4082367875863433681332203403145435568316851327593401208105741076214120093531))


# ---------------------------------------------------------------- layout helpers (fr.Element etc.)
def fr_array(vals):
    out = np.empty((len(vals), 4), dtype=np.uint64)
    for i, v in enumerate(vals):
        m = v % R_MOD * _MONT % R_MOD
        out[i] = (m & _M64, (m >> 64) & _M64, (m >> 128) & _M64, m >> 192)
    return out


def _fp_limbs(x):
    m = x % P_MOD * _MONT % P_MOD
    return [m & _M64, (m >> 64) & _M64, (m >> 128) & _M64, m >> 192]


def g1_point(pt):
    return np.array(_fp_limbs(pt[0]) + _fp_limbs(pt[1]), dtype=np.uint64)


def g2_point(pt):
    (x0, x1), (y0, y1) = pt
    return np.array(_fp_limbs(x0) + _fp_limbs(x1) + _fp_limbs(y0) + _fp_limbs(y1), dtype=np.uint64)


def _fp_from(limbs):
    v = int(limbs[0]) | int(limbs[1]) << 64 | int(limbs[2]) << 128 | int(limbs[3]) << 192
    return v * pow(_MONT, -1, P_MOD) % P_MOD


# ---------------------------------------------------------------- constraint system (host)
@dataclass
class R1CS:
    """Rank-1 system: wires [0, nb_public) public (wire 0 = 1), rest private.
    constraints: list of (L, R, O), each [(wire, coeff)].  Optional single BSB22 commitment."""
    nb_wires: int
    nb_public: int
    constraints: list
    private_committed: list = field(default_factory=list)
    public_committed: list = field(default_factory=list)
    commitment_wire: int = -1


@dataclass
class SparseR1CS:
    """A constraint system as gnark stores it (constraint/r1cs.go): an interned coefficient table and, per matrix,
    CSR arrays by constraint of Term{CID, VID} (provekit.InternedR1CS has the same shape).  Constraint j of L holds
    the terms l_wire[l_row[j]:l_row[j+1]] with coefficients coeffs[l_coeff[...]]; likewise R and O.  This is what
    b200g16_setup takes (struct b200g16_r1cs_desc)."""
    nb_wires: int
    nb_public: int
    coeffs: np.ndarray             # (n, 4) fr.Element, Montgomery
    l_row: np.ndarray              # uint64, n_constraints + 1
    l_wire: np.ndarray             # uint32
    l_coeff: np.ndarray            # uint32
    r_row: np.ndarray
    r_wire: np.ndarray
    r_coeff: np.ndarray
    o_row: np.ndarray
    o_wire: np.ndarray
    o_coeff: np.ndarray
    private_committed: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.uint32))
    public_committed: list = field(default_factory=list)
    commitment_wire: int = -1

    def __getitem__(self, name):   # the mapping lib.Context.setup reads
        return getattr(self, name)

    @staticmethod
    def from_r1cs(r1cs):
        """Intern the coefficients of a Python R1CS and lay its three matrices out as CSR; every term is kept, in
        order (repeated wires and zero coefficients included)."""
        ids = {}
        out = {}
        for k, p in enumerate("lro"):
            row, wires, cids = [0], [], []
            for con in r1cs.constraints:
                for i, c in con[k]:
                    wires.append(i)
                    cids.append(ids.setdefault(c % R_MOD, len(ids)))
                row.append(len(wires))
            out[p + "_row"] = np.array(row, dtype=np.uint64)
            out[p + "_wire"] = np.array(wires, dtype=np.uint32)
            out[p + "_coeff"] = np.array(cids, dtype=np.uint32)
        table = sorted(ids, key=ids.get)
        return SparseR1CS(r1cs.nb_wires, r1cs.nb_public, fr_array(table) if table else np.zeros((0, 4), np.uint64),
                          private_committed=np.array(r1cs.private_committed, dtype=np.uint32),
                          public_committed=list(r1cs.public_committed), commitment_wire=r1cs.commitment_wire, **out)

    @functools.cached_property
    def constraints(self):
        """[(L, R, O)] with [(wire, coeff)] terms, as R1CS.constraints (what solve_abc reads).  Built from the arrays on
        first access and kept: the host prover walks it once per solve_abc, and rebuilding it per access costs seconds
        at 2^16 constraints.  Change the arrays of a SparseR1CS before that first access, not after."""
        cf = [_fr_from(c) for c in np.asarray(self.coeffs, dtype=np.uint64).reshape(-1, 4)]
        mats = []
        for p in "lro":
            row, wire, cid = getattr(self, p + "_row"), getattr(self, p + "_wire").tolist(), getattr(self, p + "_coeff").tolist()
            mats.append([[(wire[e], cf[cid[e]]) for e in range(int(row[j]), int(row[j + 1]))] for j in range(len(row) - 1)])
        return list(zip(*mats))


def _fr_from(limbs):
    v = int(limbs[0]) | int(limbs[1]) << 64 | int(limbs[2]) << 128 | int(limbs[3]) << 192
    return v * pow(_MONT, -1, R_MOD) % R_MOD


def _lc(lc, w):
    return sum(c * w[i] for i, c in lc) % R_MOD


def solve_abc(r1cs, w):
    """solution.A/B/C of gnark's r1cs.Solve for an already complete assignment."""
    return ([_lc(L, w) for L, _, _ in r1cs.constraints],
            [_lc(Rr, w) for _, Rr, _ in r1cs.constraints],
            [_lc(O, w) for _, _, O in r1cs.constraints])


# ---------------------------------------------------------------- keys / proof (gnark field names)
@dataclass
class PedersenProvingKey:          # gnark-crypto fr/pedersen.ProvingKey
    Basis: np.ndarray
    BasisExpSigma: np.ndarray
    basis_dev: object = None
    basis_exp_sigma_dev: object = None


@dataclass
class ProvingKey:                  # groth16_bn254.ProvingKey
    log2_domain: int
    G1_Alpha: np.ndarray
    G1_Beta: np.ndarray
    G1_Delta: np.ndarray
    G1_A: object
    G1_B: object
    G1_Z: object
    G1_K: object
    G2_Beta: np.ndarray
    G2_Delta: np.ndarray
    G2_B: object
    InfinityA: np.ndarray
    InfinityB: np.ndarray
    k_skip: np.ndarray
    CommitmentKeys: list = field(default_factory=list)
    _dev: object = None            # device handle, filled lazily on first Prove (like gnark's icicle pk)
    _ctx: object = None
    _owned: list = field(default_factory=list)   # resident vectors DeviceSetup made; free() releases them

    def device_handle(self, ctx, precompute=False):
        """precompute=True: attach window tables to the resident point vectors at upload time
        (b200g16_bases_precompute) — more HBM, fewer additions per MSM, identical proofs."""
        if self._dev is None:
            self._dev = ctx.pk_upload(self.log2_domain, len(self.InfinityA), self.G1_A, self.G1_B, self.G1_K,
                                      self.G1_Z, self.G2_B, self.G1_Alpha, self.G1_Beta, self.G1_Delta,
                                      self.G2_Beta, self.G2_Delta, self.InfinityA, self.InfinityB, self.k_skip,
                                      precompute=precompute)
            self._ctx = ctx
        return self._dev

    def free(self):
        if self._dev is not None:
            self._ctx.pk_free(self._dev)
            self._dev = None
        for ck in self.CommitmentKeys:
            for b in (ck.basis_dev, ck.basis_exp_sigma_dev):
                if b is not None:
                    b.free()
            ck.basis_dev = ck.basis_exp_sigma_dev = None
        for b in self._owned:
            b.free()
        self._owned = []


@dataclass
class VerifyingKey:                # groth16_bn254.VerifyingKey
    G1_Alpha: np.ndarray
    G1_K: np.ndarray
    G2_Beta: np.ndarray
    G2_Gamma: np.ndarray
    G2_Delta: np.ndarray
    PedersenG: np.ndarray = None
    PedersenGSigmaNeg: np.ndarray = None
    PublicAndCommitmentCommitted: list = field(default_factory=list)
    has_commitment: bool = False
    G1_Beta: np.ndarray = None     # carried by gnark's vk and its wire format; Verify does not use them
    G1_Delta: np.ndarray = None


@dataclass
class Proof:                       # groth16_bn254.Proof
    Ar: np.ndarray
    Krs: np.ndarray
    Bs: np.ndarray
    Commitments: list = field(default_factory=list)
    CommitmentPok: np.ndarray = None
    debug: dict = field(default_factory=dict)   # intermediate MSM outputs, h (parity checks)


def proof_write_to(ctx, proof, raw=False):
    """(*Proof).WriteTo (raw=False, compressed points) / WriteRawTo (raw=True) -> bytes:
    Ar | Bs | Krs | uint32 len(Commitments) | Commitments... | CommitmentPok
    (gnark backend/groth16/bn254/marshal.go; point encodings by b200g16_g1/g2_encode)."""
    pok = proof.CommitmentPok if proof.CommitmentPok is not None else np.zeros(8, dtype=np.uint64)
    g1 = np.stack([np.asarray(p, dtype=np.uint64).reshape(8) for p in [proof.Ar, proof.Krs, *proof.Commitments, pok]])
    e1 = ctx.encode_points(g1, group=1, raw=raw)
    e2 = ctx.encode_points(np.asarray(proof.Bs, dtype=np.uint64).reshape(1, 16), group=2, raw=raw)
    k = len(proof.Commitments)
    return (e1[0].tobytes() + e2[0].tobytes() + e1[1].tobytes() + k.to_bytes(4, "big")
            + b"".join(e1[2 + i].tobytes() for i in range(k)) + e1[2 + k].tobytes())


class _PointReader:
    """gnark-crypto's Decoder reads every point by its own flag bits: 0b00 = uncompressed record (64 / 128 bytes,
    all zero = infinity), anything else = compressed record (32 / 64 bytes, 0b01 = infinity).  Records are
    collected while the stream is walked and decoded in two GPU batches (compressed / uncompressed)."""

    def __init__(self, data, what):
        self.data, self.o, self.what, self.items = bytes(data), 0, what, []

    def take(self, k):
        if self.o + k > len(self.data):
            raise ValueError(f"{self.what}: short buffer")
        v = self.data[self.o:self.o + k]
        self.o += k
        return v

    def u32(self):
        return int.from_bytes(self.take(4), "big")

    def point(self, group):
        """Registers the next point; returns its index into the result of decode()."""
        if self.o >= len(self.data):
            raise ValueError(f"{self.what}: short buffer")
        raw = (self.data[self.o] & 0xC0) == 0
        size = (32 if group == 1 else 64) * (2 if raw else 1)
        self.items.append((group, raw, self.take(size)))
        return len(self.items) - 1

    def decode(self, ctx):
        out = [None] * len(self.items)
        for group in (1, 2):
            for raw in (False, True):
                idx = [i for i, it in enumerate(self.items) if it[0] == group and it[1] == raw]
                if not idx:
                    continue
                pts, ok = ctx.decode_points(b"".join(self.items[i][2] for i in idx), group=group, raw=raw)
                if not ok.all():
                    raise ValueError(f"{self.what}: invalid point encoding")
                for j, i in enumerate(idx):
                    out[i] = pts[j]
        return out


def proof_read_from(ctx, data, raw=None):
    """(*Proof).ReadFrom -> Proof; raises ValueError on an invalid encoding (gnark returns the decoder's error).
    Compressed and raw streams are both accepted (per-point flag bits, like gnark-crypto's Decoder); `raw` is
    ignored and kept for the callers of the previous signature."""
    rd = _PointReader(data, "groth16.Proof.ReadFrom")
    ar, bs, krs = rd.point(1), rd.point(2), rd.point(1)
    k = rd.u32()
    if k > (len(rd.data) - rd.o) // 32:
        raise ValueError("groth16.Proof.ReadFrom: short buffer")
    coms = [rd.point(1) for _ in range(k)]
    pok = rd.point(1)
    p = rd.decode(ctx)
    return Proof(p[ar], p[krs], p[bs], [p[i] for i in coms], p[pok])


def vk_write_to(ctx, vk, raw=False):
    """(*VerifyingKey).WriteTo / WriteRawTo -> bytes (gnark backend/groth16/bn254/marshal.go, as recalled):
    G1.Alpha | G1.Beta | G2.Beta | G2.Gamma | G1.Delta | G2.Delta | u32 len(K) | K... |
    PublicAndCommitmentCommitted as [][]uint64 (u32 outer length, then u32 length + big-endian u64s each) |
    u32 #commitment keys | per key: pedersen G | GSigmaNeg (G2)."""
    zero1 = np.zeros(8, dtype=np.uint64)
    g1 = np.stack([np.asarray(p if p is not None else zero1, dtype=np.uint64).reshape(8)
                   for p in [vk.G1_Alpha, vk.G1_Beta, vk.G1_Delta]] + [np.asarray(k, dtype=np.uint64).reshape(8) for k in vk.G1_K])
    g2_list = [vk.G2_Beta, vk.G2_Gamma, vk.G2_Delta] + ([vk.PedersenG, vk.PedersenGSigmaNeg] if vk.has_commitment else [])
    e1 = ctx.encode_points(g1, group=1, raw=raw)
    e2 = ctx.encode_points(np.stack([np.asarray(q, dtype=np.uint64).reshape(16) for q in g2_list]), group=2, raw=raw)
    out = e1[0].tobytes() + e1[1].tobytes() + e2[0].tobytes() + e2[1].tobytes() + e1[2].tobytes() + e2[2].tobytes()
    out += len(vk.G1_K).to_bytes(4, "big") + b"".join(e1[3 + i].tobytes() for i in range(len(vk.G1_K)))
    groups = [list(vk.PublicAndCommitmentCommitted)] if vk.has_commitment else []
    out += len(groups).to_bytes(4, "big")
    for g in groups:
        out += len(g).to_bytes(4, "big") + b"".join(int(x).to_bytes(8, "big") for x in g)
    out += (1 if vk.has_commitment else 0).to_bytes(4, "big")
    if vk.has_commitment:
        out += e2[3].tobytes() + e2[4].tobytes()
    return out


def vk_read_from(ctx, data, raw=None):
    """(*VerifyingKey).ReadFrom -> VerifyingKey; raises ValueError on an invalid encoding.  Accepts compressed
    and raw streams (per-point flag bits); `raw` is ignored."""
    rd = _PointReader(data, "groth16.VerifyingKey.ReadFrom")
    a1, b1, b2, g2, d1, d2 = rd.point(1), rd.point(1), rd.point(2), rd.point(2), rd.point(1), rd.point(2)
    nk = rd.u32()
    if nk > (len(rd.data) - rd.o) // 32:
        raise ValueError("groth16.VerifyingKey.ReadFrom: short buffer")
    ks = [rd.point(1) for _ in range(nk)]
    groups = []
    for _ in range(rd.u32()):
        m = rd.u32()
        groups.append([int.from_bytes(rd.take(8), "big") for _ in range(m)])
    nck = rd.u32()
    if nck > 1 or nck != len(groups):
        raise ValueError("groth16.VerifyingKey.ReadFrom: this backend supports at most one commitment")
    ped = [rd.point(2), rd.point(2)] if nck else []
    p = rd.decode(ctx)
    vk = VerifyingKey(p[a1], np.stack([p[i] for i in ks]) if ks else np.zeros((0, 8), np.uint64), p[b2], p[g2], p[d2],
                      G1_Beta=p[b1], G1_Delta=p[d1])
    if nck:
        vk.PedersenG, vk.PedersenGSigmaNeg = p[ped[0]], p[ped[1]]
        vk.PublicAndCommitmentCommitted = groups[0]
        vk.has_commitment = True
    return vk


# ---------------------------------------------------------------- ProvingKey wire format
ROOT_2_28 = 19103219067921713944291392827692070036145651957329286315305642004821462161904


def domain_write_to(log2n, with_precompute=True):
    """(*fft.Domain).WriteTo (gnark-crypto ecc/bn254/fr/fft/domain.go, as recalled): Cardinality u64 | CardinalityInv |
    Generator | GeneratorInv | FrMultiplicativeGen | FrMultiplicativeGenInv (fr.Element = 32 bytes big-endian,
    canonical) | withPrecompute (1 byte)."""
    n = 1 << log2n
    gen = pow(ROOT_2_28, 1 << (28 - log2n), R_MOD)
    vals = [pow(n, -1, R_MOD), gen, pow(gen, -1, R_MOD), 5, pow(5, -1, R_MOD)]
    return n.to_bytes(8, "big") + b"".join(v.to_bytes(32, "big") for v in vals) + bytes([1 if with_precompute else 0])


def domain_read_from(rd):
    n = int.from_bytes(rd.take(8), "big")
    vals = [int.from_bytes(rd.take(32), "big") for _ in range(5)]
    rd.take(1)
    if n == 0 or n & (n - 1) or n > (1 << 28):
        raise ValueError("fft.Domain.ReadFrom: cardinality is not a power of two <= 2^28")
    log2n = n.bit_length() - 1
    if domain_write_to(log2n)[8:-1] != b"".join(v.to_bytes(32, "big") for v in vals):
        raise ValueError("fft.Domain.ReadFrom: generator / inverses do not belong to this cardinality")
    return log2n


def pk_write_to(ctx, pk, raw=False):
    """(*ProvingKey).WriteTo / WriteRawTo (gnark backend/groth16/bn254/marshal.go, as recalled):
    Domain | G1.Alpha | G1.Beta | G1.Delta | G1.A | G1.B | G1.Z | G1.K | G2.Beta | G2.Delta | G2.B | nbWires u64 |
    NbInfinityA u64 | NbInfinityB u64 | InfinityA []bool (nbWires bytes, no length) | InfinityB | u32 #commitment keys |
    per key: pedersen Basis | BasisExpSigma.  Point slices: u32 length + points.  The point encodings run batched on
    the GPU (b200g16_g1/g2_encode)."""
    def host(v):
        return v.download() if hasattr(v, "download") else np.asarray(v, dtype=np.uint64)
    g1_vecs = [host(v).reshape(-1, 8) for v in (pk.G1_A, pk.G1_B, pk.G1_Z, pk.G1_K)]
    ped = [host(x).reshape(-1, 8) for ck in pk.CommitmentKeys for x in (ck.Basis, ck.BasisExpSigma)]
    singles = np.stack([np.asarray(p, dtype=np.uint64).reshape(8) for p in (pk.G1_Alpha, pk.G1_Beta, pk.G1_Delta)])
    allg1 = np.concatenate([singles] + g1_vecs + ped)
    e1 = ctx.encode_points(allg1, group=1, raw=raw)
    g2 = np.concatenate([np.stack([np.asarray(pk.G2_Beta, np.uint64).reshape(16), np.asarray(pk.G2_Delta, np.uint64).reshape(16)]),
                         host(pk.G2_B).reshape(-1, 16)])
    e2 = ctx.encode_points(g2, group=2, raw=raw)
    out = [domain_write_to(pk.log2_domain), e1[0].tobytes(), e1[1].tobytes(), e1[2].tobytes()]
    o = 3
    for v in g1_vecs:
        out += [len(v).to_bytes(4, "big"), e1[o:o + len(v)].tobytes()]
        o += len(v)
    out += [e2[0].tobytes(), e2[1].tobytes(), (len(g2) - 2).to_bytes(4, "big"), e2[2:].tobytes()]
    ia, ib = np.asarray(pk.InfinityA, dtype=np.uint8), np.asarray(pk.InfinityB, dtype=np.uint8)
    out += [len(ia).to_bytes(8, "big"), int(ia.sum()).to_bytes(8, "big"), int(ib.sum()).to_bytes(8, "big"),
            (ia != 0).astype(np.uint8).tobytes(), (ib != 0).astype(np.uint8).tobytes(), len(pk.CommitmentKeys).to_bytes(4, "big")]
    for v in ped:
        out += [len(v).to_bytes(4, "big"), e1[o:o + len(v)].tobytes()]
        o += len(v)
    return b"".join(out)


def pk_read_from(ctx, data, k_skip=None):
    """(*ProvingKey).ReadFrom -> ProvingKey (compressed or raw stream, per-point flag bits).  A compressed key costs one
    square root per point: decoded in GPU batches.  k_skip (public + committed + commitment wires; gnark derives it from
    the constraint system at prove time, it is not part of the key) may be given here or set on the result later."""
    rd = _PointReader(data, "groth16.ProvingKey.ReadFrom")
    log2n = domain_read_from(rd)

    def vec(group):
        n = rd.u32()
        if n > (len(rd.data) - rd.o) // 32:
            raise ValueError("groth16.ProvingKey.ReadFrom: short buffer")
        return [rd.point(group) for _ in range(n)]
    alpha, beta, delta = rd.point(1), rd.point(1), rd.point(1)
    A, B, Z, K = vec(1), vec(1), vec(1), vec(1)
    beta2, delta2 = rd.point(2), rd.point(2)
    B2 = vec(2)
    nb_wires = int.from_bytes(rd.take(8), "big")
    nia, nib = int.from_bytes(rd.take(8), "big"), int.from_bytes(rd.take(8), "big")
    if 2 * nb_wires > len(rd.data) - rd.o:
        raise ValueError("groth16.ProvingKey.ReadFrom: short buffer")
    ia = np.frombuffer(rd.take(nb_wires), dtype=np.uint8).copy()
    ib = np.frombuffer(rd.take(nb_wires), dtype=np.uint8).copy()
    if int((ia != 0).sum()) != nia or int((ib != 0).sum()) != nib or len(A) != nb_wires - nia or len(B) != nb_wires - nib or len(B2) != len(B):
        raise ValueError("groth16.ProvingKey.ReadFrom: infinity flags do not match the point vectors")
    if len(Z) + 1 != (1 << log2n):
        raise ValueError("groth16.ProvingKey.ReadFrom: len(G1.Z) != N - 1")
    cks = [(vec(1), vec(1)) for _ in range(rd.u32())]
    p = rd.decode(ctx)

    def arr(idx, w):
        return np.stack([p[i] for i in idx]) if idx else np.zeros((0, w), dtype=np.uint64)
    pk = ProvingKey(log2n, p[alpha], p[beta], p[delta], arr(A, 8), arr(B, 8), arr(Z, 8), arr(K, 8), p[beta2], p[delta2],
                    arr(B2, 16), ia, ib, None if k_skip is None else np.asarray(k_skip, dtype=np.uint8),
                    [PedersenProvingKey(arr(b, 8), arr(bs, 8)) for b, bs in cks])
    return pk


@dataclass
class ToxicWaste:
    tau: int
    alpha: int
    beta: int
    gamma: int
    delta: int
    sigma: int

    @staticmethod
    def random():
        return ToxicWaste(*[1 + secrets.randbelow(R_MOD - 1) for _ in range(6)])


# ---------------------------------------------------------------- hash_to_field (RFC 9380, SHA-256)
def _expand_xmd(msg, dst, length):
    ell = (length + 31) // 32
    dstp = dst + bytes([len(dst)])
    b0 = hashlib.sha256(bytes(64) + msg + length.to_bytes(2, "big") + b"\x00" + dstp).digest()
    bi = hashlib.sha256(b0 + b"\x01" + dstp).digest()
    out = bi
    for i in range(2, ell + 1):
        bi = hashlib.sha256(bytes(x ^ y for x, y in zip(b0, bi)) + bytes([i]) + dstp).digest()
        out += bi
    return out[:length]


def commitment_challenge(commitment_limbs, public_committed_values):
    """gnark prove.go: hash_to_field("bsb22-commitment")(commitment.Marshal() || committed publics)."""
    c = np.asarray(commitment_limbs, dtype=np.uint64)
    if not c.any():
        raw = bytes(64)             # Marshal() = RawBytes(): the uncompressed point at infinity is all zero on bn254
    else:
        raw = _fp_from(c[:4]).to_bytes(32, "big") + _fp_from(c[4:]).to_bytes(32, "big")
    msg = raw + b"".join(int(v % R_MOD).to_bytes(32, "big") for v in public_committed_values)
    return int.from_bytes(_expand_xmd(msg, b"bsb22-commitment", 48), "big") % R_MOD


# ---------------------------------------------------------------- Setup
def _bitrev(i, logn):
    return int(format(i, "0%db" % logn)[::-1], 2) if logn else 0


def Setup(ctx, r1cs, toxic=None):
    """groth16.Setup(ccs) -> (pk, vk).  `toxic` may be fixed for reproducible tests."""
    tw = toxic or ToxicWaste.random()
    m = len(r1cs.constraints)
    logn = max(m - 1, 0).bit_length()
    n = 1 << logn
    w_gen = pow(_ROOT_2_28, 1 << (28 - logn), R_MOD)
    nw = r1cs.nb_wires
    A, B, Cc = [0] * nw, [0] * nw, [0] * nw
    zn = (pow(tw.tau, n, R_MOD) - 1) * pow(n, -1, R_MOD) % R_MOD
    wj = 1
    for L, Rr, O in r1cs.constraints:           # setupABC: Lagrange basis at tau
        lag = zn * wj % R_MOD * pow((tw.tau - wj) % R_MOD, -1, R_MOD) % R_MOD
        for i, c in L:
            A[i] = (A[i] + c * lag) % R_MOD
        for i, c in Rr:
            B[i] = (B[i] + c * lag) % R_MOD
        for i, c in O:
            Cc[i] = (Cc[i] + c * lag) % R_MOD
        wj = wj * w_gen % R_MOD
    gi, di = pow(tw.gamma, -1, R_MOD), pow(tw.delta, -1, R_MOD)
    committed = set(r1cs.private_committed)
    kval = lambda i: (tw.beta * A[i] + tw.alpha * B[i] + Cc[i]) % R_MOD
    k_priv, k_pub, k_ped = [], [], []
    k_skip = np.ones(nw, dtype=np.uint8)
    for i in range(nw):
        if i < r1cs.nb_public:
            k_pub.append(kval(i) * gi % R_MOD)
        elif i in committed or i == r1cs.commitment_wire:
            continue
        else:
            k_priv.append(kval(i) * di % R_MOD)
            k_skip[i] = 0
    if r1cs.commitment_wire >= 0:
        k_pub.append(kval(r1cs.commitment_wire) * gi % R_MOD)
        k_ped = [kval(i) * gi % R_MOD for i in r1cs.private_committed]
    zdt = (pow(tw.tau, n, R_MOD) - 1) * di % R_MOD
    zs, t = [], zdt
    for _ in range(n):
        zs.append(t)
        t = t * tw.tau % R_MOD
    zs = [zs[_bitrev(i, logn)] for i in range(n)][:n - 1]
    inf_a = np.array([a == 0 for a in A], dtype=np.uint8)
    inf_b = np.array([b == 0 for b in B], dtype=np.uint8)
    sa, sb = [a for a in A if a], [b for b in B if b]
    g1 = g1_point(G1_GEN)
    g2 = g2_point(G2_GEN)
    scal = sa + sb + zs + k_priv + k_pub + k_ped + [tw.alpha, tw.beta, tw.delta]
    pts = ctx.fixed_base_mul(g1, fr_array(scal), group=1)      # BatchScalarMultiplicationG1
    o = 0

    def take(k):
        nonlocal o
        v = pts[o:o + k].copy()
        o += k
        return v
    pkA, pkB, pkZ, pkK, vkK, ped = take(len(sa)), take(len(sb)), take(n - 1), take(len(k_priv)), \
        take(len(k_pub)), take(len(k_ped))
    alpha1, beta1, delta1 = take(3)
    pts2 = ctx.fixed_base_mul(g2, fr_array(sb + [tw.beta, tw.delta, tw.gamma]), group=2)
    pkB2 = pts2[:len(sb)].copy()
    beta2, delta2, gamma2 = pts2[len(sb)], pts2[len(sb) + 1], pts2[len(sb) + 2]
    pk = ProvingKey(logn, alpha1, beta1, delta1, pkA, pkB, pkZ, pkK, beta2, delta2, pkB2, inf_a, inf_b, k_skip)
    vk = VerifyingKey(alpha1, vkK, beta2, gamma2, delta2, G1_Beta=beta1, G1_Delta=delta1)
    if r1cs.commitment_wire >= 0:
        # pedersen.Setup: BasisExpSigma = sigma * Basis; vk = (G, -sigma * G)
        bes = ctx.fixed_base_mul(g1, fr_array([k * tw.sigma % R_MOD for k in k_ped]), group=1)
        pk.CommitmentKeys = [PedersenProvingKey(ped, bes)]
        vk.PedersenG = g2
        vk.PedersenGSigmaNeg = ctx.fixed_base_mul(g2, fr_array([(-tw.sigma) % R_MOD]), group=2)[0]
        vk.PublicAndCommitmentCommitted = list(r1cs.public_committed)
        vk.has_commitment = True
    return pk, vk


def DeviceSetup(ctx, r1cs, toxic=None, precompute=False):
    """groth16.Setup(ccs) -> (pk, vk) computed on the GPU by b200g16_setup: the same key as Setup for the same toxic
    waste, bit for bit.  r1cs: an R1CS or a SparseR1CS.  The proving key's point vectors stay resident (G1_A, G1_B,
    G1_K, G1_Z, G2_B and the Pedersen basis_dev / basis_exp_sigma_dev are Bases); Prove, BatchProve, pk_write_to and
    the verifier take the key as it is.  precompute=True attaches window tables to the five prove vectors.
    pk.free() releases them."""
    tw = toxic or ToxicWaste.random()
    sp = r1cs if isinstance(r1cs, SparseR1CS) else SparseR1CS.from_r1cs(r1cs)
    t = fr_array([tw.tau, tw.alpha, tw.beta, tw.gamma, tw.delta, tw.sigma])
    o = ctx.setup(sp, *t)
    owned = [o[n] for n in lib.SETUP_VECTORS if o[n] is not None]
    vk_k = o["vk_k"].download()
    o["vk_k"].free()
    owned.remove(o["vk_k"])
    if precompute:
        for n in ("a", "b", "k", "z", "b2"):
            if len(o[n]):
                o[n].precompute(0)
    pk = ProvingKey(o["log2_domain"], o["g1_alpha"], o["g1_beta"], o["g1_delta"], o["a"], o["b"], o["z"], o["k"],
                    o["g2_beta"], o["g2_delta"], o["b2"], o["infinity_a"], o["infinity_b"], o["k_skip"], _owned=owned)
    vk = VerifyingKey(o["g1_alpha"], vk_k, o["g2_beta"], o["g2_gamma"], o["g2_delta"], G1_Beta=o["g1_beta"],
                      G1_Delta=o["g1_delta"])
    if sp.commitment_wire >= 0:
        basis, bes = o["ped_basis"], o["ped_basis_exp_sigma"]
        pk.CommitmentKeys = [PedersenProvingKey(basis, bes, basis_dev=basis, basis_exp_sigma_dev=bes)]
        owned.remove(basis)
        owned.remove(bes)
        vk.PedersenG, vk.PedersenGSigmaNeg = o["ped_g"], o["ped_g_sigma_neg"]
        vk.PublicAndCommitmentCommitted = list(sp.public_committed)
        vk.has_commitment = True
    return pk, vk


# ---------------------------------------------------------------- Prove
def Prove(ctx, r1cs, pk, witness, r=None, s=None, resolve=None, want_h=False):
    """groth16.Prove(ccs, pk, fullWitness, opts...).

    witness: full wire assignment (list of ints); for a circuit with a commitment the commitment
    wire is filled here, exactly where gnark's solver would call the BSB22 hint: Pedersen-commit to
    the committed wires on the GPU, hash, write the challenge; `resolve(witness)` then lets the
    caller (standing in for the solver) finish wires that depend on the challenge.
    r, s: blinding scalars; sampled like gnark does when omitted."""
    w = list(witness)
    proof_commitments, pok = [], None
    if r1cs.commitment_wire >= 0:
        ck = pk.CommitmentKeys[0]
        if ck.basis_dev is None:
            ck.basis_dev = ctx.upload_g1(ck.Basis)
            ck.basis_exp_sigma_dev = ctx.upload_g1(ck.BasisExpSigma)
        vals = fr_array([w[i] for i in r1cs.private_committed])
        com = ctx.msm(ck.basis_dev, vals)                        # pedersen Commit (inside Solve)
        w[r1cs.commitment_wire] = commitment_challenge(com, [w[i] for i in r1cs.public_committed])
        if resolve is not None:
            resolve(w)
        # pedersen ProveKnowledge (1 commitment: fold = id): enqueued now, collected after the prove's own MSMs
        pok_ticket = ctx.msm_begin(ck.basis_exp_sigma_dev, vals)
        proof_commitments = [com]
    a, b, c = solve_abc(r1cs, w)
    r = secrets.randbelow(R_MOD) if r is None else r
    s = secrets.randbelow(R_MOD) if s is None else s
    out, h = ctx.prove(pk.device_handle(ctx), fr_array(w), fr_array(a), fr_array(b), fr_array(c),
                       fr_array([r])[0], fr_array([s])[0], want_h=want_h, log2_domain=pk.log2_domain)
    if r1cs.commitment_wire >= 0:
        pok = ctx.msm_end(pok_ticket)
    dbg = dict(out)
    dbg["h"] = h
    dbg["witness"] = w
    return Proof(out["ar"], out["krs"], out["bs"], proof_commitments, pok, dbg)


def BatchProve(ctx, r1cs, pk, witnesses, rs=None, ss=None, resolve=None):
    """k proofs of one circuit in one b200g16_prove_batch call -> list of k Proofs, proof j equal to
    Prove(ctx, r1cs, pk, witnesses[j], rs[j], ss[j], resolve).

    With a commitment, the Pedersen Commit of all k witnesses is one batch MSM over the commitment basis; each
    witness's commitment wire is then filled from its own commitment (and `resolve` finishes that witness), and
    ProveKnowledge is one batch MSM over BasisExpSigma.  rs, ss: k blinding scalars each; drawn like Prove draws
    them when omitted."""
    ws = [list(w) for w in witnesses]
    k = len(ws)
    rs = [secrets.randbelow(R_MOD) for _ in range(k)] if rs is None else list(rs)
    ss = [secrets.randbelow(R_MOD) for _ in range(k)] if ss is None else list(ss)
    if len(rs) != k or len(ss) != k:
        raise ValueError("groth16.BatchProve: one r and one s per witness")
    if k == 0:
        return []
    coms, poks = [[] for _ in range(k)], [None] * k
    if r1cs.commitment_wire >= 0:
        ck = pk.CommitmentKeys[0]
        if ck.basis_dev is None:
            ck.basis_dev = ctx.upload_g1(ck.Basis)
            ck.basis_exp_sigma_dev = ctx.upload_g1(ck.BasisExpSigma)
        vals = np.stack([fr_array([w[i] for i in r1cs.private_committed]).reshape(-1, 4) for w in ws])
        com = ctx.msm_batch(ck.basis_dev, vals)                     # pedersen Commit of every witness
        for j, w in enumerate(ws):
            w[r1cs.commitment_wire] = commitment_challenge(com[j], [w[i] for i in r1cs.public_committed])
            if resolve is not None:
                resolve(w)
        pok = ctx.msm_batch(ck.basis_exp_sigma_dev, vals)           # pedersen ProveKnowledge of every witness
        coms = [[com[j]] for j in range(k)]
        poks = [pok[j] for j in range(k)]
    abc = [solve_abc(r1cs, w) for w in ws]
    outs = ctx.prove_batch(pk.device_handle(ctx), np.stack([fr_array(w).reshape(-1, 4) for w in ws]),
                           *[np.stack([fr_array(t[i]).reshape(-1, 4) for t in abc]) for i in range(3)],
                           fr_array(rs).reshape(k, 4), fr_array(ss).reshape(k, 4))
    proofs = []
    for j, out in enumerate(outs):
        dbg = dict(out)
        dbg["witness"] = ws[j]
        proofs.append(Proof(out["ar"], out["krs"], out["bs"], coms[j], poks[j], dbg))
    return proofs


class GroupProvingKey:
    """A ProvingKey (from Setup or DeviceSetup) on every device of a lib.Group, for GroupBatchProve.

    The key is first made resident on one device: where its vectors already are (DeviceSetup, or a key Prove has
    uploaded), else on `ctx` (default: the group's first member).  It is then replicated over the group
    (b200g16_group_pk_replicate: device-to-device copies, window tables included).  With a commitment, the Pedersen
    bases reach each member's device the same way (b200g16_bases_copy).  free() releases the replica and the copies,
    never pk itself; call it before the group is closed."""

    def __init__(self, group, pk, ctx=None, precompute=False):
        self.group, self.pk = group, pk
        if pk._dev is not None:
            src_ctx = pk._ctx
        elif isinstance(pk.G1_A, lib.Bases):
            src_ctx = pk.G1_A.ctx
        else:
            src_ctx = ctx if ctx is not None else group.ctx(0)
        self.ctxs = [group.ctx(i) for i in range(len(group))]
        self.handle = group.pk_replicate(pk.device_handle(src_ctx, precompute=precompute))
        self._copies = []
        self.pedersen = None        # per member: (Basis, BasisExpSigma) on its device
        if pk.CommitmentKeys:
            ck = pk.CommitmentKeys[0]
            if ck.basis_dev is None:
                ck.basis_dev = src_ctx.upload_g1(ck.Basis)
                ck.basis_exp_sigma_dev = src_ctx.upload_g1(ck.BasisExpSigma)
            on_device = {}
            for c in self.ctxs:
                if c.device not in on_device:
                    if c.device == ck.basis_dev.ctx.device:
                        on_device[c.device] = (ck.basis_dev, ck.basis_exp_sigma_dev)
                    else:
                        on_device[c.device] = (c.bases_copy(ck.basis_dev), c.bases_copy(ck.basis_exp_sigma_dev))
                        self._copies += on_device[c.device]
            self.pedersen = [on_device[c.device] for c in self.ctxs]

    @property
    def log2_domain(self):
        return self.pk.log2_domain

    def free(self):
        if self.handle is not None:
            self.group.pk_free(self.handle)
            self.handle = None
        for b in self._copies:
            b.free()
        self._copies = []
        self.pedersen = None


def _ranges(k, n):
    """Contiguous ranges of k items over n members, sizes differing by at most one (the library's split)."""
    base, rem = divmod(k, n)
    out, lo = [], 0
    for i in range(n):
        hi = lo + base + (1 if i < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def _on_members(ctxs, k, fn):
    """fn(i, lo, hi) for every member with a non-empty range, one thread per member (the library calls release the
    GIL); the first exception is raised."""
    import threading
    errs = []

    def run(i, lo, hi):
        try:
            fn(i, lo, hi)
        except BaseException as e:   # noqa: BLE001 - re-raised below
            errs.append(e)
    th = [threading.Thread(target=run, args=(i, lo, hi)) for i, (lo, hi) in enumerate(_ranges(k, len(ctxs))) if hi > lo]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]


def GroupBatchProve(group, r1cs, gpk, witnesses, rs=None, ss=None, resolve=None):
    """BatchProve over the devices of a group with a GroupProvingKey: the same k proofs, bit for bit, in one
    b200g16_group_prove_batch call (contiguous ranges of proofs per member).  With a commitment, the Pedersen Commit
    and ProveKnowledge batch MSMs are split over the members the same way, one thread each."""
    ws = [list(w) for w in witnesses]
    k = len(ws)
    rs = [secrets.randbelow(R_MOD) for _ in range(k)] if rs is None else list(rs)
    ss = [secrets.randbelow(R_MOD) for _ in range(k)] if ss is None else list(ss)
    if len(rs) != k or len(ss) != k:
        raise ValueError("groth16.GroupBatchProve: one r and one s per witness")
    if k == 0:
        return []
    coms, poks = [[] for _ in range(k)], [None] * k
    if r1cs.commitment_wire >= 0:
        vals = np.stack([fr_array([w[i] for i in r1cs.private_committed]).reshape(-1, 4) for w in ws])
        com, pok = [None] * k, [None] * k

        def commit(i, lo, hi):
            com[lo:hi] = list(gpk.ctxs[i].msm_batch(gpk.pedersen[i][0], vals[lo:hi]))
        _on_members(gpk.ctxs, k, commit)                            # pedersen Commit of every witness
        for j, w in enumerate(ws):
            w[r1cs.commitment_wire] = commitment_challenge(com[j], [w[i] for i in r1cs.public_committed])
            if resolve is not None:
                resolve(w)

        def knowledge(i, lo, hi):
            pok[lo:hi] = list(gpk.ctxs[i].msm_batch(gpk.pedersen[i][1], vals[lo:hi]))
        _on_members(gpk.ctxs, k, knowledge)                         # pedersen ProveKnowledge of every witness
        coms = [[com[j]] for j in range(k)]
        poks = pok
    abc = [solve_abc(r1cs, w) for w in ws]
    outs = group.prove_batch(gpk.handle, np.stack([fr_array(w).reshape(-1, 4) for w in ws]),
                             *[np.stack([fr_array(t[i]).reshape(-1, 4) for t in abc]) for i in range(3)],
                             fr_array(rs).reshape(k, 4), fr_array(ss).reshape(k, 4))
    proofs = []
    for j, out in enumerate(outs):
        dbg = dict(out)
        dbg["witness"] = ws[j]
        proofs.append(Proof(out["ar"], out["krs"], out["bs"], coms[j], poks[j], dbg))
    return proofs


def _verify_inputs(proof, vk, public_witness):
    """The public inputs b200g16_verify takes for one proof (the public witness, then the BSB22 challenge when the
    circuit has a commitment) and the proof's commitment and proof of knowledge (None without one)."""
    pub = [int(v) % R_MOD for v in public_witness]
    com = pok = None
    if vk.has_commitment:
        if not proof.Commitments or proof.CommitmentPok is None:
            raise ValueError("groth16.Verify: proof carries no commitment but the circuit has one")
        com, pok = proof.Commitments[0], proof.CommitmentPok
        # PublicAndCommitmentCommitted holds wire indexes (wire 0 = the constant one)
        committed = [1 if i == 0 else pub[i - 1] for i in vk.PublicAndCommitmentCommitted]
        pub.append(commitment_challenge(com, committed))
    return pub, com, pok


def Verify(ctx, proof, vk, public_witness):
    """groth16.Verify(proof, vk, publicWitness) -> None, raises on an invalid proof (gnark returns
    an error).  public_witness: values of the public wires WITHOUT the constant-one wire, as in
    gnark's witness.Public().  Runs b200g16_verify: the public-input MSM and the pairing product
    on the GPU; only the BSB22 challenge hash (SHA-256 over ~100 bytes) is computed here."""
    pub, com, pok = _verify_inputs(proof, vk, public_witness)
    ok = ctx.verify(vk.G1_Alpha, vk.G2_Beta, vk.G2_Gamma, vk.G2_Delta, vk.G1_K, proof.Ar, proof.Bs, proof.Krs,
                    fr_array(pub) if pub else np.zeros((0, 4), dtype=np.uint64), commitment=com, pok=pok,
                    ped_g=vk.PedersenG if vk.has_commitment else None,
                    ped_g_sigma_neg=vk.PedersenGSigmaNeg if vk.has_commitment else None)
    if not ok:
        raise ValueError("groth16.Verify: pairing check failed")


def BatchVerify(ctx, proofs, vk, public_witnesses, coeffs=None):
    """Verify k proofs of one circuit in one call (b200g16_verify_batch) -> list of k bools, each equal to what
    Verify decides for that proof alone.  public_witnesses[i] is proof i's public witness, as Verify takes it.

    coeffs: k nonzero integers < 2^128 (then k more with a commitment) for the small-exponent batch test.  They must be
    unpredictable to whoever made the proofs; by default they are drawn with secrets.randbits(128).  Passing them
    makes a run reproducible, like r and s in Prove.  Malformed input raises as in Verify."""
    k = len(proofs)
    if len(public_witnesses) != k:
        raise ValueError("groth16.BatchVerify: %d proofs but %d public witnesses" % (k, len(public_witnesses)))
    n_coef = 2 * k if vk.has_commitment else k
    if coeffs is None:
        coeffs = []
        while len(coeffs) < n_coef:
            c = secrets.randbits(128)
            if c:
                coeffs.append(c)
    if len(coeffs) != n_coef:
        raise ValueError("groth16.BatchVerify: %d coefficients, expected %d" % (len(coeffs), n_coef))
    if any(not 0 < int(c) < 1 << 128 for c in coeffs):
        raise ValueError("groth16.BatchVerify: coefficients must be nonzero and below 2^128")
    co = np.array([(int(c) & _M64, int(c) >> 64) for c in coeffs], dtype=np.uint64).reshape(-1, 2)
    n_pub = len(vk.G1_K) - 1
    pubs = np.zeros((k, n_pub, 4), dtype=np.uint64)
    coms, poks = [], []
    for i, (proof, pw) in enumerate(zip(proofs, public_witnesses)):
        pub, com, pok = _verify_inputs(proof, vk, pw)
        if len(pub) != n_pub:
            raise lib.B200Error("groth16.BatchVerify: proof %d has %d public inputs, vk.G1.K expects %d"
                                % (i, len(pub), n_pub))
        if pub:
            pubs[i] = fr_array(pub)
        coms.append(com)
        poks.append(pok)
    stack = lambda pts, w: np.array([np.asarray(p, dtype=np.uint64).reshape(w) for p in pts],
                                    dtype=np.uint64).reshape(k, w)
    _, each = ctx.verify_batch(vk.G1_Alpha, vk.G2_Beta, vk.G2_Gamma, vk.G2_Delta, vk.G1_K,
                               stack([p.Ar for p in proofs], 8), stack([p.Bs for p in proofs], 16),
                               stack([p.Krs for p in proofs], 8), pubs, co,
                               commitments=stack(coms, 8) if vk.has_commitment else None,
                               poks=stack(poks, 8) if vk.has_commitment else None,
                               ped_g=vk.PedersenG if vk.has_commitment else None,
                               ped_g_sigma_neg=vk.PedersenGSigmaNeg if vk.has_commitment else None)
    return [bool(x) for x in each]
