"""Groth16 setup at scale, TEST INFRASTRUCTURE (used by tests/ and tools/setup_bench.py; never by the product):

  setup_abc        ctypes binding of oracle/c/oracle_setup.c, the C restatement of gnark's setupABC (built by
                   `make -C oracle -f setup.mk`, done by __graft_entry__.build())
  synthetic_csr    numpy CSR constraint systems of 2^16 - 2^24 constraints shaped like oracle.groth16.synthetic_r1cs,
                   plus the stress shapes the GPU setup must survive
  csr_witness      a satisfying witness of a generated system (python ints)

A system is a dict with the fields of gnark_whir_b200.groth16.SparseR1CS (and of struct b200g16_r1cs_desc):
nb_wires, nb_public, coeffs ((n, 4) Montgomery), l_row / l_wire / l_coeff, r_*, o_* (row: uint64 CSR offsets by
constraint, wire / coeff: uint32 term arrays), private_committed, public_committed, commitment_wire."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import bn254 as bn
from .bn254 import R

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "liboracle_setup.so")
_lib = None
_vp = C.c_void_p


def build():
    subprocess.run(["make", "-s", "-C", _HERE, "-f", "setup.mk"], check=True)


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        lib = C.CDLL(LIB_PATH)
        lib.oracle_setup_abc.restype = C.c_int
        lib.oracle_setup_abc.argtypes = [C.c_size_t, C.c_size_t, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        _lib = lib
    return _lib


def setup_abc(sys_, tau_mont):
    """gnark's setupABC in C: (A, B, C) per wire, each (n_wires, 4) Montgomery.  tau_mont: 4 limbs."""
    m = len(sys_["l_row"]) - 1
    nw = int(sys_["nb_wires"])
    keep = [np.ascontiguousarray(sys_["coeffs"], dtype=np.uint64).reshape(-1, 4)]
    ptr = lambda a: a.ctypes.data_as(_vp)
    rows, wires, cids = (C.c_void_p * 3)(), (C.c_void_p * 3)(), (C.c_void_p * 3)()
    for k, p in enumerate("lro"):
        r = np.ascontiguousarray(sys_[p + "_row"], dtype=np.uint64)
        w = np.ascontiguousarray(sys_[p + "_wire"], dtype=np.uint32)
        c = np.ascontiguousarray(sys_[p + "_coeff"], dtype=np.uint32)
        keep += [r, w, c]
        rows[k], wires[k], cids[k] = ptr(r).value, ptr(w).value, ptr(c).value
    tau = np.ascontiguousarray(tau_mont, dtype=np.uint64).reshape(4)
    out = [np.zeros((nw, 4), dtype=np.uint64) for _ in range(3)]
    st = load().oracle_setup_abc(m, nw, ptr(keep[0]), rows, wires, cids, ptr(tau), *[ptr(o) for o in out])
    if st:
        raise ValueError("oracle_setup_abc: tau^N = 1 or out of memory")
    return tuple(out)


def _csr(counts):
    row = np.zeros(len(counts) + 1, dtype=np.uint64)
    np.cumsum(counts, out=row[1:])
    return row


def synthetic_csr(m, seed, nb_public=3, n_inputs=64, stress=False, hot_wire_rows=False, unused_wires=0):
    """m constraints (L) * (R) = (O) over nb_public public wires, n_inputs private input wires and one output wire per
    constraint.  L has 1-3 terms, R 1-2, O one; constraint j's L and R read public, input and earlier output wires
    only (so csr_witness solves it in order).  Coefficients: 70% are 1, 30% drawn from 252 random field elements;
    wire 0 (the constant one) is the whole of R in 30% of the rows.  unused_wires: extra wires no term names.
    stress: row 0 of L holds 2^16 terms, every 7th O row is empty, 10% of the L rows name a wire twice and 1% of all
    terms have coefficient 0 (not satisfiable any more).  hot_wire_rows: wire 1 is added to every L row."""
    rs = np.random.Generator(np.random.PCG64(seed))
    base = nb_public + n_inputs
    nw = base + m + unused_wires
    table = [1, 0, 2, R - 1] + [int(x) for x in rs.integers(1, 1 << 62, size=252)]
    table = [v * (1 << 190) % R if i >= 4 else v for i, v in enumerate(table)]
    coeffs = bn.fr_to_mont_array(table)

    def cids(n):
        c = np.where(rs.random(n) < 0.7, 0, rs.integers(4, len(table), size=n)).astype(np.uint32)
        if stress:
            c[rs.random(n) < 0.01] = 1
        return c

    nl = rs.integers(1, 4, size=m)
    if hot_wire_rows:
        nl = nl + 1
    if stress:
        nl[0] = 1 << 16
    nr = rs.integers(1, 3, size=m)
    only_one = rs.random(m) < 0.3
    nr[only_one] = 1
    no = np.ones(m, dtype=np.int64)
    if stress:
        no[::7] = 0
    l_row, r_row, o_row = _csr(nl), _csr(nr), _csr(no)

    def earlier(row, counts):   # per term: a random wire the row may read (public, input, or an earlier output)
        limit = base + np.repeat(np.arange(m, dtype=np.int64), counts)
        return (rs.random(int(row[-1])) * limit).astype(np.uint32)
    l_wire = earlier(l_row, nl)
    if hot_wire_rows:
        l_wire[l_row[:-1].astype(np.int64)] = 1
    if stress:
        two = np.nonzero((nl >= 2) & (rs.random(m) < 0.1))[0]
        s = l_row[two].astype(np.int64)
        l_wire[s + 1] = l_wire[s]
    r_wire = earlier(r_row, nr)
    r_wire[r_row[:-1][only_one].astype(np.int64)] = 0
    o_wire = (base + np.nonzero(no)[0]).astype(np.uint32)
    o_coeff = np.zeros(len(o_wire), dtype=np.uint32)
    if stress:
        o_coeff = cids(len(o_wire))
    return dict(nb_wires=nw, nb_public=nb_public, coeffs=coeffs, l_row=l_row, l_wire=l_wire, l_coeff=cids(len(l_wire)),
                r_row=r_row, r_wire=r_wire, r_coeff=cids(len(r_wire)), o_row=o_row, o_wire=o_wire, o_coeff=o_coeff,
                private_committed=np.zeros(0, dtype=np.uint32), public_committed=[], commitment_wire=-1)


def csr_witness(sys_, seed):
    """A satisfying full assignment of a synthetic_csr system without stress shapes (python ints)."""
    rs = np.random.Generator(np.random.PCG64(seed))
    nw, npub = sys_["nb_wires"], sys_["nb_public"]
    base = int(sys_["o_wire"][0]) if len(sys_["o_wire"]) else nw
    w = [0] * nw
    w[0] = 1
    for i in range(1, base):
        u = rs.random()
        w[i] = int(rs.integers(0, 2)) if u < 0.4 else int(rs.integers(0, 256)) if u < 0.7 or i < npub else \
            int(rs.integers(1, 1 << 62)) * (1 << 190) % R
    cf = bn.fr_from_mont_array(np.asarray(sys_["coeffs"], dtype=np.uint64).reshape(-1, 4))

    def lc(p, j):
        a, b = int(sys_[p + "_row"][j]), int(sys_[p + "_row"][j + 1])
        return sum(cf[c] * w[i] for i, c in zip(sys_[p + "_wire"][a:b].tolist(), sys_[p + "_coeff"][a:b].tolist())) % R
    for j in range(len(sys_["l_row"]) - 1):
        w[base + j] = lc("l", j) * lc("r", j) % R
    return w
