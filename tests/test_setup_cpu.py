"""Groth16 setup pieces that need no GPU: the C restatement of gnark's setupABC (oracle_setup_abc) against the python
oracle, SparseR1CS.from_r1cs, the synthetic CSR generator, and the layout of the setup's public structs."""
import os
import random
import subprocess

import numpy as np
import pytest

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import bn254 as bn
from oracle import groth16 as og
from oracle import setup_port as sp
from oracle.bn254 import R
from oracle.ntt import Domain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _edge_r1cs(m, seed):
    """m constraints with empty rows, repeated wires in a row, zero coefficients and wires no term names."""
    rng = random.Random(seed)
    nw, npub = m + 12, 2

    def lc(k):
        return [(rng.randrange(nw - 3), rng.choice([0, 1, 1, 2, rng.randrange(R)])) for _ in range(k)]
    cons = []
    for j in range(m):
        L = lc(rng.randrange(0, 4))
        if L and rng.random() < 0.3:
            L.append((L[0][0], rng.randrange(R)))           # the same wire twice in one row
        cons.append((L, lc(rng.randrange(0, 3)), lc(rng.randrange(0, 2))))
    return og.R1CS(nw, npub, cons)


def _oracle_abc(r1cs, tau):
    return [bn.fr_to_mont_array(v) for v in og.wire_polys_at_tau(r1cs, Domain(r1cs.nb_constraints), tau)]


@pytest.mark.parametrize("m", [1, 2, 3, 4, 5, 8, 9, 16, 17, 64, 65])
def test_setup_abc_matches_python_oracle(m):
    r1cs = _edge_r1cs(m, 1000 + m)
    tau = random.Random(m).randrange(1, R)
    got = sp.setup_abc(g16.SparseR1CS.from_r1cs(r1cs), bn.fr_to_mont_array([tau])[0])
    for g, e in zip(got, _oracle_abc(r1cs, tau)):
        assert np.array_equal(g, e)


def test_setup_abc_synthetic_circuit_matches_python_oracle():
    rng = random.Random(5)
    r1cs, _ = og.synthetic_r1cs(100, 4, rng, with_commitment=True)
    tau = rng.randrange(1, R)
    got = sp.setup_abc(g16.SparseR1CS.from_r1cs(r1cs), bn.fr_to_mont_array([tau])[0])
    for g, e in zip(got, _oracle_abc(r1cs, tau)):
        assert np.array_equal(g, e)


def test_setup_abc_refuses_tau_in_domain():
    r1cs = _edge_r1cs(8, 3)
    w = Domain(8).gen
    with pytest.raises(ValueError):
        sp.setup_abc(g16.SparseR1CS.from_r1cs(r1cs), bn.fr_to_mont_array([pow(w, 3, R)])[0])


def test_from_r1cs_keeps_every_term():
    r1cs = _edge_r1cs(40, 11)
    r1cs.commitment_wire, r1cs.private_committed, r1cs.public_committed = 45, [3, 7, 9], [1]
    s = g16.SparseR1CS.from_r1cs(r1cs)
    assert s.constraints == [tuple([(i, c % R) for i, c in t] for t in con) for con in r1cs.constraints]
    assert len(s.l_row) == len(s.r_row) == len(s.o_row) == 41
    assert s.l_row.dtype == np.uint64 and s.l_wire.dtype == np.uint32 and s.l_coeff.dtype == np.uint32
    assert len({tuple(c) for c in s.coeffs.tolist()}) == len(s.coeffs)        # interned: each value once
    assert s.commitment_wire == 45 and s.private_committed.tolist() == [3, 7, 9] and s.public_committed == [1]


@pytest.mark.parametrize("stress", [False, True])
def test_synthetic_csr_shape(stress):
    d = sp.synthetic_csr(1 << 10, 7, stress=stress, hot_wire_rows=stress, unused_wires=5)
    m = 1 << 10
    for p in "lro":
        row = d[p + "_row"]
        assert len(row) == m + 1 and row[0] == 0 and np.all(np.diff(row.astype(np.int64)) >= 0)
        assert len(d[p + "_wire"]) == len(d[p + "_coeff"]) == row[-1]
        assert d[p + "_wire"].max() < d["nb_wires"] - 5 and d[p + "_coeff"].max() < len(d["coeffs"])
    rlen = np.diff(d["r_row"].astype(np.int64))
    r0 = (rlen == 1) & (d["r_wire"][d["r_row"][:-1].astype(np.int64)] == 0)
    assert 0.25 < r0.mean() < 0.45
    if stress:
        assert np.diff(d["l_row"].astype(np.int64)).max() == 1 << 16
        assert (np.diff(d["o_row"].astype(np.int64)) == 0).any()


def test_csr_witness_satisfies():
    d = sp.synthetic_csr(300, 9)
    w = sp.csr_witness(d, 4)
    a, b, c = og.solve_abc(g16.SparseR1CS(**d), w)
    assert all(x * y % R == z for x, y, z in zip(a, b, c))


@pytest.mark.parametrize("fault", ["short_r_row", "long_o_row", "no_rows", "few_terms"])
def test_r1cs_desc_refuses_arrays_the_library_would_overrun(fault):
    s = g16.SparseR1CS.from_r1cs(_edge_r1cs(16, 2))
    if fault == "short_r_row":
        s.r_row = s.r_row[:-1].copy()
    elif fault == "long_o_row":
        s.o_row = np.append(s.o_row, s.o_row[-1])
    elif fault == "no_rows":
        s.l_row = s.r_row = s.o_row = np.zeros(0, dtype=np.uint64)
    else:
        s.l_wire = s.l_wire[:-1].copy()
    with pytest.raises(lib.B200Error):
        lib._r1cs_desc(s)
    lib._r1cs_desc(g16.SparseR1CS.from_r1cs(_edge_r1cs(16, 2)))     # the well-formed system passes


def test_setup_structs_layout(tmp_path):
    asserts = []
    for cname, cls in (("b200g16_r1cs_desc", lib.R1csDesc), ("b200g16_toxic", lib.Toxic),
                       ("b200g16_setup_out", lib.SetupOut)):
        import ctypes
        asserts.append(f'_Static_assert(sizeof({cname}) == {ctypes.sizeof(cls)}, "{cname}");')
        for name, _ in cls._fields_:
            asserts.append(f'_Static_assert(offsetof({cname}, {name}) == {getattr(cls, name).offset}, "{cname}.{name}");')
    src = tmp_path / "setup_layout.c"
    src.write_text("#include <stddef.h>\n#include \"b200g16.h\"\n" + "\n".join(asserts) + "\nint main(void) { return 0; }\n")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), "-c",
                    str(src), "-o", str(tmp_path / "setup_layout.o")], check=True)
