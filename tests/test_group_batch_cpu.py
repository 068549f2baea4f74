"""CPU side of the group batch prove (b200g16_bases_copy, b200g16_group_pk_replicate, b200g16_group_prove_batch):
the declarations are valid C and bound in lib.SIGNATURES with their arity, NULL arguments are refused without a
device, and Group.prove_batch refuses row shapes that would let the library read past a numpy buffer before any
library call (as the batch prove and the setup descriptor builder do)."""
import os
import subprocess

import numpy as np
import pytest

from gnark_whir_b200 import lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_new_declarations_are_bound():
    src = open(os.path.join(ROOT, "include", "b200g16.h")).read()
    for name, arity in (("b200g16_bases_copy", 3), ("b200g16_group_pk_replicate", 3), ("b200g16_group_prove_batch", 12)):
        assert name + "(" in src
        assert len(lib.SIGNATURES[name][1]) == arity, name
        assert hasattr(lib.load(), name)


def test_header_compiles_as_c11_and_refuses_null(tmp_path):
    libdir = os.path.join(ROOT, "gnark_whir_b200")
    exe = str(tmp_path / "abi_check_group_batch")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "host_harness", "abi_check_group_batch.c"), "-L", libdir, "-lb200g16",
                    "-Wl,-rpath," + libdir, "-o", exe], check=True)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert out.stdout.startswith("ok:")


class _NoLibrary:
    """Stands in for the library: any call fails the test (the shape checks must come first)."""

    def __getattr__(self, name):
        raise AssertionError(f"{name} reached the library")


def _rows(k=3, nw=10, nc=7):
    z = lambda *s: np.zeros(s, dtype=np.uint64)
    return z(k, nw, 4), z(k, nc, 4), z(k, nc, 4), z(k, nc, 4), z(k, 4), z(k, 4)


@pytest.mark.parametrize("case", ["a_rows", "c_len", "wires_2d", "r_count", "s_count", "b_limbs"])
def test_group_prove_batch_refuses_mismatched_rows(monkeypatch, case):
    wires, a, b, c, r, s = _rows()
    if case == "a_rows":
        a = a[:2]
    elif case == "c_len":
        c = c[:, :6]
    elif case == "wires_2d":
        wires = wires.reshape(-1, 4)
    elif case == "r_count":
        r = r[:2]
    elif case == "s_count":
        s = np.zeros((4, 4), dtype=np.uint64)
    elif case == "b_limbs":
        b = np.zeros((3, 7, 3), dtype=np.uint64)
    g = lib.Group.__new__(lib.Group)
    g.h, g.devices = lib._vp(1), [0]
    monkeypatch.setattr(lib, "load", lambda: _NoLibrary())
    with pytest.raises(lib.B200Error, match="group prove_batch"):
        g.prove_batch(lib._vp(1), wires, a, b, c, r, s)
