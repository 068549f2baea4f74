"""The Keccak duplex's op walk on the CPU: gnark_whir_b200/csrc/keccak_duplex.cuh, compiled for the host by
tests/host_harness/duplex_host.cc, applied to a byte-array state and compared with oracle/keccak.py's Sponge (the
restatement of keccakSponge.Digest) on random and hand-picked scripts, split into calls at every op boundary; the
layout of the public structs; the Python helpers that build digests and scripts.

The script / oracle helpers at the top are shared with tests/test_gpu_keccak_duplex.py."""
import ctypes as C
import os
import random
import re
import subprocess

import numpy as np
import pytest

from gnark_whir_b200 import lib
from oracle import keccak as ok

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "host_harness", "duplex_host.cc")
OUT = os.path.join(HERE, "host_harness", "_build", "duplex_host.so")
CSRC = os.path.join(ROOT, "gnark_whir_b200", "csrc")

LENGTHS = [0, 1, 7, 8, 9, 135, 136, 137, 271, 272, 273, 1000]


def random_script(rs, n_ops=None, lengths=LENGTHS):
    n_ops = rs.randint(1, 12) if n_ops is None else n_ops
    return [(rs.choice(("absorb", "squeeze")), rs.choice(lengths)) for _ in range(n_ops)]


def script_bytes(script):
    return (sum(n for k, n in script if k == "absorb"), sum(n for k, n in script if k == "squeeze"))


def sponge_from(digest=None, tag=b""):
    """An oracle Sponge: NewKeccakWithTag(tag), or the state a KECCAK_DIGEST record holds."""
    s = ok.Sponge(tag)
    if digest is not None:
        s.state = bytearray(np.asarray(digest["state"], dtype="<u8").tobytes())
        s.absorb_pos, s.squeeze_pos = int(digest["absorb_pos"]), int(digest["squeeze_pos"])
    return s


def oracle_run(sponge, script, data):
    """Run the script on an oracle Sponge, absorbing from `data` in order; -> the squeezed bytes."""
    out, off = bytearray(), 0
    for kind, n in script:
        if kind == "absorb":
            sponge.absorb(bytes(data[off:off + n]))
            off += n
        else:
            out += sponge.squeeze(n)
    return bytes(out)


def sponge_digest(sponge):
    """An oracle Sponge's state as a KECCAK_DIGEST record."""
    d = np.zeros((), dtype=lib.KECCAK_DIGEST)
    d["state"] = np.frombuffer(bytes(sponge.state), dtype="<u8")
    d["absorb_pos"], d["squeeze_pos"] = sponge.absorb_pos, sponge.squeeze_pos
    return d


@pytest.fixture(scope="module")
def host():
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-I", CSRC, "-o", OUT], check=True)
    L = C.CDLL(OUT)
    L.host_duplex.restype = C.c_long
    L.host_duplex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                              C.POINTER(C.c_uint64)]
    return L


class Walk:
    """A state run through the header's segment walk (host build)."""

    def __init__(self, L, tag=b"", sponge=None):
        self.L = L
        src = sponge if sponge is not None else ok.Sponge(tag)
        self.state = np.frombuffer(bytes(src.state), dtype=np.uint8).copy()
        self.pos = np.array([src.absorb_pos, src.squeeze_pos], dtype=np.uint32)
        self.n_perm = C.c_uint64(0)

    def run(self, script, data):
        ops, A, S = lib.duplex_script(script)
        inp = np.frombuffer(bytes(data) + b"\0", dtype=np.uint8)
        out = np.zeros(S + 1, dtype=np.uint8)
        segs = self.L.host_duplex(self.state.ctypes.data, self.pos.ctypes.data, ops.ctypes.data, len(script),
                                  inp.ctypes.data, out.ctypes.data, C.byref(self.n_perm))
        assert segs >= 0, "a segment left its rate block"
        return bytes(out[:S])

    def same_as(self, sponge):
        return (bytes(self.state) == bytes(sponge.state) and int(self.pos[0]) == sponge.absorb_pos
                and int(self.pos[1]) == sponge.squeeze_pos)


def check_script(L, script, tag=b"", data=None, rs=None):
    A, _ = script_bytes(script)
    if data is None:
        data = bytes(rs.getrandbits(8) for _ in range(A))
    ref = ok.Sponge(tag)
    want = oracle_run(ref, script, data)
    w = Walk(L, tag)
    assert w.run(script, data) == want, script
    assert w.same_as(ref), script
    assert w.n_perm.value == ref.n_permutes, script
    return data, want, ref


@pytest.mark.parametrize("tag_len", [0, 1, 63, 64])
def test_random_scripts_match_oracle(host, tag_len):
    rs = random.Random(1000 + tag_len)
    for _ in range(10):
        tag = bytes(rs.getrandbits(8) for _ in range(tag_len))
        check_script(host, random_script(rs), tag, rs=rs)


@pytest.mark.parametrize("name,script", [
    ("squeeze-squeeze inside one block", [("absorb", 9), ("squeeze", 7), ("squeeze", 8), ("squeeze", 121)]),
    ("squeeze-squeeze crossing a block", [("absorb", 9), ("squeeze", 100), ("squeeze", 100)]),
    ("absorb after a permuting squeeze", [("absorb", 40), ("squeeze", 32), ("absorb", 50), ("squeeze", 32)]),
    ("absorb after a squeeze that did not permute",
     [("absorb", 40), ("squeeze", 32), ("squeeze", 8), ("absorb", 17), ("squeeze", 9)]),
    ("absorb(0) forces the next permutation", [("absorb", 10), ("squeeze", 5), ("absorb", 0), ("squeeze", 5)]),
    ("absorb(0) on a fresh sponge", [("absorb", 0), ("squeeze", 32)]),
    ("squeeze on a fresh sponge", [("squeeze", 300)]),
    ("full block absorbed, not yet permuted", [("absorb", 136)]),
    ("full block then one more byte", [("absorb", 136), ("absorb", 1), ("squeeze", 1)]),
    ("two full blocks then squeeze", [("absorb", 272), ("squeeze", 136), ("squeeze", 1)]),
    ("squeeze(0) changes nothing", [("absorb", 3), ("squeeze", 0), ("absorb", 4), ("squeeze", 0)]),
    ("only empty ops", [("absorb", 0), ("squeeze", 0)]),
])
def test_edge_scripts_match_oracle(host, name, script):
    rs = random.Random(name)
    for tag_len in (0, 64):
        check_script(host, script, bytes(range(1, tag_len + 1)), rs=rs)


def test_full_block_carried_across_calls(host):
    """absorb_pos == 136 with the block unpermuted is a state that survives the end of a call."""
    rs = random.Random(7)
    data = bytes(rs.getrandbits(8) for _ in range(136 + 20))
    ref = ok.Sponge()
    want = oracle_run(ref, [("absorb", 136), ("absorb", 20), ("squeeze", 64)], data)
    w = Walk(host)
    w.run([("absorb", 136)], data[:136])
    assert int(w.pos[0]) == 136 and int(w.pos[1]) == 136 and w.n_perm.value == 0
    assert w.run([("absorb", 20), ("squeeze", 64)], data[136:]) == want
    assert w.same_as(ref) and w.n_perm.value == ref.n_permutes


def test_split_at_every_op_boundary(host):
    """Cutting a script into two or three calls with the state carried between them gives the one call's result."""
    rs = random.Random(99)
    for trial in range(12):
        script = random_script(rs, n_ops=rs.randint(3, 8))
        tag = bytes(rs.getrandbits(8) for _ in range(rs.choice((0, 1, 63, 64))))
        data, want, ref = check_script(host, script, tag, rs=rs)
        cuts = [(i,) for i in range(1, len(script))] + [(i, j) for i in range(1, len(script))
                                                         for j in range(i + 1, len(script))]
        for cut in cuts:
            w = Walk(host, tag)
            got, a_off = b"", 0
            for lo, hi in zip((0,) + cut, cut + (len(script),)):
                part = script[lo:hi]
                A, _ = script_bytes(part)
                got += w.run(part, data[a_off:a_off + A])
                a_off += A
            assert got == want, (script, cut)
            assert w.same_as(ref) and w.n_perm.value == ref.n_permutes, (script, cut)


def test_continue_from_any_positions(host):
    """Digests the caller wrote by hand: every pair of positions in 0..136 at the edges."""
    rs = random.Random(5)
    edge = [0, 1, 7, 8, 135, 136]
    script = [("squeeze", 9), ("absorb", 140), ("squeeze", 3), ("absorb", 0), ("squeeze", 1)]
    A, _ = script_bytes(script)
    for ap in edge:
        for sp in edge:
            start = ok.Sponge()
            start.state = bytearray(rs.getrandbits(8) for _ in range(200))
            start.absorb_pos, start.squeeze_pos = ap, sp
            data = bytes(rs.getrandbits(8) for _ in range(A))
            w = Walk(host, sponge=start)
            ref = ok.Sponge()
            ref.state, ref.absorb_pos, ref.squeeze_pos = bytearray(start.state), ap, sp
            assert w.run(script, data) == oracle_run(ref, script, data), (ap, sp)
            assert w.same_as(ref) and w.n_perm.value == ref.n_permutes


def test_public_struct_layout(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text("""#include <stddef.h>
#include "b200g16.h"
_Static_assert(sizeof(b200g16_keccak_digest) == 208, "digest size");
_Static_assert(offsetof(b200g16_keccak_digest, absorb_pos) == 200, "absorb_pos");
_Static_assert(offsetof(b200g16_keccak_digest, squeeze_pos) == 204, "squeeze_pos");
_Static_assert(sizeof(b200g16_duplex_op) == 8, "op size");
_Static_assert(offsetof(b200g16_duplex_op, len) == 4, "op len");
int main(void) { return 0; }
""")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), "-c",
                    str(src), "-o", str(tmp_path / "layout.o")], check=True)
    assert lib.KECCAK_DIGEST.itemsize == 208
    assert lib.KECCAK_DIGEST.fields["absorb_pos"][1] == 200 and lib.KECCAK_DIGEST.fields["squeeze_pos"][1] == 204


def test_digest_helper_matches_oracle():
    tags = [b"", b"\x01", bytes(range(63)), bytes(range(100, 164))]
    d = lib.keccak_digests(len(tags), tags)
    for rec, t in zip(d, tags):
        s = ok.Sponge(t)
        assert rec.tobytes() == bytes(s.state) + (0).to_bytes(4, "little") + (136).to_bytes(4, "little")
    assert (lib.keccak_digests(3, b"ab")["state"] == lib.keccak_digests(3, [b"ab"] * 3)["state"]).all()
    with pytest.raises(lib.B200Error):
        lib.keccak_digests(1, [bytes(65)])


def test_script_helper():
    ops, A, S = lib.duplex_script([("absorb", 5), ("squeeze", 7), ("absorb", 0), ("squeeze", 1)])
    assert ops.dtype == np.uint32 and ops.tolist() == [[0, 5], [1, 7], [0, 0], [1, 1]] and (A, S) == (5, 8)
    for bad in ([("mix", 1)], [("absorb", -1)], [("squeeze", 1 << 32)]):
        with pytest.raises(lib.B200Error):
            lib.duplex_script(bad)


def test_warp_threshold_matches_library():
    src = open(os.path.join(CSRC, "keccak.cu")).read()
    m = re.search(r"constexpr size_t DUPLEX_WARP_MAX = (\d+);", src)
    assert m and int(m.group(1)) == lib.KECCAK_DUPLEX_WARP_MAX
