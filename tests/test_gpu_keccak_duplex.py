"""GPU parity of b200g16_keccak_duplex_batch(_dev): the whole keccakSponge.Digest (tags, Absorb / Squeeze in any
order, state carried across calls) for a batch of sponges, byte-exact against oracle/keccak.py's Sponge for every
sponge checked, in both kernel forms (one thread per sponge, one warp per sponge) and on both the host and the
device-pointer path; argument errors leave the digests untouched and the ctx usable."""
import ctypes as C
import random

import numpy as np
import pytest

from gnark_whir_b200 import groth16 as g16
from gnark_whir_b200 import lib
from oracle import cport
from oracle import keccak as ok
from tests.test_keccak_duplex_cpu import oracle_run, random_script, script_bytes, sponge_digest, sponge_from

pytestmark = pytest.mark.gpu

W = lib.KECCAK_DUPLEX_WARP_MAX
FORMS = [None, "0", "1"]   # B200G16_DUPLEX_WARP: by n, thread form forced, warp form forced
ERR_ARG = -2   # B200G16_ERR_ARG
TRANSCRIPT = [("absorb", 32), ("squeeze", 32), ("absorb", 512), ("squeeze", 64), ("absorb", 8), ("squeeze", 32)]


def rand_bytes(rs, shape):
    return rs.integers(0, 256, size=shape, dtype=np.uint8)


def sample_rows(n, rs, k=48):
    edge = {0, 1, 31, 32, 33, n // 2, n - 2, n - 1, W - 1, W, W + 1}
    rows = {i for i in edge if 0 <= i < n}
    if n <= 257:
        return sorted(range(n))
    return sorted(rows | set(rs.choice(n, size=min(k, n), replace=False).tolist()))


def check_rows(script, data, out, digests, rows, start):
    """start(i) -> the oracle Sponge sponge i starts from."""
    for i in rows:
        s = start(i)
        assert bytes(out[i]) == oracle_run(s, script, data[i]), (i, script)
        assert digests[i].tobytes() == sponge_digest(s).tobytes(), i


def set_form(monkeypatch, form):
    if form is None:
        monkeypatch.delenv("B200G16_DUPLEX_WARP", raising=False)
    else:
        monkeypatch.setenv("B200G16_DUPLEX_WARP", form)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 257, W, W + 1, 1 << 16])
def test_random_scripts_both_forms(ctx, monkeypatch, n):
    rr = random.Random(n)
    big = n > 4096
    script = random_script(rr, n_ops=rr.randint(3, 6) if big else None,
                           lengths=[0, 1, 7, 8, 9, 135, 136, 137, 271, 272, 273] if big else
                           [0, 1, 7, 8, 9, 135, 136, 137, 271, 272, 273, 1000])
    A, S = script_bytes(script)
    rs = np.random.Generator(np.random.PCG64(n))
    data = rand_bytes(rs, (n, A))
    tag = bytes(rand_bytes(rs, rr.choice((0, 1, 63, 64))))
    results = []
    for form in FORMS:
        set_form(monkeypatch, form)
        results.append(ctx.keccak_duplex_batch(script, data, tag=tag))
    out, dg = results[0]
    for o, d in results[1:]:
        assert np.array_equal(o, out) and d.tobytes() == dg.tobytes()
    check_rows(script, data, out, dg, sample_rows(n, rs), lambda i: ok.Sponge(tag))


@pytest.mark.parametrize("form", FORMS)
def test_per_sponge_tags_and_three_calls(ctx, monkeypatch, form):
    """Per-sponge tags written into the digests, then the script cut into three calls with the digests carried on
    the host; the same on device memory (torch), with input and output rows that are not multiples of 8 and start at
    odd addresses."""
    torch = pytest.importorskip("torch")
    set_form(monkeypatch, form)
    n = 300
    rr = random.Random(3)
    rs = np.random.Generator(np.random.PCG64(3))
    parts = [[("absorb", 13), ("squeeze", 9)], [("absorb", 136), ("absorb", 0)],
             [("squeeze", 141), ("absorb", 273), ("squeeze", 7)]]
    tags = [bytes(rand_bytes(rs, rr.choice((0, 1, 63, 64)))) for _ in range(n)]
    full = sum(parts, [])
    A, S = script_bytes(full)
    data = rand_bytes(rs, (n, A))
    # host digests
    dg, outs, a0 = lib.keccak_digests(n, tags), [], 0
    for p in parts:
        pa, _ = script_bytes(p)
        o, dg = ctx.keccak_duplex_batch(p, data[:, a0:a0 + pa], digests=dg)
        outs.append(o)
        a0 += pa
    out = np.concatenate(outs, axis=1)
    check_rows(full, data, out, dg, range(n), lambda i: ok.Sponge(tags[i]))
    one, dg1 = ctx.keccak_duplex_batch(full, data, digests=lib.keccak_digests(n, tags))
    assert np.array_equal(one, out) and dg1.tobytes() == dg.tobytes()
    # device digests, unaligned rows
    d_dg = torch.from_numpy(lib.keccak_digests(n, tags).view(np.uint8).copy()).cuda()
    d_out_all = []
    for p in parts:
        pa, ps = script_bytes(p)
        a0 = sum(script_bytes(q)[0] for q in parts[:parts.index(p)])
        buf_in = torch.zeros(n * pa + 1, dtype=torch.uint8, device="cuda")
        buf_in[1:] = torch.from_numpy(np.ascontiguousarray(data[:, a0:a0 + pa]).reshape(-1)).cuda()
        buf_out = torch.zeros(n * ps + 3, dtype=torch.uint8, device="cuda")
        ctx.keccak_duplex_batch_dev(d_dg.data_ptr(), n, p, buf_in.data_ptr() + 1, buf_out.data_ptr() + 3)
        torch.cuda.synchronize()
        assert int(buf_out[:3].sum()) == 0
        d_out_all.append(buf_out[3:].cpu().numpy().reshape(n, ps))
    assert np.array_equal(np.concatenate(d_out_all, axis=1), out)
    assert d_dg.cpu().numpy().tobytes() == dg.tobytes()


@pytest.mark.parametrize("form", FORMS)
def test_dev_shared_tag(ctx, monkeypatch, form):
    torch = pytest.importorskip("torch")
    set_form(monkeypatch, form)
    n = 1000
    rs = np.random.Generator(np.random.PCG64(11))
    tag = bytes(rand_bytes(rs, 64))
    script = [("absorb", 5), ("squeeze", 3), ("squeeze", 140), ("absorb", 271)]
    A, S = script_bytes(script)
    data = rand_bytes(rs, (n, A))
    d_in = torch.from_numpy(data.reshape(-1).copy()).cuda()
    d_out = torch.zeros(n * S, dtype=torch.uint8, device="cuda")
    d_dg = torch.full((n * 208,), 0xAB, dtype=torch.uint8, device="cuda")   # not read under a tag
    ctx.keccak_duplex_batch_dev(d_dg.data_ptr(), n, script, d_in.data_ptr(), d_out.data_ptr(), tag=tag)
    torch.cuda.synchronize()
    out = d_out.cpu().numpy().reshape(n, S)
    dg = d_dg.cpu().numpy().view(lib.KECCAK_DIGEST)
    check_rows(script, data, out, dg, sample_rows(n, rs), lambda i: ok.Sponge(tag))
    h_out, h_dg = ctx.keccak_duplex_batch(script, data, tag=tag)
    assert np.array_equal(h_out, out) and h_dg.tobytes() == dg.tobytes()


def test_continue_from_hand_written_states(ctx, monkeypatch):
    """Digests holding arbitrary states and positions (absorb_pos 136 with the block unpermuted included)."""
    n = 64
    rr = random.Random(17)
    starts = []
    for i in range(n):
        s = ok.Sponge()
        s.state = bytearray(rr.getrandbits(8) for _ in range(200))
        s.absorb_pos, s.squeeze_pos = rr.choice((0, 1, 8, 135, 136)), rr.choice((0, 7, 135, 136))
        starts.append(s)
    dg = np.array([sponge_digest(s) for s in starts], dtype=lib.KECCAK_DIGEST)
    script = [("squeeze", 9), ("absorb", 140), ("squeeze", 3), ("absorb", 0), ("squeeze", 1)]
    A, _ = script_bytes(script)
    data = rand_bytes(np.random.Generator(np.random.PCG64(17)), (n, A))
    for form in FORMS[1:]:
        set_form(monkeypatch, form)
        out, got = ctx.keccak_duplex_batch(script, data, digests=dg)
        check_rows(script, data, out, got, range(n), lambda i: sponge_from(sponge_digest(starts[i])))


@pytest.mark.parametrize("in_len,out_len", [(0, 32), (7, 1), (136, 32), (137, 200), (512, 32)])
def test_matches_one_shot_sponge(ctx, in_len, out_len):
    n = 777
    data = rand_bytes(np.random.Generator(np.random.PCG64(in_len)), (n, in_len))
    want = ctx.keccak_sponge_batch(data, out_len)
    got, _ = ctx.keccak_duplex_batch([("absorb", in_len), ("squeeze", out_len)], data, tag=b"")
    assert np.array_equal(got, want)


def _raw(ctx, dg, n, tag, tag_len, ops, n_ops, inp, out):
    return lib.load().b200g16_keccak_duplex_batch(ctx.h, dg, n, tag, tag_len, ops, n_ops, inp, out)


def test_argument_errors_write_nothing(ctx):
    torch = pytest.importorskip("torch")
    n = 4
    rs = np.random.Generator(np.random.PCG64(23))
    dg = lib.keccak_digests(n, [b"x"] * n)
    dg["state"] = rs.integers(0, 1 << 63, size=(n, 25), dtype=np.uint64)
    ops, A, S = lib.duplex_script([("absorb", 10), ("squeeze", 10)])
    inp = rand_bytes(rs, (n, A))
    out = np.full((n, S), 7, dtype=np.uint8)
    tag = np.zeros(80, dtype=np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    before = dg.tobytes()
    bad_kind = ops.copy()
    bad_kind[1, 0] = 2
    bad_pos = dg.copy()
    bad_pos["squeeze_pos"][2] = 137
    bad_pos_a = dg.copy()
    bad_pos_a["absorb_pos"][3] = 1 << 31
    huge = 1 << 40
    big_ops = np.array([[0, 1 << 30], [1, 1 << 30]], dtype=np.uint32)
    cases = {
        "tag_len 65": (p(dg), n, p(tag), 65, p(ops), 2, p(inp), p(out)),
        "op kind 2": (p(dg), n, None, 0, p(bad_kind), 2, p(inp), p(out)),
        "null inputs": (p(dg), n, None, 0, p(ops), 2, None, p(out)),
        "null outputs": (p(dg), n, None, 0, p(ops), 2, p(inp), None),
        "n x A overflows": (p(dg), huge, None, 0, p(big_ops), 1, p(inp), p(out)),
        "n x S overflows": (p(dg), huge, None, 0, p(big_ops[1:]), 1, p(inp), p(out)),
        "null digests": (None, n, None, 0, p(ops), 2, p(inp), p(out)),
        "null ops": (p(dg), n, None, 0, None, 2, p(inp), p(out)),
    }
    for name, args in cases.items():
        assert _raw(ctx, *args) == ERR_ARG, name
        assert dg.tobytes() == before and (out == 7).all(), name
    for bad in (bad_pos, bad_pos_a):
        keep = bad.tobytes()
        assert _raw(ctx, p(bad), n, None, 0, p(ops), 2, p(inp), p(out)) == ERR_ARG
        assert bad.tobytes() == keep and (out == 7).all()
    # the device path checks every position before any digest changes
    d_in = torch.from_numpy(inp.reshape(-1).copy()).cuda()
    d_out = torch.full((n * S,), 7, dtype=torch.uint8, device="cuda")
    for bad in (bad_pos, bad_pos_a):
        d_dg = torch.from_numpy(bad.view(np.uint8).copy()).cuda()
        with pytest.raises(lib.B200Error):
            ctx.keccak_duplex_batch_dev(d_dg.data_ptr(), n, [("absorb", 10), ("squeeze", 10)], d_in.data_ptr(),
                                        d_out.data_ptr())
        torch.cuda.synchronize()
        assert d_dg.cpu().numpy().tobytes() == bad.tobytes() and int((d_out != 7).sum()) == 0
    d_dg = torch.from_numpy(dg.view(np.uint8).copy()).cuda()
    dev = lib.load().b200g16_keccak_duplex_batch_dev
    assert dev(ctx.h, C.c_void_p(d_dg.data_ptr()), n, None, 0, p(bad_kind), 2, C.c_void_p(d_in.data_ptr()),
               C.c_void_p(d_out.data_ptr())) == ERR_ARG
    assert dev(ctx.h, C.c_void_p(d_dg.data_ptr()), n, p(tag), 65, p(ops), 2, C.c_void_p(d_in.data_ptr()),
               C.c_void_p(d_out.data_ptr())) == ERR_ARG
    assert dev(ctx.h, C.c_void_p(d_dg.data_ptr()), n, None, 0, p(ops), 2, None, C.c_void_p(d_out.data_ptr())) == ERR_ARG
    torch.cuda.synchronize()
    assert d_dg.cpu().numpy().tobytes() == before and int((d_out != 7).sum()) == 0
    # empty batches and empty scripts succeed and touch nothing
    assert _raw(ctx, p(dg), 0, None, 0, p(ops), 2, None, None) == 0
    assert _raw(ctx, p(dg), n, None, 0, p(ops), 0, None, None) == 0
    assert dg.tobytes() == before
    # an empty script under a tag leaves the fresh tagged state
    e_out, e_dg = ctx.keccak_duplex_batch([], np.zeros((n, 0), dtype=np.uint8), digests=dg, tag=b"\x01\x02")
    assert e_out.shape == (n, 0) and e_dg.tobytes() == lib.keccak_digests(n, b"\x01\x02").tobytes()
    # the ctx still runs a sponge and an MSM correctly
    got, _ = ctx.keccak_duplex_batch([("absorb", 10), ("squeeze", 10)], inp, tag=b"")
    assert np.array_equal(got, ctx.keccak_sponge_batch(inp, 10))
    for i in range(n):
        assert bytes(got[i]) == ok.sponge_hash(bytes(inp[i]), 10)
    g1 = g16.g1_point(g16.G1_GEN)
    ks = rs.integers(0, 1 << 62, size=(2000, 4), dtype=np.uint64)
    sc = rs.integers(0, 1 << 62, size=(2000, 4), dtype=np.uint64)
    bases = ctx.fixed_base_mul(g1, ks, group=1, resident=True)
    try:
        assert np.array_equal(ctx.msm(bases, sc), cport.g1_gen_mul(cport.fr_dot(ks, sc)))
    finally:
        bases.free()
