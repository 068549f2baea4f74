"""GPU parity AT THE BENCHMARKED SIZES (the sizes bench.py times), full outputs against the C restatement:

  prove 2^20 / 2^22   known-discrete-log pk with window tables (oracle/synth.py): each of the five MultiExp outputs
                      == [sum w_i k_i] G, h == C computeH (every element), Ar / Bs / Krs == closed form; through BOTH
                      b200g16_prove (host buffers) and b200g16_prove_dev, three times back to back on one ctx
                      (rotating MSM buffer sets, Bs1 reusing Bs2's sorted lists while its tail still runs,
                      a / b / c arriving on the copy stream), WHIR-shaped witness          /root/reference/mt.go:496
  G2 MSM 2^20         closed form
  NTT 2^22 / 2^24     every output element vs the C port for DIF/DIT x coset x inverse (the 4-column-tile passes of
                      large transforms are only taken at these sizes); computeH 2^22 full output vs the C port
  bench.py --dump-outputs   (small sizes) the written MSM point, commitment and PoK equal their closed forms
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from gnark_whir_b200 import lib
from oracle import cport, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()


@pytest.mark.parametrize("log2n", [20, 22])
def test_prove_known_dlog_key_host_and_device_paths(ctx, log2n):
    N = 1 << log2n
    rs = np.random.Generator(np.random.PCG64(4200 + log2n))
    key = synth.KnownDlogKey(ctx, log2n, seed=77 + log2n, precompute=True)
    try:
        wires = synth.whir_mix(rs, N)
        a, b, c = synth.rand_fr(rs, N - 5), synth.rand_fr(rs, N - 5), synth.rand_fr(rs, N - 5)   # ragged: zero padded
        r, s = synth.rand_fr(rs, 1)[0], synth.rand_fr(rs, 1)[0]
        exp, h_exp = key.expected(wires, a, b, c, r, s)
        for it in range(3):                                   # host buffers: H2D of witness, a, b, c inside
            got, h = ctx.prove(key.handle, wires, a, b, c, r, s, want_h=(it == 0), log2_domain=log2n)
            assert synth.check_proof(got, exp) == [], f"host path, pass {it}"
            if it == 0:
                assert np.array_equal(h, h_exp), "h differs from the C restatement of computeH"
        pad = np.zeros((N, 4), dtype=np.uint64)
        d_w = _dev(wires)
        for it in range(3):                                   # device-resident inputs (computeH works in place)
            bufs = []
            for v in (a, b, c):
                pad[:] = 0
                pad[:v.shape[0]] = v
                bufs.append(_dev(pad))
            torch.cuda.synchronize()
            got = ctx.prove_dev(key.handle, d_w.data_ptr(), bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), r, s)
            assert synth.check_proof(got, exp) == [], f"device path, pass {it}"
            if it == 2:
                assert np.array_equal(bufs[0].cpu().numpy().view(np.uint64), h_exp)
        # interleaved: a lone MSM between two proves must not disturb the rotating buffer sets
        one = ctx.msm(key.vec["a"], d_w.data_ptr(), n=N)
        assert np.array_equal(one, exp["msm_a"])
        got, _ = ctx.prove(key.handle, wires, a, b, c, r, s)
        assert synth.check_proof(got, exp) == []
    finally:
        key.free()


def test_msm_g2_2p20_closed_form(ctx):
    rs = np.random.Generator(np.random.PCG64(31337))
    n = 1 << 20
    ks = synth.rand_fr(rs, n)
    bases = ctx.fixed_base_mul(synth.G2, ks, group=2, resident=True)
    for sc in (synth.rand_fr(rs, n), synth.whir_mix(rs, n)):
        want = cport.g2_gen_mul(cport.fr_dot(ks, sc))
        assert np.array_equal(ctx.msm(bases, sc), want)
        assert np.array_equal(ctx.msm(bases, _dev(sc).data_ptr(), n=n), want)
    bases.precompute(0)
    sc = synth.whir_mix(rs, n)
    assert np.array_equal(ctx.msm(bases, sc), cport.g2_gen_mul(cport.fr_dot(ks, sc)))
    bases.free()


@pytest.mark.parametrize("log2n", [22, 24])
def test_ntt_full_output_vs_c_port(ctx, log2n):
    rs = np.random.Generator(np.random.PCG64(900 + log2n))
    x = synth.rand_fr(rs, 1 << log2n)
    for inverse in (False, True):
        for coset in (False, True):
            for dec in (lib.DIF, lib.DIT):
                got = ctx.ntt(x, inverse=inverse, coset=coset, decimation=dec)
                want = cport.ntt(x, inverse=inverse, coset=coset, decimation=dec)
                assert np.array_equal(got, want), (log2n, inverse, coset, dec)


def test_compute_h_2p22_full_output_vs_c_port(ctx):
    rs = np.random.Generator(np.random.PCG64(2222))
    n = 1 << 22
    a, b, c = synth.rand_fr(rs, n - 3), synth.rand_fr(rs, n - 3), synth.rand_fr(rs, n - 3)      # zero padded to 2^22
    assert np.array_equal(ctx.compute_h(a, b, c, 22), cport.compute_h(a, b, c, 22))


def _run_bench(out_dir, *args):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extras",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]


def _load_point(path, rows):
    w = np.load(path)
    assert w.dtype == np.float64 and w.shape == (rows, 8)
    return w.astype("<u4").view("<u8").reshape(-1).astype(np.uint64)


def test_bench_dump_outputs_msm(tmp_path):
    log2n = 14
    _run_bench(tmp_path, "--logn", str(log2n))
    assert sorted(os.listdir(tmp_path)) == ["msm_g1.npy"]
    rs = np.random.Generator(np.random.PCG64(bench.SEED))       # bench.run_b200's inputs on rank 0
    ks = bench.rand_fr(rs, 1 << log2n)
    sc = bench.rand_fr(rs, 1 << log2n)
    assert np.array_equal(_load_point(tmp_path / "msm_g1.npy", 2), cport.g1_gen_mul(cport.fr_dot(ks, sc)))


def test_bench_dump_outputs_prove(tmp_path):
    L = 10
    _run_bench(tmp_path, "--workload", "prove", "--prove-logn", str(L))
    g1 = ["ar", "bs1", "commitment", "krs", "msm_a", "msm_b1", "msm_k", "msm_z", "pok"]
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}.npy" for n in g1 + ["bs", "msm_b2"])
    for n in g1:
        _load_point(tmp_path / f"{n}.npy", 2)
    for n in ("bs", "msm_b2"):
        _load_point(tmp_path / f"{n}.npy", 4)
    N = 1 << L                                                   # bench.prove_bench's inputs
    rs = np.random.Generator(np.random.PCG64(bench.SEED + 17 * L))
    wires = synth.whir_mix(rs, N)
    for n in (N, N, N, 1, 1):                                    # a, b, c, r, s
        bench.rand_fr(rs, n)
    nc = N // 8
    kc = bench.rand_fr(rs, 2 * nc).reshape(2, nc, 4)
    committed = wires[1:1 + nc]
    assert np.array_equal(_load_point(tmp_path / "commitment.npy", 2), cport.g1_gen_mul(cport.fr_dot(kc[0], committed)))
    assert np.array_equal(_load_point(tmp_path / "pok.npy", 2), cport.g1_gen_mul(cport.fr_dot(kc[1], committed)))
