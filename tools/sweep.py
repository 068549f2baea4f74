"""Config sweeps of BASELINE.json (run under gpurun): one JSON line per point -> stdout.

  configs[1]  G1 MSM 2^16..2^24 (uniform + WHIR-shaped scalars), G2 MSM 2^16..2^22, each checked
              against the closed form [sum s_i k_i]G computed by the C oracle
  configs[2]  Fr NTT / computeH 2^18..2^26 (round-trip checked)
  configs[3]  Keccak: raw 2^24 permutations, Merkle recompute for Q in {64,128,256} queries
              (latency) and 2^20 independent paths (throughput), checked against the C oracle
Timing: CUDA events on the library stream (b200g16_last_timings) or torch events around the call,
best of 3 after one warm-up; inputs resident in HBM."""
import json
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from gnark_whir_b200 import groth16 as g16  # noqa: E402
from gnark_whir_b200 import lib  # noqa: E402
from oracle import cport  # noqa: E402  (checker only)

rs = np.random.Generator(np.random.PCG64(20261018))
TMAD_PEAK = None


def rand_fr(n):
    a = rs.integers(0, 1 << 62, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 60) - 1)
    return a


def emit(**kw):
    print(json.dumps(kw), flush=True)


def t_ms(fn, reps=3):
    fn()
    best = 1e30
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def window_sweep(ctx):
    """Table-mode window width per (shard) size: whole-MSM device time for c = 15..21 at 2^18..2^22 (the per-GPU shard
    sizes of an 8-way sharded 2^21..2^24 job), uniform scalars.  Feeds msm_pick_table_window."""
    gen = g16.g1_point(g16.G1_GEN)
    arg = [a for a in sys.argv if a.startswith("--logs=")]
    for logn in ([int(x) for x in arg[0][7:].split(",")] if arg else (18, 19, 20, 21, 22, 24)):
        n = 1 << logn
        ks = rand_fr(n)
        sc = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
        want = cport.g1_gen_mul(cport.fr_dot(ks, sc.cpu().numpy().view(np.uint64)))
        for c in (range(15, 22) if logn < 24 else (20, 21, 22)):
            bases = ctx.fixed_base_mul(gen, ks, group=1, resident=True)
            bases.precompute(c)
            best, ok = None, True
            for _ in range(5):
                ok = ok and bool(np.array_equal(ctx.msm(bases, sc.data_ptr(), n=n), want))
                ph = ctx.last_timings()
                if best is None or sum(ph) < sum(best):
                    best = ph
            emit(config="msm_table_window", log2n=logn, window_bits=c, adds_per_point=ctx.msm_plan(bases, n)[1],
                 device_ms=round(sum(best), 3), phases_ms=[round(x, 3) for x in best], bit_exact_vs_oracle=ok)
            bases.free()


def affine_sweep(ctx):
    """Batched-affine bucket accumulation (csrc/msm_affine.cuh) against the mixed XYZZ accumulation on the same sorted
    lists: G1 2^20..2^24 and G2 2^20..2^22, window tables, uniform and WHIR-shaped scalars, pair-tree levels 1..4."""
    tbl = torch.from_numpy(g16.fr_array(list(range(256))).view(np.int64)).cuda()
    args = [a for a in sys.argv if a.startswith("--logs=")]
    for group, logs in ((1, [20, 22, 24]), (2, [20, 22])):
        if args:
            logs = [int(x) for x in args[0][7:].split(",") if (group == 1) == (int(x) > 0)]
            logs = [abs(x) for x in logs]
        gen = g16.g1_point(g16.G1_GEN) if group == 1 else g16.g2_point(g16.G2_GEN)
        for logn in logs:
            n = 1 << logn
            ks = rand_fr(n)
            bases = ctx.fixed_base_mul(gen, ks, group=group, resident=True)
            bases.precompute(0)
            d_uni = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
            u = torch.rand(n, device="cuda")
            sv = torch.randint(0, 256, (n,), device="cuda")
            d_mix = d_uni.clone()
            m01, mb = u < 0.4, (u >= 0.4) & (u < 0.7)
            d_mix[m01] = tbl[sv[m01] & 1]
            d_mix[mb] = tbl[sv[mb]]
            for name, d_sc in (("uniform", d_uni), ("whir_mix", d_mix)):
                host_sc = d_sc.cpu().numpy().view(np.uint64)
                dot = cport.fr_dot(ks, host_sc)
                want = cport.g1_gen_mul(dot) if group == 1 else ctx.fixed_base_mul(gen, dot.reshape(1, 4), group=2)[0]
                for mode, levels in ((0, 0), (2, 1), (2, 2), (2, 3), (2, 4)):
                    ctx.set_msm_batch_affine(mode, levels, 0)
                    best, ok = None, True
                    for _ in range(4):
                        ok = ok and bool(np.array_equal(ctx.msm(bases, d_sc.data_ptr(), n=n), want))
                        ph = ctx.last_timings()
                        if best is None or sum(ph) < sum(best):
                            best = ph
                    emit(config="msm_batch_affine", group=f"G{group}", log2n=logn, scalars=name,
                         accumulate="xyzz" if mode == 0 else f"affine_L{levels}", device_ms=round(sum(best), 3),
                         accumulate_ms=round(best[2], 3), phases_ms=[round(x, 3) for x in best], bit_exact_vs_oracle=ok)
                ctx.set_msm_batch_affine(0, 0, 0)
            bases.free()
            del d_uni, d_mix


def affine_debug(ctx):
    """Batched-affine against XYZZ on the same inputs, small sizes, every level count."""
    for logn in (8, 10, 12, 14, 15, 16, 17):
        n = 1 << logn
        ks = rand_fr(n)
        bases = ctx.fixed_base_mul(g16.g1_point(g16.G1_GEN), ks, group=1, resident=True)
        d_sc = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
        ctx.set_msm_batch_affine(0, 0, 0)
        want = ctx.msm(bases, d_sc.data_ptr(), n=n)
        res = {}
        for name, levels, mp in (("L0", 1, 1 << 30), ("L1", 1, 1), ("L2", 2, 1), ("L3", 3, 1), ("L4", 4, 1)):
            ctx.set_msm_batch_affine(2, levels, mp)
            res[name] = bool(np.array_equal(ctx.msm(bases, d_sc.data_ptr(), n=n), want))
        emit(config="affine_debug", log2n=logn, plan=ctx.msm_plan(bases, n), **res)
        bases.free()
    ctx.set_msm_batch_affine(0, 3, 192)


def window_mix_sweep(ctx):
    """Table window for WITNESS-shaped scalars (40% 0/1, 30% bytes, 30% uniform: the A / B1 / B2 / K MSMs of a prove) next
    to uniform ones, G1 and G2, c = 15..20 at 2^18..2^22: whole-MSM device time, checked against the closed form."""
    tbl = torch.from_numpy(g16.fr_array(list(range(256))).view(np.int64)).cuda()
    arg = [a for a in sys.argv if a.startswith("--logs=")]
    logs = [int(x) for x in arg[0][7:].split(",")] if arg else [18, 20, 22]
    for group in (1, 2):
        gen = g16.g1_point(g16.G1_GEN) if group == 1 else g16.g2_point(g16.G2_GEN)
        for logn in logs:
            n = 1 << logn
            ks = rand_fr(n)
            d_uni = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
            u = torch.rand(n, device="cuda")
            sv = torch.randint(0, 256, (n,), device="cuda")
            d_mix = d_uni.clone()
            m01, mb = u < 0.4, (u >= 0.4) & (u < 0.7)
            d_mix[m01] = tbl[sv[m01] & 1]
            d_mix[mb] = tbl[sv[mb]]
            want = {}
            for name, d_sc in (("uniform", d_uni), ("whir_mix", d_mix)):
                dot = cport.fr_dot(ks, d_sc.cpu().numpy().view(np.uint64))
                want[name] = cport.g1_gen_mul(dot) if group == 1 else ctx.fixed_base_mul(gen, dot.reshape(1, 4), group=2)[0]
            for c in range(15, 21):
                bases = ctx.fixed_base_mul(gen, ks, group=group, resident=True)
                bases.precompute(c)
                for name, d_sc in (("uniform", d_uni), ("whir_mix", d_mix)):
                    best, ok = None, True
                    for _ in range(4):
                        ok = ok and bool(np.array_equal(ctx.msm(bases, d_sc.data_ptr(), n=n), want[name]))
                        ph = ctx.last_timings()
                        if best is None or sum(ph) < sum(best):
                            best = ph
                    emit(config="msm_table_window_mix", group=f"G{group}", log2n=logn, scalars=name, window_bits=c,
                         adds_per_point=ctx.msm_plan(bases, n)[1], device_ms=round(sum(best), 3),
                         phases_ms=[round(x, 3) for x in best], bit_exact_vs_oracle=ok)
                bases.free()
            del d_uni, d_mix


def reduce_ab(ctx):
    """Bucket-reduction phase of the G1 MSM with a c = 20 table at 2^20 / 2^21 / 2^24 points (uniform scalars); run once
    with B200G16_REDUCE_INLINE=0 and once with 1 (the knob is read once per process)."""
    import os
    g2 = "--g2" in sys.argv
    gen = g16.g2_point(g16.G2_GEN) if g2 else g16.g1_point(g16.G1_GEN)
    arg = [a for a in sys.argv if a.startswith("--logs=")]
    for logn in ([int(x) for x in arg[0][7:].split(",")] if arg else (20, 21, 24)):
        n = 1 << logn
        ks = rand_fr(n)
        sc = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
        dot = cport.fr_dot(ks, sc.cpu().numpy().view(np.uint64))
        want = ctx.fixed_base_mul(gen, dot.reshape(1, 4), group=2)[0] if g2 else cport.g1_gen_mul(dot)
        bases = ctx.fixed_base_mul(gen, ks, group=2 if g2 else 1, resident=True)
        bases.precompute(20)
        best, ok = None, True
        for _ in range(6):
            ok = ok and bool(np.array_equal(ctx.msm(bases, sc.data_ptr(), n=n), want))
            ph = ctx.last_timings()
            if best is None or sum(ph) < sum(best):
                best = ph
        emit(config="msm_reduce_ab", group="G2" if g2 else "G1", reduce_inline=os.environ.get("B200G16_REDUCE_INLINE", "default"),
             log2n=logn,
             device_ms=round(sum(best), 3), phases_ms=[round(x, 3) for x in best], bit_exact_vs_oracle=ok)
        bases.free()


def merkle_sweep(ctx):
    """Latency kernel of the Merkle recompute (csrc/keccak.cu k_merkle_paths_warp): warps per CTA x exchange mechanism
    (B200G16_MERKLE_WARP = 10 * warps + smem) at 64..4096 paths, height 20, 512 B leaves, byte-exact vs the C oracle."""
    import os
    from ctypes import c_void_p
    L = lib.load()
    height, leaf_len = 20, 512
    for q in (64, 128, 256, 1024, 4096):
        leaves = torch.randint(0, 256, (q, leaf_len), dtype=torch.uint8, device="cuda")
        sib = torch.randint(0, 256, (q, 32), dtype=torch.uint8, device="cuda")
        auth = torch.randint(0, 256, (q, height - 1, 32), dtype=torch.uint8, device="cuda")
        idx = torch.randint(0, 1 << 20, (q,), dtype=torch.int64, device="cuda")
        roots = torch.zeros((q, 32), dtype=torch.uint8, device="cuda")
        exp = cport.merkle_paths(leaves.cpu().numpy(), sib.cpu().numpy(), auth.cpu().numpy(),
                                 idx.cpu().numpy().astype(np.uint64))

        def run():
            lib._check(L.b200g16_keccak_merkle_paths_dev(ctx.h, c_void_p(leaves.data_ptr()), leaf_len,
                                                         c_void_p(sib.data_ptr()), c_void_p(auth.data_ptr()),
                                                         c_void_p(idx.data_ptr()), height, q, None,
                                                         c_void_p(roots.data_ptr()), None))
        for cfg in (40, 20, 10, 41, 21, 11):
            os.environ["B200G16_MERKLE_WARP"] = str(cfg)
            roots.zero_()
            ms = t_ms(run, reps=10)
            ok = bool(np.array_equal(roots.cpu().numpy(), exp))
            # 50 calls enqueued back to back between one pair of events: the kernel's own time without the launch gap
            ms_train = t_ms(lambda: [run() for _ in range(50)], reps=3) / 50
            emit(config="keccak_merkle_paths_warp", paths=q, warps_per_cta=cfg // 10, exchange="smem" if cfg % 10 else "shfl",
                 ms=round(ms, 4), ms_back_to_back=round(ms_train, 4), byte_exact_vs_oracle=ok)
    os.environ.pop("B200G16_MERKLE_WARP", None)


def main():
    global TMAD_PEAK
    big = "--big" in sys.argv
    ctx = lib.Context(0)
    if "--windows" in sys.argv:
        window_sweep(ctx)
        ctx.close()
        return
    if "--affine-debug" in sys.argv:
        affine_debug(ctx)
        ctx.close()
        return
    if "--windows-mix" in sys.argv:
        window_mix_sweep(ctx)
        ctx.close()
        return
    if "--reduce-ab" in sys.argv:
        reduce_ab(ctx)
        ctx.close()
        return
    if "--merkle" in sys.argv:
        merkle_sweep(ctx)
        ctx.close()
        return
    if "--affine" in sys.argv:
        affine_sweep(ctx)
        ctx.close()
        return
    rate, _ = ctx.modmul_probe(8, 4, 2000)
    TMAD_PEAK = rate * 136 / 1e12
    emit(probe="modmul", Gmodmul_s=round(rate / 1e9, 2), TMAD_s=round(TMAD_PEAK, 3))
    tbl = torch.from_numpy(g16.fr_array(list(range(256))).view(np.int64)).cuda()

    # ---- MSM sweeps
    only_ntt = "--ntt" in sys.argv      # NTT / computeH section alone, up to 2^26
    big = big or only_ntt
    for group, logs in ((1, [16, 18, 20, 22, 24]), (2, [16, 18, 20, 22])):
        gen = g16.g1_point(g16.G1_GEN) if group == 1 else g16.g2_point(g16.G2_GEN)
        for logn in ([] if only_ntt else logs):
            n = 1 << logn
            ks = rand_fr(n)
            bases = ctx.fixed_base_mul(gen, ks, group=group, resident=True)
            sc = rand_fr(n)
            d_uni = torch.from_numpy(sc.view(np.int64)).cuda()
            u = torch.rand(n, device="cuda")
            sv = torch.randint(0, 256, (n,), device="cuda")
            d_mix = d_uni.clone()
            m01, mb = u < 0.4, (u >= 0.4) & (u < 0.7)
            d_mix[m01] = tbl[sv[m01] & 1]
            d_mix[mb] = tbl[sv[mb]]
            for name, d_sc, table in (("uniform", d_uni, False), ("whir_mix", d_mix, False),
                                      ("uniform", d_uni, True), ("whir_mix", d_mix, True)):
                if table and not bases.window():
                    bases.precompute(0)           # window table over the resident bases, built once
                c_bits, adds = ctx.msm_plan(bases, n)
                best, out = None, None
                for _ in range(4):
                    out = ctx.msm(bases, d_sc.data_ptr(), n=n)
                    ph = ctx.last_timings()
                    if best is None or sum(ph) < sum(best):
                        best = ph
                host_sc = d_sc.cpu().numpy().view(np.uint64)
                if group == 1:
                    ok = bool(np.array_equal(out, cport.g1_gen_mul(cport.fr_dot(ks, host_sc))))
                else:       # G2: closed form [sum s_i k_i]G2 through the library's own fixed-base kernel
                    dot = cport.fr_dot(ks, host_sc)
                    ok = bool(np.array_equal(out, ctx.fixed_base_mul(gen, dot.reshape(1, 4), group=2)[0]))
                ms = sum(best)
                emit(config="msm", group=f"G{group}", log2n=logn, scalars=name, window_table=table, window_bits=c_bits,
                     adds_per_point=adds, device_ms=round(ms, 3),
                     Mpts_s=round(n / ms / 1e3, 2), phases_ms=[round(x, 3) for x in best], bit_exact_vs_oracle=ok)
            bases.free()
            del d_uni, d_mix
    if "--msm" in sys.argv:     # the MSM section alone
        ctx.close()
        return

    # ---- NTT / computeH sweeps
    for logn in ([18, 20, 22, 24, 26] if big else [18, 20, 22, 24]):
        n = 1 << logn
        a = torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
        ref = a.clone()
        ctx.ntt_dev(a.data_ptr(), logn, coset=True, decimation=lib.DIF)
        ctx.ntt_dev(a.data_ptr(), logn, inverse=True, coset=True, decimation=lib.DIT)
        roundtrip = bool(torch.equal(a, ref))
        ms = t_ms(lambda: ctx.ntt_dev(a.data_ptr(), logn, decimation=lib.DIF))
        tmad = (n / 2) * logn * 136 / ms / 1e9
        emit(config="ntt", log2n=logn, ms=round(ms, 4), GBs_64N=round(64 * n / ms / 1e6, 1), TMAD_s=round(tmad, 3),
             frac_integer_peak=round(tmad / TMAD_PEAK, 3), roundtrip_exact=roundtrip)
        b, c = torch.from_numpy(rand_fr(n).view(np.int64)).cuda(), torch.from_numpy(rand_fr(n).view(np.int64)).cuda()
        ms = t_ms(lambda: ctx.compute_h_dev(a.data_ptr(), b.data_ptr(), c.data_ptr(), logn))
        emit(config="compute_h", log2n=logn, ms=round(ms, 4), GBs_576N=round(576 * n / ms / 1e6, 1),
             phases_ms=[round(x, 4) for x in ctx.last_timings()])
        del a, b, c, ref

    if only_ntt:
        ctx.close()
        return
    # ---- Keccak
    nk = 1 << 24
    st = torch.randint(0, 1 << 62, (nk, 25), dtype=torch.int64, device="cuda")
    ms = t_ms(lambda: ctx.keccak_f_batch_dev(st.data_ptr(), nk))
    emit(config="keccak_f_batch", states=nk, ms=round(ms, 4), Gperm_s=round(nk / ms / 1e6, 3), GBs_400B=round(400 * nk / ms / 1e6, 1))
    del st
    from ctypes import c_void_p
    L = lib.load()
    height, leaf_len = 20, 512
    for q in (64, 128, 256, 1 << 20):
        leaves = torch.randint(0, 256, (q, leaf_len), dtype=torch.uint8, device="cuda")
        sib = torch.randint(0, 256, (q, 32), dtype=torch.uint8, device="cuda")
        auth = torch.randint(0, 256, (q, height - 1, 32), dtype=torch.uint8, device="cuda")
        idx = torch.randint(0, 1 << 20, (q,), dtype=torch.int64, device="cuda")
        roots = torch.zeros((q, 32), dtype=torch.uint8, device="cuda")

        def run():
            lib._check(L.b200g16_keccak_merkle_paths_dev(ctx.h, c_void_p(leaves.data_ptr()), leaf_len,
                                                         c_void_p(sib.data_ptr()), c_void_p(auth.data_ptr()),
                                                         c_void_p(idx.data_ptr()), height, q, None,
                                                         c_void_p(roots.data_ptr()), None))
        ms = t_ms(run)
        m = min(q, 512)
        exp = cport.merkle_paths(leaves[:m].cpu().numpy(), sib[:m].cpu().numpy(), auth[:m].cpu().numpy(),
                                 idx[:m].cpu().numpy().astype(np.uint64))
        ok = bool(np.array_equal(roots[:m].cpu().numpy(), exp))
        emit(config="keccak_merkle_paths", paths=q, height=height, leaf_len=leaf_len, ms=round(ms, 4),
             Mpaths_s=round(q / ms / 1e3, 3), Gperm_s=round(24 * q / ms / 1e6, 4), byte_exact_vs_oracle=ok)
    ctx.close()


if __name__ == "__main__":
    main()
