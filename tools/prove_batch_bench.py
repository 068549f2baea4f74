"""Batch prove and batch MSM against loops of single calls, on one GPU -> profiles/r03d_prove_batch.jsonl (or --out).

Line 1: the GPU's name, power limit and max SM clock, read in the same process.  Then one line per configuration:
  prove_dev  b200g16_prove_batch_dev on k device-resident witnesses against a loop of k b200g16_prove_dev calls over
             the same inputs (log2 N in --prove-logs, k in --ks), known-discrete-log key with window tables;
  prove_host b200g16_prove_batch from host arrays against a loop of b200g16_prove (--host-log);
  msm        b200g16_msm_g1_batch / _g2_batch (device scalars) against a loop of b200g16_msm_g1_dev / _g2_dev.
Every configuration is gated on the closed forms (oracle/synth.py: the first and the last proof / row) before it is
timed.  Times: median of --reps calls each (host clock around a call, which ends in a stream synchronisation), per
proof (or per vector), the loop / batch ratio, and the batch call's b200g16_last_timings phases."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gnark_whir_b200 import lib  # noqa: E402
from oracle import cport  # noqa: E402
from oracle.synth import G1, G2, KnownDlogKey, check_proof, rand_fr, whir_mix  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def median_ms(fn, reps, before=None):
    ts = []
    for _ in range(reps):
        if before:
            before()
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def prove_rows(ctx, key, k, rs, device, reps, torch):
    N = key.N
    ncons = N - 1
    wires = np.stack([whir_mix(rs, N) for _ in range(k)])
    abc = [np.stack([rand_fr(rs, ncons) for _ in range(k)]) for _ in range(3)]
    r, s = rand_fr(rs, k), rand_fr(rs, k)
    gate = sorted({0, k - 1})
    exp = {j: key.expected(wires[j], abc[0][j], abc[1][j], abc[2][j], r[j], s[j], nthreads=0)[0] for j in gate}
    if device:
        pad = lambda x: np.concatenate([x, np.zeros((k, N - ncons, 4), dtype=np.uint64)], axis=1).reshape(-1, 4)
        dw = torch.from_numpy(wires.reshape(-1, 4).view(np.int64)).cuda()
        src = [torch.from_numpy(pad(x).view(np.int64)).cuda() for x in abc]
        work = [torch.empty_like(x) for x in src]

        def refill():
            for w, x in zip(work, src):
                w.copy_(x)
            torch.cuda.synchronize()
        p = [w.data_ptr() for w in work]
        row = N * 32
        batch = lambda: ctx.prove_batch_dev(key.handle, k, dw.data_ptr(), p[0], p[1], p[2], r, s)
        loop = lambda: [ctx.prove_dev(key.handle, dw.data_ptr() + j * N * 32, p[0] + j * row, p[1] + j * row,
                                      p[2] + j * row, r[j], s[j]) for j in range(k)]
    else:
        refill = None
        batch = lambda: ctx.prove_batch(key.handle, wires, abc[0], abc[1], abc[2], r, s)
        loop = lambda: [ctx.prove(key.handle, wires[j], abc[0][j], abc[1][j], abc[2][j], r[j], s[j])[0] for j in range(k)]
    if refill:
        refill()
    got = batch()
    for j in gate:
        assert check_proof(got[j], exp[j]) == [], f"batch proof {j} differs from the closed form"
    if refill:
        refill()
    got = loop()
    for j in gate:
        assert check_proof(got[j], exp[j]) == [], f"loop proof {j} differs from the closed form"
    t_loop = median_ms(loop, reps, refill)
    t_batch = median_ms(batch, reps, refill)
    phases = ctx.last_timings()
    return t_batch, t_loop, phases


def msm_rows(ctx, b, ks, n, k, group, rs, reps, torch):
    sc = np.stack([rand_fr(rs, n) for _ in range(k)])
    dev = torch.from_numpy(sc.reshape(-1, 4).view(np.int64)).cuda()
    got = ctx.msm_batch(b, dev.data_ptr(), n=n, k=k)
    mul = cport.g1_gen_mul if group == 1 else cport.g2_gen_mul
    for j in sorted({0, k - 1}):
        assert np.array_equal(got[j], mul(cport.fr_dot(ks[:n], sc[j]))), f"msm row {j} differs from the closed form"
    batch = lambda: ctx.msm_batch(b, dev.data_ptr(), n=n, k=k)
    loop = lambda: [ctx.msm(b, dev.data_ptr() + j * n * 32, n=n) for j in range(k)]
    t_loop = median_ms(loop, reps)
    t_batch = median_ms(batch, reps)
    return t_batch, t_loop, ctx.last_timings()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03d_prove_batch.jsonl"))
    ap.add_argument("--prove-logs", default="16,18,20,22")
    ap.add_argument("--ks", default="1,2,4,8,16,32")
    ap.add_argument("--host-log", type=int, default=20)
    ap.add_argument("--msm-logs", default="16,18,20,22")
    ap.add_argument("--g2-log", type=int, default=20, help="0: no G2 rows")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    ks = [int(x) for x in a.ks.split(",")]
    rs = np.random.Generator(np.random.PCG64(20261023))
    lines = [gpu_info()]
    print(json.dumps(lines[0]), flush=True)

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
        with open(a.out, "w") as f:
            for x in lines:
                f.write(json.dumps(x) + "\n")
    with lib.Context(0) as ctx:
        for L in [int(x) for x in a.prove_logs.split(",") if x]:
            key = KnownDlogKey(ctx, L, seed=1000 + L)
            try:
                for mode in (["prove_dev", "prove_host"] if L == a.host_log else ["prove_dev"]):
                    for k in ks:
                        tb, tl, ph = prove_rows(ctx, key, k, rs, mode == "prove_dev", a.reps, torch)
                        emit({"kind": mode, "log2n": L, "k": k, "batch_ms": round(tb, 3), "loop_ms": round(tl, 3),
                              "batch_ms_per_proof": round(tb / k, 3), "loop_ms_per_proof": round(tl / k, 3),
                              "loop_over_batch": round(tl / tb, 3), "reps": a.reps,
                              "batch_phases_ms": [round(x, 3) for x in ph]})
            finally:
                key.free()
        for group, logs in ((1, [int(x) for x in a.msm_logs.split(",") if x]), (2, [a.g2_log] if a.g2_log else [])):
            for L in logs:
                n = 1 << L
                kk = rand_fr(rs, n)
                b = ctx.fixed_base_mul(G1 if group == 1 else G2, kk, group=group, resident=True)
                try:
                    b.precompute(0)
                    for k in ks:
                        tb, tl, ph = msm_rows(ctx, b, kk, n, k, group, rs, a.reps, torch)
                        emit({"kind": "msm_g%d_table" % group, "log2n": L, "window": b.window(), "k": k,
                              "batch_ms": round(tb, 3), "loop_ms": round(tl, 3),
                              "batch_ms_per_vector": round(tb / k, 3), "loop_over_batch": round(tl / tb, 3),
                              "reps": a.reps, "batch_phases_ms": [round(x, 3) for x in ph]})
                finally:
                    b.free()


if __name__ == "__main__":
    main()
