"""Measure b200g16_verify_batch against single b200g16_verify calls in the same process.

For k in {1, 16, 256, 1024, 4096, 16384} x {with, without a BSB22 commitment}, n_public = 8, simulated proofs
(tests/test_gpu_verify_batch.py SimBatch: known-dlog verifying key, proofs minted on the GPU).  Every timed
configuration is gated first (untimed): the valid batch must be accepted with every ok_each entry set, and the same
batch with one tampered proof (Krs + G at k/2) must be rejected naming exactly that proof; that call's phase times
give the cost of the per-proof pass on a failing batch.  Then the median of --reps calls on the valid batch (host
clock around the call, which ends in a device synchronise; inputs come from host memory as a caller's would).

Writes one JSON line per configuration, after a first line with the card's name, power limit and max SM clock.
    python tools/verify_batch_bench.py --out profiles/r03b_verify_batch.jsonl
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from gnark_whir_b200 import lib  # noqa: E402
from tests.test_gpu_verify_batch import G1, SimBatch  # noqa: E402

PHASES = ["upload", "per_proof", "fold_msm", "product", "final_exp", "per_proof_pass"]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def coeff_words(rng, n):
    c = [rng.randrange(1, 1 << 128) for _ in range(n)]
    return np.array([(x & (2**64 - 1), x >> 64) for x in c], dtype=np.uint64).reshape(n, 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03b_verify_batch.jsonl"))
    ap.add_argument("--ks", default="1,16,256,1024,4096,16384")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--n-public", type=int, default=8)
    args = ap.parse_args()
    ks = [int(x) for x in args.ks.split(",")]
    rng = random.Random(20261020)
    lines = [dict(gpu_info(), kind="device")]
    print(json.dumps(lines[0]), flush=True)
    with lib.Context(0) as ctx:
        def batch(sim, arrays, coeffs, **kw):
            ar, bs, krs, pubs, com, pok = arrays
            v = sim.vk
            return ctx.verify_batch(v.G1_Alpha, v.G2_Beta, v.G2_Gamma, v.G2_Delta, v.G1_K, ar, bs, krs, pubs, coeffs,
                                    commitments=com, poks=pok, ped_g=v.PedersenG if v.has_commitment else None,
                                    ped_g_sigma_neg=v.PedersenGSigmaNeg if v.has_commitment else None, **kw)

        single_ms = {}
        for com in (False, True):
            sim = SimBatch(ctx, 4, args.n_public, com, seed=7 + com)
            ar, bs, krs, pubs, coms, poks = sim.arrays()
            v = sim.vk

            def one(i):
                return ctx.verify(v.G1_Alpha, v.G2_Beta, v.G2_Gamma, v.G2_Delta, v.G1_K, ar[i], bs[i], krs[i], pubs[i],
                                  commitment=coms[i] if com else None, pok=poks[i] if com else None,
                                  ped_g=v.PedersenG if com else None, ped_g_sigma_neg=v.PedersenGSigmaNeg if com else None)
            for i in range(4):                                   # warm-up and gate
                assert one(i)
            ts = []
            for r in range(args.reps):
                t0 = time.perf_counter()
                ok = one(r % 4)
                ts.append((time.perf_counter() - t0) * 1e3)
                assert ok
            single_ms[com] = statistics.median(ts)
            rec = {"kind": "single_verify", "commitment": com, "n_public": args.n_public,
                   "median_ms": round(single_ms[com], 3), "min_ms": round(min(ts), 3)}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
            warm = batch(sim, sim.arrays(), coeff_words(rng, 8 if com else 4))   # warm the batch path
            assert warm[0]

        for com in (False, True):
            for k in ks:
                sim = SimBatch(ctx, k, args.n_public, com, seed=1000 + k + com)
                arrays = sim.arrays()
                co = coeff_words(rng, 2 * k if com else k)
                ok, each = batch(sim, arrays, co)
                assert ok and each.all(), (k, com)
                t = k // 2
                bad = list(arrays)
                bad[2] = arrays[2].copy()
                bad[2][t] = lib.g1_add(bad[2][t], G1)
                t0 = time.perf_counter()
                ok, each = batch(sim, bad, co)
                fail_ms = (time.perf_counter() - t0) * 1e3
                fail_phases = ctx.last_timings()
                assert not ok and np.flatnonzero(~each).tolist() == [t], (k, com)
                ts, ph = [], []
                for _ in range(args.reps):
                    co = coeff_words(rng, 2 * k if com else k)
                    t0 = time.perf_counter()
                    ok, _ = batch(sim, arrays, co)
                    ts.append((time.perf_counter() - t0) * 1e3)
                    ph.append(ctx.last_timings())
                    assert ok
                med = statistics.median(ts)
                rec = {"kind": "verify_batch", "k": k, "commitment": com, "n_public": args.n_public, "reps": args.reps,
                       "median_ms": round(med, 3), "min_ms": round(min(ts), 3),
                       "phases_ms": {PHASES[i]: round(statistics.median(p[i] for p in ph), 3) for i in range(5)},
                       "proofs_per_s": round(k / med * 1e3, 1),
                       "single_verify_ms": round(single_ms[com], 3),
                       "call_vs_single": round(med / single_ms[com], 3),
                       "throughput_vs_single_loop": round(k * single_ms[com] / med, 1),
                       "failing_batch_ms": round(fail_ms, 3),
                       "failing_batch_phases_ms": {PHASES[i]: round(x, 3) for i, x in enumerate(fail_phases)}}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
