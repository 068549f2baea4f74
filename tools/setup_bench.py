"""Groth16 setup on one GPU (b200g16_setup) against what a caller has without it -> one jsonl line per size.

Line 1: the GPU's name, power limit and max SM clock, read in the same process.  Then, for each 2^log2m constraints
of an oracle.setup_port.synthetic_csr system (--logs):
  gpu_ms          wall time of b200g16_setup from host arrays to resident key + host flags (median of --reps calls
                  after one warm-up call), and its b200g16_last_timings phases;
  cpu_abc_ms      the C restatement of gnark's setupABC (oracle_setup_abc, single-threaded like gnark's) on the
                  host's cores;
  gpu_fixed_ms    today's GPU fixed-base call for the same number of points (b200g16_bases_from_scalars_g1 for
                  |A| + |B| + (N - 1) + |K| + |vk.K| + 3 G1 points, _g2 for |B| + 3 G2 points, random scalars);
  today_ms        cpu_abc_ms + gpu_fixed_ms: what a Go caller gets now (gnark's setupABC, then the GPU's
                  BatchScalarMultiplication).  The K / Z scalar loops gnark also runs on the host are not counted.
Every size is gated before it is timed: b200g16_setup_wire_polys equals the C oracle's A, B, C, and 8 sampled
points of pk.A and pk.G2.B equal b200g16_g1/_g2_scalar_mul of the oracle's scalars."""
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
from oracle import bn254 as bn  # noqa: E402
from oracle import setup_port as sp  # noqa: E402
from oracle.synth import G1, G2, rand_fr  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def free_key(o):
    for n in lib.SETUP_VECTORS:
        if o[n] is not None:
            o[n].free()


def run_size(ctx, log2m, reps, seed):
    d = sp.synthetic_csr(1 << log2m, seed)
    rs = np.random.Generator(np.random.PCG64(seed))
    toxic = rand_fr(rs, 6)
    t0 = time.perf_counter()
    exp = sp.setup_abc(d, toxic[0])
    cpu_abc_ms = (time.perf_counter() - t0) * 1e3
    got = ctx.setup_wire_polys(d, toxic[0])
    if not all(np.array_equal(g, e) for g, e in zip(got, exp)):
        raise SystemExit(f"2^{log2m}: b200g16_setup_wire_polys differs from the C oracle")
    o = ctx.setup(d, *toxic)
    nz_a = np.nonzero(exp[0].any(axis=1))[0]
    nz_b = np.nonzero(exp[1].any(axis=1))[0]
    for j in rs.integers(0, len(nz_a), size=8).tolist():
        if not np.array_equal(o["a"].download(j, 1)[0], lib.g1_scalar_mul(G1, exp[0][nz_a[j]])):
            raise SystemExit(f"2^{log2m}: pk.A[{j}] differs")
    for j in rs.integers(0, len(nz_b), size=8).tolist():
        if not np.array_equal(o["b2"].download(j, 1)[0], lib.g2_scalar_mul(G2, exp[1][nz_b[j]])):
            raise SystemExit(f"2^{log2m}: pk.G2.B[{j}] differs")
    sizes = {n: len(o[n]) for n in ("a", "b", "k", "z", "vk_k")}
    free_key(o)
    times, phases = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        o = ctx.setup(d, *toxic)
        times.append((time.perf_counter() - t0) * 1e3)
        phases.append(ctx.last_timings())
        free_key(o)
    n1 = sum(sizes.values()) + 3
    n2 = sizes["b"] + 3
    sc1, sc2 = rand_fr(rs, n1), rand_fr(rs, n2)
    fixed = []
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        b1 = ctx.fixed_base_mul(G1, sc1, group=1, resident=True)
        b2 = ctx.fixed_base_mul(G2, sc2, group=2, resident=True)
        fixed.append((time.perf_counter() - t0) * 1e3)
        b1.free()
        b2.free()
    gpu_fixed_ms = statistics.median(fixed[1:])
    names = ["upload_check", "powers_lagrange", "acc_L", "acc_R", "acc_O", "k_compact", "points_g1", "points_g2",
             "download"]
    med_phase = {n: round(statistics.median(p[i] for p in phases), 3) for i, n in enumerate(names)}
    gpu_ms = statistics.median(times)
    return {"log2m": log2m, "n_wires": int(d["nb_wires"]), "nnz": [int(d[p + "_row"][-1]) for p in "lro"],
            "sizes": sizes, "gpu_ms": round(gpu_ms, 3), "gpu_ms_all": [round(t, 3) for t in times],
            "phases_ms": med_phase, "cpu_abc_ms": round(cpu_abc_ms, 1), "gpu_fixed_ms": round(gpu_fixed_ms, 3),
            "today_ms": round(cpu_abc_ms + gpu_fixed_ms, 1), "speedup": round((cpu_abc_ms + gpu_fixed_ms) / gpu_ms, 2),
            "gated": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,18,20,22,24")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [json.dumps(gpu_info())]
    print(lines[0], flush=True)
    with lib.Context(0) as ctx:
        for L in [int(x) for x in a.logs.split(",")]:
            row = run_size(ctx, L, a.reps, 1000 + L)
            lines.append(json.dumps(row))
            print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
