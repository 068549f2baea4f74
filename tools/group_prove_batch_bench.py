"""Batch prove over a device group (b200g16_group_prove_batch with a replicated key) against one-ctx
b200g16_prove_batch on the same inputs -> profiles/r03g_group_prove_batch.jsonl (or --out).

Line 1: the name, power limit and max SM clock of every GPU, read in the same process, and the device count.  Then:
  group_prove  log2 N in --logs, n in --ns distinct devices, k = m * n for m in --per-device, host arrays pinned
               (b200g16_host_register) or pageable: ms per call, ms per proof and proofs/s for the group and for one
               ctx on device 0, their ratio, each member's 8 phases, and two host-to-device rates per member: the
               witness upload phase (n_wires * 32 B per proof over phase 0) and all the rows a member reads
               ((n_wires + 3 n_constraints) * 32 B per proof) over the whole call, a lower bound on what its link
               sustained;
  replicate    b200g16_group_pk_replicate of a key with window tables over n devices against b200g16_pk_upload with
               precompute on every device at once (one host thread each), with the bytes the replicas copied.
A configuration needing more devices than the machine has, or more host memory for its inputs than --max-input-gb,
is written as "not measured".  Every line is gated first on a known-discrete-log key's closed forms (oracle/synth.py:
the first and the last proof of the batch).  Inputs: --pool distinct proofs, repeated to k rows.  Times: median of
--reps calls (host clock around a call, which ends in a stream synchronisation on every device)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gnark_whir_b200 import lib  # noqa: E402
from oracle.synth import KnownDlogKey, check_proof, rand_fr, whir_mix  # noqa: E402


def gpu_info():
    rows = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip().splitlines()
    out = []
    for q in rows:
        name, power, clock = [x.strip() for x in q.split(",")]
        out.append({"gpu": name, "power_limit": power, "max_sm_clock": clock})
    return out


def median_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def ranges(k, n):
    base, rem = divmod(k, n)
    out, lo = [], 0
    for i in range(n):
        hi = lo + base + (1 if i < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def make_inputs(key, k, pool, rs):
    """k proofs' rows: `pool` distinct proofs repeated; the closed forms of the first and the last proof."""
    N = key.N
    ncons = N - 1
    p = min(pool, k)
    w0 = np.stack([whir_mix(rs, N) for _ in range(p)])
    abc0 = [np.stack([rand_fr(rs, ncons) for _ in range(p)]) for _ in range(3)]
    r0, s0 = rand_fr(rs, p), rand_fr(rs, p)
    idx = np.arange(k) % p
    rows = [np.ascontiguousarray(x[idx]) for x in [w0] + abc0 + [r0, s0]]
    exp = {j: key.expected(w0[idx[j]], abc0[0][idx[j]], abc0[1][idx[j]], abc0[2][idx[j]], r0[idx[j]], s0[idx[j]])[0]
           for j in sorted({0, k - 1})}
    return rows, exp, ncons


def in_parallel(fns):
    errs = []

    def run(f):
        try:
            f()
        except BaseException as e:  # noqa: BLE001 - re-raised below
            errs.append(e)
    th = [threading.Thread(target=run, args=(f,)) for f in fns]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03g_group_prove_batch.jsonl"))
    ap.add_argument("--logs", default="18,20,22")
    ap.add_argument("--ns", default="1,2,4,8")
    ap.add_argument("--per-device", default="8,32", help="k = m * n for each m")
    ap.add_argument("--replicate-logs", default="20,22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pool", type=int, default=4)
    ap.add_argument("--max-input-gb", type=float, default=24.0)
    a = ap.parse_args()
    import torch
    n_gpus = torch.cuda.device_count()
    rs = np.random.Generator(np.random.PCG64(20261024))
    lines = [{"gpus": gpu_info(), "device_count": n_gpus}]
    print(json.dumps(lines[0]), flush=True)

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)
        with open(a.out, "w") as f:
            for x in lines:
                f.write(json.dumps(x) + "\n")
    ns = [int(x) for x in a.ns.split(",") if x]
    per_dev = [int(x) for x in a.per_device.split(",") if x]
    with lib.Context(0) as ctx:
        for L in [int(x) for x in a.logs.split(",") if x]:
            key = KnownDlogKey(ctx, L, seed=3000 + L)
            try:
                for n in ns:
                    for m in per_dev:
                        k = m * n
                        base = {"kind": "group_prove", "log2n": L, "n_devices": n, "k": k}
                        row_bytes = (key.N + 3 * (key.N - 1)) * 32
                        if n > n_gpus:
                            emit(dict(base, status=f"not measured: {n} devices, the machine has {n_gpus}"))
                            continue
                        if k * row_bytes > a.max_input_gb * 1e9:
                            emit(dict(base, status=f"not measured: {k * row_bytes / 1e9:.1f} GB of inputs > "
                                                   f"--max-input-gb {a.max_input_gb}"))
                            continue
                        rows, exp, ncons = make_inputs(key, k, a.pool, rs)
                        wires, A, B, Cc, r, s = rows
                        with lib.Group(list(range(n))) as g:
                            gpk = g.pk_replicate(key.handle)
                            try:
                                for pinned in (True, False):
                                    if pinned:
                                        for x in (wires, A, B, Cc):
                                            lib.host_register(x)
                                    try:
                                        got = g.prove_batch(gpk, wires, A, B, Cc, r, s)
                                        one = ctx.prove_batch(key.handle, wires, A, B, Cc, r, s)
                                        for j, e in exp.items():
                                            assert check_proof(got[j], e) == [], f"group proof {j}: closed form"
                                            assert check_proof(one[j], e) == [], f"one-ctx proof {j}: closed form"
                                        t_group = median_ms(lambda: g.prove_batch(gpk, wires, A, B, Cc, r, s), a.reps)
                                        phases = [g.ctx(i).last_timings() for i in range(n)]
                                        t_one = median_ms(lambda: ctx.prove_batch(key.handle, wires, A, B, Cc, r, s),
                                                          a.reps)
                                    finally:
                                        if pinned:
                                            for x in (wires, A, B, Cc):
                                                lib.host_unregister(x)
                                    members = []
                                    for i, (lo, hi) in enumerate(ranges(k, n)):
                                        ph = phases[i]
                                        members.append({
                                            "device": i, "proofs": hi - lo, "phases_ms": [round(x, 3) for x in ph],
                                            "wire_upload_GBps": round((hi - lo) * key.N * 32 / (ph[0] * 1e6), 2)
                                            if ph and ph[0] > 0 else None,
                                            "rows_over_call_GBps": round((hi - lo) * row_bytes / (t_group * 1e6), 2)})
                                    emit(dict(base, host="pinned" if pinned else "pageable", reps=a.reps,
                                              group_ms=round(t_group, 3), group_ms_per_proof=round(t_group / k, 3),
                                              group_proofs_per_s=round(k / t_group * 1e3, 1),
                                              one_ctx_ms=round(t_one, 3), one_ctx_ms_per_proof=round(t_one / k, 3),
                                              one_ctx_proofs_per_s=round(k / t_one * 1e3, 1),
                                              speedup_over_one_ctx=round(t_one / t_group, 3), members=members))
                            finally:
                                g.pk_free(gpk)
                        del rows, wires, A, B, Cc
            finally:
                key.free()
        for L in [int(x) for x in a.replicate_logs.split(",") if x]:
            key = KnownDlogKey(ctx, L, seed=4000 + L, precompute=True)
            try:
                host = {nm: key.vec[nm].download() for nm in ("a", "b", "k", "z", "b2")}
                p = key.points
                vec_bytes = sum(v.n * (ctx.msm_plan(v)[1] if v.window() else 1) * (64 if nm != "b2" else 128)
                                for nm, v in key.vec.items())
                for n in ns:
                    if n < 2:
                        continue
                    base = {"kind": "replicate", "log2n": L, "n_devices": n}
                    if n > n_gpus:
                        emit(dict(base, status=f"not measured: {n} devices, the machine has {n_gpus}"))
                        continue
                    (wires, A, B, Cc, r, s), exps, _ = make_inputs(key, n, 1, rs)
                    exp = exps[0]
                    with lib.Group(list(range(n))) as g:
                        ts = []
                        for _ in range(a.reps):
                            t0 = time.perf_counter()
                            gpk = g.pk_replicate(key.handle)
                            ts.append((time.perf_counter() - t0) * 1e3)
                            got = g.prove_batch(gpk, wires, A, B, Cc, r, s)
                            for j in range(n):
                                assert check_proof(got[j], exp) == [], f"replica proof {j}: closed form"
                            g.pk_free(gpk)
                        t_rep = statistics.median(ts)
                        ctxs = [g.ctx(i) for i in range(n)]
                        tu = []
                        for _ in range(a.reps):
                            made = [None] * n

                            def up(i):
                                made[i] = ctxs[i].pk_upload(L, key.N, host["a"], host["b"], host["k"], host["z"],
                                                            host["b2"], p["alpha"], p["beta"], p["delta"], p["beta2"],
                                                            p["delta2"], key.zeros, key.zeros, key.k_skip,
                                                            precompute=True)
                            t0 = time.perf_counter()
                            in_parallel([lambda i=i: up(i) for i in range(n)])
                            tu.append((time.perf_counter() - t0) * 1e3)
                            for h in made:
                                ctx.pk_free(h)
                        t_up = statistics.median(tu)
                    emit(dict(base, reps=a.reps, windows=[key.vec[nm].window() for nm in ("a", "b", "k", "z", "b2")],
                              replicate_ms=round(t_rep, 3), bytes_copied=vec_bytes * (n - 1),
                              copy_GBps=round(vec_bytes * (n - 1) / (t_rep * 1e6), 2),
                              upload_precompute_every_device_ms=round(t_up, 3),
                              upload_over_replicate=round(t_up / t_rep, 3)))
            finally:
                key.free()


if __name__ == "__main__":
    main()
