"""bench.py — BN254 G1 MSM throughput on B200 (BASELINE.json configs[1]), plus the other parts of the metric
("Groth16 prove ms; BN254 MSM Mpts/s, NTT GB/s") as extras of the same JSON line.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      # CPU arm: the C port of gnark's MultiExp on host cores, SAME size
  python bench.py --workload prove ...      # second metric: synthetic WHIR-verifier-shaped Groth16 prove
  python bench.py --dump-outputs DIR ...    # also writes the last timed step's result as DIR/<name>.npy

A "step" is one multi-scalar multiplication of 2^logn points (default 2^24, uniform scalars), bases resident in
HBM.  With N ranks the point range is sharded N ways (strong scaling), each rank runs a local Pippenger, and one
all_gather of N partial points + N-1 host additions produce the result on every rank.
  value         scalars already resident in HBM (b200g16_msm_g1_dev)
  e2e           scalars in pinned HOST memory through b200g16_msm_g1 (H2D inside the timed region)
  e2e_pageable  the same call on ordinary (pageable) host memory — what a Go slice is without b200g16_host_register
Every timed configuration is gated first: the result (the COMBINED point at N > 1; every MSM output, h and the proof
for the prove) must equal the oracle's closed form (oracle/synth.py, C restatement) or the run refuses to time it.
"""
import argparse
import glob
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20261018
MAD_PER_MODMUL = 136          # 2*8*8 + 8 32x32 multiply-adds per Montgomery product (SURVEY §8d)
MODMUL_PER_MADD = 10          # XYZZ mixed add: 8M + 2S
# executed by k_accumulate per mixed add: 6 products, 2 dedicated squares (sqr_ptx: 108), and y3 = R(Q-X3) - Y*PPP
# as one fused two-term product (dot2_ptx: 200 instead of 2 x 136)
EXECUTED_MAD_PER_MADD = 6 * 136 + 2 * 108 + 200
R_MOD = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001


def rand_fr(rs, n):
    a = rs.integers(0, 1 << 62, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 60) - 1)        # < 2^252 < r: every row is a valid Montgomery residue
    return a


def dump_outputs(dirname, points):
    """--dump-outputs: each group element (uint64 limbs as the C-ABI returns them: affine x then y, Montgomery form)
    as DIR/<name>.npy, float64 rows of eight little-endian 32-bit words (exact in float64), one row per base-field
    coordinate, so that two builds can be compared bit for bit."""
    os.makedirs(dirname, exist_ok=True)
    for name, p in points.items():
        words = np.ascontiguousarray(p, dtype="<u8").view("<u4").reshape(-1, 8)
        np.save(os.path.join(dirname, f"{name}.npy"), words.astype(np.float64))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def load_ncu_traffic(kernel, logn, table):
    """DRAM bytes per launch of the dominant kernel from the newest ncu capture under profiles/ (a JSON artefact
    written next to the capture, stamped with the commit it was taken at); None when there is none for this shape."""
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_traffic*.json"))):
        try:
            d = json.load(open(path))
        except Exception:
            continue
        if d.get("kernel") == kernel and d.get("log2n") == logn and bool(d.get("window_table")) == bool(table):
            best = dict(d, file=os.path.relpath(path, ROOT))
    return best


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if v > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    """All the host threads this process may use.  torchrun exports OMP_NUM_THREADS=1 to every rank, which
    would silently run the CPU arm on one core — the thread count is passed to the C port explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_msm_sample(log_sample, steps, warmup):
    from oracle import cport
    nt = host_threads()
    rs = np.random.Generator(np.random.PCG64(SEED))
    n = 1 << log_sample
    k0, d = rand_fr(rs, 1), rand_fr(rs, 1)
    pts = cport.g1_progression(k0, d, n)
    sc = rand_fr(rs, n)
    for _ in range(warmup):
        cport.msm_g1(pts[: max(1, n >> 4)], sc[: max(1, n >> 4)], nt)
    times = []
    out = None
    for _ in range(steps):
        t0 = time.perf_counter()
        out = cport.msm_g1(pts, sc, nt)
        times.append(time.perf_counter() - t0)
    ok = bool(np.array_equal(out, cport.g1_gen_mul(cport.fr_dot_progression(sc, k0, d))))
    return n, times, nt, ok


def cpu_prove_sample(L, steps):
    """The C restatement of gnark's Prove after Solve (oracle_groth16_prove) on a synthetic key of 2^L constraints
    whose points are an arithmetic progression of known discrete logs (made on the CPU; no GPU involved)."""
    from oracle import cport, synth
    nt = host_threads()
    rs = np.random.Generator(np.random.PCG64(SEED + 5))
    N = 1 << L
    pts = [cport.g1_progression(rand_fr(rs, 1), rand_fr(rs, 1), n) for n in (N, N, N - 1, N - 1)]
    gk = rand_fr(rs, 2)
    g2 = np.stack([cport.g2_gen_mul(gk[0]), cport.g2_gen_mul(gk[1])])
    b2 = np.tile(g2, ((N + 1) // 2, 1))[:N]            # the G2 work does not depend on the points being distinct
    small1 = pts[0][:3].copy()
    wires = synth.whir_mix(rs, N)
    a, b, c = rand_fr(rs, N), rand_fr(rs, N), rand_fr(rs, N)
    r, s = rand_fr(rs, 1)[0], rand_fr(rs, 1)[0]
    k_skip = np.zeros(N, np.uint8)
    k_skip[0] = 1
    zeros = np.zeros(N, np.uint8)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cport.groth16_prove(L, pts[0], pts[1], pts[2], pts[3], b2, small1[0], small1[1], small1[2], g2[0], g2[1],
                            zeros, zeros, k_skip, wires, a, b, c, r, s, nthreads=nt)
        times.append((time.perf_counter() - t0) * 1e3)
    return times, nt


def run_reference(args, rank):
    if rank != 0:
        return
    if args.workload == "prove":
        L = min(args.prove_logns[0], args.cpu_prove_logn)
        times, cores = cpu_prove_sample(L, max(1, args.steps))
        ms = sum(times) / len(times)
        sample = (f"C restatement of gnark's groth16 Prove after Solve (oracle/c/oracle_groth16.c: computeH + 4 G1 + 1 G2 "
                  f"MultiExp + assembly; gnark itself cannot be built here: no Go toolchain), 2^{L} constraints, {cores} OpenMP threads")
        print(json.dumps({
            "impl": "reference", "metric": "WHIR-verifier-shaped Groth16 prove latency", "value": round(ms, 2), "unit": "ms",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 2),
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": f"synthetic Groth16 prove, 2^{L} constraints (bounded sample of the 2^{args.prove_logns[0]} workload)"
                                   if L != args.prove_logns[0] else f"synthetic Groth16 prove, 2^{L} constraints",
                       "same_size_as_gpu_arm": L == args.prove_logns[0]},
            "cpu_baseline": {"value": round(ms, 2), "unit": "ms", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": round(ms, 2), "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    log_sample = args.logn if args.cpu_logn is None else min(args.logn, args.cpu_logn)
    n, times, cores, ok = cpu_msm_sample(log_sample, args.steps, min(args.warmup, 1))
    ms = 1e3 * sum(times) / len(times)
    val = n / (ms * 1e3)
    sample = (f"C port of gnark-crypto MultiExp (oracle/c/oracle.c; gnark itself cannot be built here: no Go "
              f"toolchain), G1 MSM of 2^{log_sample} points per step, uniform scalars, {cores} OpenMP threads")
    wl = (f"G1 MSM 2^{args.logn} points (BASELINE.json configs[1]), uniform scalars" if log_sample == args.logn else
          f"G1 MSM, bounded sample 2^{log_sample} points of the 2^{args.logn}-point workload")
    print(json.dumps({
        "impl": "reference", "metric": "BN254 G1 MSM throughput", "value": round(val, 4), "unit": "Mpts/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": wl, "points": n, "same_size_as_gpu_arm": log_sample == args.logn, "result_checked": ok},
        "cpu_baseline": {"value": round(val, 4), "unit": "Mpts/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(val, 4), "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------------------------- helpers
class Dist:
    """torch.distributed plumbing shared by the workloads (world of one works without a process group)."""

    def __init__(self, local_rank, world):
        import torch
        self.torch, self.world = torch, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            import datetime

            import torch.distributed as dist
            self.dist = dist
            # a rank that dies must not leave the others waiting in a collective for NCCL's default half hour
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=600))

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def reduce(self, x, op="max"):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather_fr(self, fr_mont):
        """all_gather of one Fr element per rank (uint64[4]) -> list of python ints (canonical values)."""
        from oracle import bn254 as bn
        a = np.ascontiguousarray(fr_mont, dtype=np.uint64).reshape(1, 4)
        if self.world == 1:
            return bn.fr_from_mont_array(a)
        t = self.torch.from_numpy(a.view(np.int64).copy()).to(self.dev)
        outs = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(outs, t)
        return [bn.fr_from_mont_array(o.cpu().numpy().view(np.uint64))[0] for o in outs]

    def finish(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def to_dev(torch, dev, a, pin=False):
    t = torch.from_numpy(np.ascontiguousarray(a).view(np.int64))
    return t.pin_memory() if pin else t.to(dev)


# --------------------------------------------------------------------------------------------- prove benchmark
def prove_bench(ctx, D, rank, L, args, steps, warmup, want_e2e, want_cpu, dump_dir=None):
    """Synthetic WHIR-verifier-shaped Groth16 prove of 2^L constraints and as many wires on a known-discrete-log key
    (oracle/synth.py) sharded by point range over the ranks.  Inside the timed region, per step: the BSB22
    Pedersen commitment MSM (gnark runs it inside Solve), the prove (5 MSMs + computeH), the Pedersen
    proof-of-knowledge MSM.  Gate: every MSM output, h, Ar / Bs / Krs, commitment and PoK equal the
    closed forms computed by the C restatement on rank 0.  With dump_dir, rank 0 writes the proof, commitment
    and PoK of the last timed step there."""
    import torch

    from gnark_whir_b200 import lib, sharded
    from oracle import bn254 as bn
    from oracle import cport, synth
    world, dev = D.world, D.dev
    N = 1 << L
    lens = {"a": N, "b": N, "k": N - 1, "z": N - 1}
    spans = {k: sharded.shard_range(v, rank, world) for k, v in lens.items()} if world > 1 else None
    t0 = time.perf_counter()
    key = synth.KnownDlogKey(ctx, L, seed=SEED + L, precompute=args.table, lo_hi=spans)
    setup_ms = (time.perf_counter() - t0) * 1e3
    rs = np.random.Generator(np.random.PCG64(SEED + 17 * L))          # identical on every rank
    wires = synth.whir_mix(rs, N)
    a, b, c = rand_fr(rs, N), rand_fr(rs, N), rand_fr(rs, N)
    rr, ss = rand_fr(rs, 1)[0], rand_fr(rs, 1)[0]
    # BSB22: the committed wires (every lookup query / result: "large for this circuit", SURVEY §8a P5) — N/8 here
    nc = N // 8
    c_lo, c_hi = sharded.shard_range(nc, rank, world)
    kc = rand_fr(rs, 2 * nc).reshape(2, nc, 4)                        # dlogs of Basis and BasisExpSigma
    ped = [ctx.fixed_base_mul(synth.G1, kc[j][c_lo:c_hi], group=1, resident=True) for j in range(2)]
    committed = wires[1:1 + nc]
    d_w = to_dev(torch, dev, wires)
    d_abc = [to_dev(torch, dev, v) for v in (a, b, c)]
    d_com = to_dev(torch, dev, committed[c_lo:c_hi])
    distributed_h = world > 1 and not args.replicated_h
    # 2 / 4 / 8 ranks: computeH split over ALL ranks (cross-GPU butterfly levels over CUDA-IPC peer memory, every rank
    # keeps only its slices of a, b, c and ends up with its slice of h = its Z shard); other rank counts: a, b, c
    # transformed on three ranks + NCCL broadcasts
    dh = sharded.DistributedH(ctx, L) if (distributed_h and world in (2, 4, 8)) else None
    if dh is not None:
        M = N // world
        abc_slices = [t[rank * M:(rank + 1) * M].contiguous() for t in d_abc]

    xch1, xch48 = sharded.PointExchange(8, device=dev), sharded.PointExchange(48, device=dev)

    def gather_sum(points, group=1):
        return xch1.combine(points, group) if world > 1 else points

    def step():
        if dh is None:
            aa, bb, cc = (t.clone() for t in d_abc)                                             # computeH works in place
            torch.cuda.synchronize()
        com = gather_sum(ctx.msm(ped[0], d_com.data_ptr(), n=c_hi - c_lo))                     # Commit (inside Solve)
        # ProveKnowledge: enqueued ahead of the prove (nothing in between needs its result), collected after it
        tk = ctx.msm_begin(ped[1], d_com.data_ptr(), n=c_hi - c_lo)
        if dh is not None:
            dh.load(*abc_slices)
            part = ctx.prove_h_dev(key.handle, d_w.data_ptr(), dh.run(), rr, ss)
            sums = sharded.sum_partials(list(xch48.gather(sharded.pack_partials(part))))
            proof = ctx.prove_finish(key.handle, sums["msm_a"], sums["msm_b1"], sums["msm_k"], sums["msm_z"], sums["msm_b2"], rr, ss)
            pok = gather_sum(ctx.msm_end(tk))
            return proof, com, pok, None
        if world == 1:
            proof = ctx.prove_dev(key.handle, d_w.data_ptr(), aa.data_ptr(), bb.data_ptr(), cc.data_ptr(), rr, ss)
        else:
            if distributed_h:
                sharded.compute_h_distributed(ctx, aa, bb, cc, L)
                part = ctx.prove_h_dev(key.handle, d_w.data_ptr(), aa.data_ptr(), rr, ss)
            else:
                part = ctx.prove_dev(key.handle, d_w.data_ptr(), aa.data_ptr(), bb.data_ptr(), cc.data_ptr(), rr, ss)
            sums = sharded.sum_partials(list(xch48.gather(sharded.pack_partials(part))))
            proof = ctx.prove_finish(key.handle, sums["msm_a"], sums["msm_b1"], sums["msm_k"], sums["msm_z"], sums["msm_b2"], rr, ss)
        pok = gather_sum(ctx.msm_end(tk))
        return proof, com, pok, aa

    # ---- gate
    proof, com, pok, h_dev = step()
    bad = []
    if rank == 0:
        exp, h_exp = key.expected(wires, a, b, c, rr, ss, host_threads())
        bad = synth.check_proof(proof, exp)
        if h_dev is not None and not np.array_equal(h_dev.cpu().numpy().view(np.uint64), h_exp):
            bad.append("h")        # (split computeH: every slice of h is covered by the combined msm_z check)
        for name, got, k in (("commitment", com, kc[0]), ("pok", pok, kc[1])):
            if not np.array_equal(got, cport.g1_gen_mul(cport.fr_dot(k, committed, host_threads()))):
                bad.append(name)
    if D.reduce(float(len(bad)), "max") > 0:
        raise SystemExit(f"bench: prove 2^{L} differs from the oracle's closed form in {bad} — refusing to time it")
    for _ in range(max(0, warmup - 1)):
        step()
    D.sync_all()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        last = step()[:3]          # not h: the next step's clone must be able to reuse its buffer
    e1.record()
    D.sync_all()
    ms = D.reduce(e0.elapsed_time(e1) / steps, "max")
    launches = ctx.launch_count() - l0
    if dump_dir and rank == 0:
        proof, com, pok = last
        dump_outputs(dump_dir, dict(proof, commitment=com, pok=pok))
    out = {"log2_constraints": L, "wires": N, "committed_wires": nc, "ms": round(ms, 3), "n_gpus": world,
           "window_tables": bool(args.table), "witness_mix": "40% 0/1, 30% bytes, 30% uniform (SURVEY §8d config 1)",
           "timed_region": "Pedersen Commit MSM + Pedersen PoK MSM (b200g16_msm_g1_begin_dev, collected after the prove) + b200g16_prove_dev (5 MSMs, computeH, host assembly); "
                           "inputs resident in HBM",
           "result_checked_vs_oracle": True, "gpu_launches_per_step": launches // max(1, steps),
           "key_setup_ms_once": round(setup_ms, 1)}
    if world > 1:
        out["parallelism"] = (f"pk point-range shards x{world}; computeH " +
                              ("replicated" if args.replicated_h else
                               (f"split over all {world} ranks (cross-GPU NTT levels over CUDA-IPC peer memory, 4 barriers)" if dh is not None
                                else "spread over 3 ranks (a, b, c) + 3 NCCL broadcasts")) +
                              "; all_gather of the partial points")
    if want_e2e and world == 1:
        # through b200g16_prove with HOST buffers (witness + a, b, c = 128 N bytes H2D inside), pinned and pageable
        def e2e(bufs, cbuf):
            def one():
                cm = ctx.msm(ped[0], cbuf)
                tk = ctx.msm_begin(ped[1], cbuf)
                res, _ = ctx.prove(key.handle, bufs[0], bufs[1], bufs[2], bufs[3], rr, ss)
                pk_ = ctx.msm_end(tk)
                return res, cm, pk_
            res, cm, pk_ = one()
            if not (np.array_equal(res["krs"], proof["krs"]) and np.array_equal(cm, com) and np.array_equal(pk_, pok)):
                raise SystemExit("bench: host-path and device-path proofs differ")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                one()
            return (time.perf_counter() - t0) * 1e3 / steps
        pinned = [to_dev(torch, dev, v, pin=True).numpy().view(np.uint64) for v in (wires, a, b, c, committed)]
        out["e2e"] = {"value": round(e2e(pinned[:4], pinned[4]), 3), "unit": "ms",
                      "h2d_bytes_per_step": int((4 * N + 2 * nc) * 32), "d2h_bytes_per_step": int(5 * 256 + 64 + 2 * 128),
                      "host_memory": "pinned"}
        out["e2e_pageable"] = {"value": round(e2e([wires, a, b, c], np.ascontiguousarray(committed)), 3), "unit": "ms",
                               "host_memory": "pageable (ordinary numpy arrays = unregistered Go slices)"}
    ph = ctx.last_timings()
    out["last_msm_phases_ms"] = [round(x, 3) for x in ph]
    if want_cpu and rank == 0:
        Lc = min(L, args.cpu_prove_logn)
        times, cores = cpu_prove_sample(Lc, 1)
        out["cpu_baseline"] = {"value": round(min(times), 1), "unit": "ms", "cores": cores, "kind": "port",
                               "sample": f"oracle_groth16_prove (C restatement of gnark's Prove after Solve), 2^{Lc} constraints, "
                                         f"{cores} OpenMP threads, 1 run" + ("" if Lc == L else f" (bounded sample of the 2^{L} prove)")}
    if dh is not None:
        dh.close()
    key.free()
    for v in ped:
        v.free()
    del d_w, d_abc, d_com
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------- GPU arm
def run_b200(args, rank, local_rank, world):
    import torch

    from gnark_whir_b200 import lib, sharded
    from oracle import bn254 as bn
    from oracle import cport          # the checker for the parity gates; never on the timed path
    from oracle import synth

    D = Dist(local_rank, world)
    dev = D.dev
    ctx = lib.Context(local_rank)
    peaks, peaks_kind = load_peaks()
    n = 1 << args.logn
    lo, hi = sharded.shard_range(n, rank, world)
    m = hi - lo
    rs = np.random.Generator(np.random.PCG64(SEED + 1000 * rank))

    # ---- inputs: bases = k_i * G generated on the GPU (known discrete logs), scalars uniform
    ks = rand_fr(rs, m)
    bases = ctx.fixed_base_mul(synth.G1, ks, group=1, resident=True)
    table_ms = None
    if args.table:
        # window table over the resident bases, built once (like the pk upload): W rows of m points
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bases.precompute(0)
        table_ms = (time.perf_counter() - t0) * 1e3
    win_c, win_W = ctx.msm_plan(bases, m)
    sc_host_t = torch.empty((m, 4), dtype=torch.int64).pin_memory()
    sc_host = sc_host_t.numpy().view(np.uint64)
    sc_host[:] = rand_fr(rs, m)
    sc_pageable = sc_host.copy()
    sc_dev = sc_host_t.to(dev)

    xch = sharded.PointExchange(8, device=dev)         # one G1 point per rank; buffers allocated once

    def step_resident():
        return xch.combine(ctx.msm(bases, sc_dev.data_ptr(), n=m), 1)

    def step_e2e():
        return xch.combine(ctx.msm(bases, sc_host), 1)     # H2D of this step's scalars happens inside

    def step_pageable():
        return xch.combine(ctx.msm(bases, sc_pageable), 1)

    sampler = ClockSampler(local_rank)     # nvidia-smi needs a moment to start: sample from the gate onwards
    if rank == 0:
        sampler.start()

    # ---- parity gate before timing: the COMBINED point (all ranks' shards) == closed form
    # [sum over ranks of <k, s>] G: per-rank dot products by the C oracle, gathered, added mod r, one scalar mul
    dots = D.gather_fr(cport.fr_dot(ks, sc_host, host_threads() if world == 1 else max(1, host_threads() // world)))
    expect = cport.g1_gen_mul(bn.fr_to_mont_array([sum(dots) % R_MOD]))
    for name, fn in (("resident", step_resident), ("host-scalar", step_e2e)):
        if not np.array_equal(fn(), expect):
            raise SystemExit(f"bench: combined GPU MSM result ({name} path) differs from the oracle's closed form — refusing to time it")
    checked = True

    # integer-pipe peak, measured live (burst): modmul/s with 4 independent chains, 8 CTAs/SM; and the raw
    # IMAD.WIDE.X carry-chain rate the multiplier is made of
    probe_rate, _ = ctx.modmul_probe(8, 4, 2000)
    tmad_peak = probe_rate * MAD_PER_MODMUL / 1e12
    raw_rate, _ = ctx.pipe_probe(2, 8, 2000)
    dfma_rate, _ = ctx.pipe_probe(6, 8, 2000)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        D.sync_all()
        l0 = ctx.launch_count()
        phases = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = None
        for _ in range(steps):
            res = fn()
            phases.append(ctx.last_timings())
        e1.record()
        D.sync_all()
        ms = D.reduce(e0.elapsed_time(e1) / steps, "max")
        return ms, phases, ctx.launch_count() - l0, res

    ms, phases, launches, res_a = timed(step_resident, args.steps, args.warmup)
    ms_e2e, _, _, res_b = timed(step_e2e, args.steps, max(1, args.warmup // 2))
    clocks = sampler.stop() if rank == 0 else None
    ms_page, _, _, res_c = timed(step_pageable, max(1, args.steps // 2), 1)
    if not (np.array_equal(res_a, expect) and np.array_equal(res_b, expect) and np.array_equal(res_c, expect)):
        raise SystemExit("bench: a timed step's result differs from the oracle's closed form")
    launches_total = int(D.reduce(launches, "sum"))

    # ---- dominant kernel: k_accumulate (phase index 2 of [digits, sort, accumulate, merge, reduce])
    acc_ms = D.reduce(statistics.mean(p[2] for p in phases if len(p) >= 5), "max")
    msm_dev_ms = D.reduce(statistics.mean(sum(p) for p in phases if len(p) >= 5), "max")
    phase_avg = [round(statistics.mean(p[i] for p in phases if len(p) >= 5), 4) for i in range(5)]
    algo_bytes = 96.0 * m                     # SURVEY §8d: 64 B point + 32 B scalar per point
    # integer roofline of the dominant kernel: mixed adds = W digits per point, 10 products of 136 MADs each
    mads = float(win_W) * m * MODMUL_PER_MADD * MAD_PER_MODMUL
    ach = mads / (acc_ms * 1e-3) / 1e12
    traffic_rec = load_ncu_traffic("k_accumulate<Fp>", args.logn, args.table) if world == 1 else None
    traffic = args.ncu_traffic if args.ncu_traffic is not None else (traffic_rec or {}).get("dram_bytes_per_launch")
    gather_bytes = float(win_W) * m * 68
    roofline = {"bound": "integer", "kernel": "k_accumulate<Fp>", "achieved": round(ach, 3), "peak": round(tmad_peak, 3),
                "unit": "TMAD/s", "frac": round(ach / tmad_peak, 4), "traffic": traffic,
                "traffic_source": ((traffic_rec or {}).get("file") if args.ncu_traffic is None else "--ncu-traffic"),
                "traffic_commit": (traffic_rec or {}).get("commit"),
                "traffic_note": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum). SURVEY's algorithmic "
                                f"input is 96 B/point = {int(algo_bytes)} B per launch; the window table turns every one of the "
                                f"{win_W} additions per point into a 64 B gather + 4 B entry = {int(gather_bytes)} B per launch "
                                f"({gather_bytes / algo_bytes:.1f}x the algorithmic bytes — the table's price; HBM is not the bound)",
                "peak_source": "b200g16_modmul_probe measured in this run (burst; 136 IMAD.WIDE-class multiply-adds per "
                               "Montgomery product); MEASURED_PEAKS.json has no integer-pipe figure",
                "peak_raw_imad_wide": round(raw_rate / 1e12, 3),
                "peak_raw_imad_wide_note": "b200g16_pipe_probe mode 2 (mad.lo.cc/madc.hi.cc carry chains = IMAD.WIDE.X), T instr/s",
                "peak_raw_dfma": round(dfma_rate / 1e12, 3),
                "algorithmic_mads_per_launch": int(mads), "window_bits": win_c, "adds_per_point": win_W,
                "frac_executed": round(ach * EXECUTED_MAD_PER_MADD / (MODMUL_PER_MADD * MAD_PER_MODMUL) / tmad_peak, 4),
                "accumulate_ms": round(acc_ms, 4), "msm_device_ms": round(msm_dev_ms, 4),
                "phases_ms[digits,sort,accumulate,merge,reduce]": phase_avg,
                "note": "achieved counts SURVEY's algorithmic 1360 multiply-adds per mixed add; the kernel executes 1232 "
                        "(dedicated Montgomery square, fused two-term product), frac_executed is the pipe's own "
                        "utilisation.  north_star: MSM is judged against the integer pipe (no dense contraction, 96 B/point "
                        "of HBM traffic against ~20k multiply-adds/point); the HBM view is roofline_hbm"}
    roofline_hbm = {"bound": "hbm", "kernel": "k_accumulate<Fp>", "achieved": round(algo_bytes / (acc_ms * 1e6), 2),
                    "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": round(algo_bytes / (acc_ms * 1e6) / peaks["hbm_gbs"], 5),
                    "peak_source": f"MEASURED_PEAKS.json ({peaks_kind})"}
    out = {
        "metric": "BN254 G1 MSM throughput", "value": round(n / (ms * 1e3), 3), "unit": "Mpts/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"G1 MSM 2^{args.logn} points (BASELINE.json configs[1]), uniform scalars, bases resident",
                   "window_table": ({"c": win_c, "rows": win_W, "build_ms_once": round(table_ms, 1),
                                     "bytes_per_gpu": int(win_W * m * 64)} if args.table else None),
                   "points": n, "points_per_gpu": m, "parallelism": f"point-range shards x{world} + all_gather of partial points",
                   "l2": "inputs (96 B/point, >= 190 MB per GPU) exceed the 126 MB L2; no flush needed",
                   "result_checked_vs_oracle": checked,
                   "gate": "combined point of all ranks == [sum_i s_i k_i] G (C oracle dot products + one scalar mul), "
                           "resident and host-scalar paths, before timing and on the last timed step"},
        "e2e": {"value": round(n / (ms_e2e * 1e3), 3), "unit": "Mpts/s", "ms_per_step": round(ms_e2e, 4),
                "h2d_bytes_per_step": int(32 * n), "d2h_bytes_per_step": int(world * ((1 if args.table else win_W) * 128 + 64)),
                "host_memory": "pinned"},
        "e2e_pageable": {"value": round(n / (ms_page * 1e3), 3), "unit": "Mpts/s", "ms_per_step": round(ms_page, 4),
                         "host_memory": "pageable numpy array (an unregistered Go slice); b200g16_host_register pins it in place"},
        "gpu_launches": launches_total,
        "clocks": clocks,
        "roofline": roofline,
        "roofline_hbm": roofline_hbm,
    }
    return ctx, D, out, dict(dev=dev, bases=bases, tmad_peak=tmad_peak, acc_ms=acc_ms, m=m, peaks=peaks, result=res_a)


def extras_single_gpu(ctx, D, st, args):
    """The other numbers of the metric, measured once at N=1 (not part of the timed MSM steps)."""
    import torch

    from gnark_whir_b200 import lib
    dev = st["dev"]
    ex = {}

    def t_ms(fn, reps=3):
        best = 1e30
        for _ in range(reps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best

    def rnd(shape):
        a = torch.randint(0, 1 << 62, shape, dtype=torch.int64, device=dev)
        a[..., 3] &= (1 << 60) - 1
        return a
    L = args.ntt_logn
    N = 1 << L
    a, b, c = rnd((N, 4)), rnd((N, 4)), rnd((N, 4))
    ctx.ntt_dev(a.data_ptr(), L, coset=True, decimation=lib.DIF)            # warm tables
    ms = t_ms(lambda: ctx.ntt_dev(a.data_ptr(), L, decimation=lib.DIF))
    ex["ntt"] = {"log2n": L, "ms": round(ms, 4), "GBs_algorithmic_64N": round(64 * N / ms / 1e6, 1),
                 "frac_hbm": round(64 * N / ms / 1e6 / st["peaks"]["hbm_gbs"], 4),
                 "TMAD_s": round((N / 2) * L * MAD_PER_MODMUL / ms / 1e9, 3),
                 "frac_integer": round((N / 2) * L * MAD_PER_MODMUL / ms / 1e9 / st["tmad_peak"], 4)}
    ms = t_ms(lambda: ctx.compute_h_dev(a.data_ptr(), b.data_ptr(), c.data_ptr(), L))
    ex["compute_h"] = {"log2n": L, "ms": round(ms, 4), "GBs_algorithmic_576N": round(576 * N / ms / 1e6, 1)}
    del a, b, c
    nk = 1 << 22
    stt = torch.randint(0, 1 << 62, (nk, 25), dtype=torch.int64, device=dev)
    ms = t_ms(lambda: ctx.keccak_f_batch_dev(stt.data_ptr(), nk))
    ex["keccak_f_batch"] = {"states": nk, "ms": round(ms, 4), "Gperm_s": round(nk / ms / 1e6, 3),
                            "GBs_400B": round(400 * nk / ms / 1e6, 1)}
    del stt
    torch.cuda.empty_cache()
    # the same MSM WITHOUT the window table (the table costs 13x the key's HBM): resident scalars, 3 steps
    try:
        from oracle import cport, synth
        rs2 = np.random.Generator(np.random.PCG64(SEED + 3))
        n2 = 1 << args.logn
        ks2 = rand_fr(rs2, n2)
        plain = ctx.fixed_base_mul(synth.G1, ks2, group=1, resident=True)
        sc2 = rand_fr(rs2, n2)
        d_sc2 = torch.from_numpy(sc2.view(np.int64)).to(dev)
        got = ctx.msm(plain, d_sc2.data_ptr(), n=n2)
        ok = bool(np.array_equal(got, cport.g1_gen_mul(cport.fr_dot(ks2, sc2, host_threads()))))
        ms = t_ms(lambda: ctx.msm(plain, d_sc2.data_ptr(), n=n2))
        c2, w2 = ctx.msm_plan(plain, n2)
        ex["msm_no_table"] = {"log2n": args.logn, "ms": round(ms, 3), "Mpts_s": round(n2 / ms / 1e3, 2), "window_bits": c2,
                              "adds_per_point": w2, "result_checked_vs_oracle": ok}
        plain.free()
        del d_sc2
        torch.cuda.empty_cache()
    except Exception as e:
        ex["msm_no_table"] = {"error": repr(e)}
    ex["groth16_prove"] = []
    for Lp in args.prove_logns:
        try:
            ex["groth16_prove"].append(prove_bench(ctx, D, 0, Lp, args, steps=3, warmup=2, want_e2e=True,
                                                   want_cpu=not args.no_cpu_baseline))
        except Exception as e:      # one size must not cost the others
            ex["groth16_prove"].append({"log2_constraints": Lp, "error": repr(e)})
    if not args.no_cpu_baseline:
        ex["cpu_port_same_box"] = cpu_extras()
    return ex


def cpu_extras():
    """The C port of the other kernels of the metric on this box's host cores (bounded samples; the
    checker, timed only as the reported CPU baseline)."""
    from oracle import cport
    rs = np.random.Generator(np.random.PCG64(SEED + 99))
    nt = host_threads()
    out = {"threads": nt, "kind": "port (oracle/c/oracle.c, OpenMP), not gnark"}

    def best_of(fn, reps=2):
        fn()
        return min(_timed(fn) for _ in range(reps))

    def _timed(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3
    a = rand_fr(rs, 1 << 20)
    out["ntt_2^20_ms"] = round(best_of(lambda: cport.ntt(a, nthreads=nt)), 2)
    a, b, c = rand_fr(rs, 1 << 18), rand_fr(rs, 1 << 18), rand_fr(rs, 1 << 18)
    out["compute_h_2^18_ms"] = round(best_of(lambda: cport.compute_h(a, b, c, 18, nthreads=nt)), 2)
    st = rs.integers(0, 1 << 63, size=(1 << 18, 25), dtype=np.uint64)
    ms = best_of(lambda: cport.keccak_f_batch(st, nthreads=nt))
    out["keccak_f_2^18_states_ms"] = round(ms, 2)
    out["keccak_Mperm_s"] = round((1 << 18) / ms / 1e3, 2)
    return out


def run_prove_workload(args, rank, local_rank, world):
    """--workload prove (BASELINE.json configs[0]/[4]): the prove benchmark as its own contract line."""
    from gnark_whir_b200 import lib
    D = Dist(local_rank, world)
    ctx = lib.Context(local_rank)
    L = args.prove_logns[0]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    res = prove_bench(ctx, D, rank, L, args, args.steps, args.warmup, want_e2e=True, want_cpu=not args.no_cpu_baseline,
                      dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        line = {"metric": "WHIR-verifier-shaped Groth16 prove latency", "value": res["ms"], "unit": "ms",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms"],
                "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": {"workload": f"synthetic Groth16 prove, 2^{L} constraints, {1 << L} wires, {res['committed_wires']} committed wires, "
                                       f"witness 40% 0/1 / 30% bytes / 30% uniform (SURVEY §8d config 1/5), inputs resident in HBM",
                           "window_tables": bool(args.table), "parallelism": res.get("parallelism", "1 GPU"),
                           "timed_region": res["timed_region"], "result_checked_vs_oracle": res["result_checked_vs_oracle"]},
                "e2e": res.get("e2e"), "e2e_pageable": res.get("e2e_pageable"),
                "gpu_launches": res["gpu_launches_per_step"] * args.steps * world, "clocks": clocks,
                "cpu_baseline": res.get("cpu_baseline")}
        print(json.dumps(line))
    ctx.close()
    D.finish()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--workload", default="msm", choices=["msm", "prove"],
                    help="msm = the headline (BASELINE configs[1]); prove = synthetic Groth16 prove (configs[0]/[4]), sharded at N>1")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--logn", type=int, default=24, help="log2 of the MSM size (whole job)")
    ap.add_argument("--cpu-logn", type=int, default=None,
                    help="log2 of the CPU arm's MSM (default: the GPU arm's size, so both arms run the same config)")
    ap.add_argument("--cpu-prove-logn", type=int, default=20, help="largest prove the C restatement is timed at")
    ap.add_argument("--ntt-logn", type=int, default=24)
    ap.add_argument("--prove-logn", default=None,
                    help="comma-separated log2 constraint counts (extras default 20,24; --workload prove default 20; "
                         "sharded extras at N>1 default 24)")
    ap.add_argument("--no-table", dest="table", action="store_false",
                    help="run the MSM without the window table over the resident bases (b200g16_bases_precompute)")
    ap.add_argument("--replicated-h", action="store_true",
                    help="prove, N>1: every rank runs the whole computeH instead of spreading it over 3 ranks")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu-traffic", type=float, default=None,
                    help="override: dram bytes per k_accumulate launch (default: newest profiles/*ncu_traffic*.json)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (the MSM "
                         "point, or the proof, commitment and PoK of --workload prove; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's results (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.prove_logn is None:
        args.prove_logns = [20] if args.workload == "prove" else ([20, 24] if world == 1 else [24])
    else:
        args.prove_logns = [int(x) for x in str(args.prove_logn).split(",") if x]
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    if args.workload == "prove":
        run_prove_workload(args, rank, local_rank, world)
        return
    ctx, D, out, st = run_b200(args, rank, local_rank, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"msm_g1": st["result"]})
    st["bases"].free()
    import torch
    torch.cuda.empty_cache()
    if not args.no_extras:
        try:
            if world == 1:
                out["extras"] = extras_single_gpu(ctx, D, st, args)
            else:           # SCALE run: 3 steps of the sharded prove (BASELINE configs[4]) next to the MSM line
                out["extras"] = {"prove_sharded": prove_bench(ctx, D, rank, args.prove_logns[0], args, steps=3, warmup=2,
                                                              want_e2e=False, want_cpu=False)}
        except Exception as e:          # extras must never cost the headline line
            out["extras"] = {"error": repr(e)}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            ls = args.logn if args.cpu_logn is None else min(args.logn, args.cpu_logn)
            n_s, times, cores, ok = cpu_msm_sample(ls, 1, 1)
            v = n_s / (min(times) * 1e6)
            out["cpu_baseline"] = {"value": round(v, 4), "unit": "Mpts/s", "cores": cores, "kind": "port",
                                   "sample": f"C port of gnark-crypto MultiExp (oracle/c/oracle.c), G1 MSM of 2^{ls} "
                                             f"points (the GPU arm's size), uniform scalars, {cores} OpenMP threads, 1 run; result_checked={ok}"}
        print(json.dumps(out))
    ctx.close()
    D.finish()


if __name__ == "__main__":
    main()
