"""Measure b200g16_keccak_duplex_batch_dev: throughput of the thread form at 2^20 sponges against k_keccak_f_batch,
and call latency of both kernel forms at small n (the evidence for DUPLEX_WARP_MAX in csrc/keccak.cu).

Scripts:
  transcript    absorb 32, squeeze 32, absorb 512, squeeze 64, absorb 8, squeeze 32 (a Fiat-Shamir transcript's shape)
  rate_aligned  absorb 1088 (eight full blocks), squeeze 136: every segment is a whole, 8-byte aligned rate block
Permutations per sponge are counted from the script by the Digest's position rules (count_permutes below) and
checked against oracle/keccak.py's Sponge.n_permutes.  Every timed configuration is gated first (untimed): a sample
of rows (outputs and final digests) must equal the oracle's.  Then the median of --reps calls, each timed with CUDA
events on torch's stream around the call (the call ends in a synchronise of the library's stream, so this is the
caller's view: op upload, kernel, synchronise).  The inputs are device buffers; the 2^20 working sets exceed the
126 MB L2, the latency ones fit it.  Rows: modes "tag" (every sponge starts from NewKeccak) and "continue" (from
the digests: adds the position check pass).

Writes one JSON line per configuration, after a first line with the card's name, power limit and max SM clock.
    python tools/duplex_bench.py --out profiles/r03c_keccak_duplex.jsonl
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from gnark_whir_b200 import lib  # noqa: E402
from oracle import keccak as ok  # noqa: E402

SCRIPTS = {
    "transcript": [("absorb", 32), ("squeeze", 32), ("absorb", 512), ("squeeze", 64), ("absorb", 8), ("squeeze", 32)],
    "rate_aligned": [("absorb", 1088), ("squeeze", 136)],
}
RATE = 136


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def count_permutes(script, absorb_pos=0, squeeze_pos=RATE):
    """Permutations the Digest issues for the script (keccakSponge.go:40-75), from the positions alone."""
    n = 0
    for kind, ln in script:
        for _ in range(ln):
            if kind == "absorb":
                if absorb_pos == RATE:
                    n, absorb_pos = n + 1, 0
                absorb_pos += 1
            else:
                if squeeze_pos == RATE:
                    n, absorb_pos, squeeze_pos = n + 1, 0, 0
                squeeze_pos += 1
        if kind == "absorb":
            squeeze_pos = RATE
    return n


def oracle_row(script, data):
    s = ok.Sponge()
    out, off = bytearray(), 0
    for kind, ln in script:
        if kind == "absorb":
            s.absorb(bytes(data[off:off + ln]))
            off += ln
        else:
            out += s.squeeze(ln)
    return bytes(out), s


def time_call(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03c_keccak_duplex.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--big", type=int, default=1 << 20)
    ap.add_argument("--small", default="1,16,64,256,1024,4096,8192,16384")
    ap.add_argument("--gate-rows", type=int, default=12)
    args = ap.parse_args()
    lines = [dict(gpu_info(), kind="device")]
    print(json.dumps(lines[0]), flush=True)
    rs = np.random.Generator(np.random.PCG64(20261020))

    def emit(rec):
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    with lib.Context(0) as ctx:
        def run_case(script_name, n, form, mode, reps):
            script = SCRIPTS[script_name]
            _, A, S = lib.duplex_script(script)
            perms = count_permutes(script)
            data = rs.integers(0, 256, size=(n, A), dtype=np.uint8)
            d_in = torch.from_numpy(data.reshape(-1)).cuda()
            d_out = torch.zeros(max(n * S, 1), dtype=torch.uint8, device="cuda")
            fresh = lib.keccak_digests(n).view(np.uint8).reshape(-1)
            d_dg = torch.from_numpy(fresh.copy()).cuda()
            if form is None:
                os.environ.pop("B200G16_DUPLEX_WARP", None)
            else:
                os.environ["B200G16_DUPLEX_WARP"] = form
            tag = b"" if mode == "tag" else None

            def call():
                ctx.keccak_duplex_batch_dev(d_dg.data_ptr(), n, script, d_in.data_ptr(), d_out.data_ptr(), tag=tag)
            # gate: outputs and final digests of sampled rows against the oracle (fresh digests in, one call)
            call()
            torch.cuda.synchronize()
            out = d_out[:n * S].cpu().numpy().reshape(n, S)
            dg = d_dg.cpu().numpy().view(lib.KECCAK_DIGEST)
            rows = sorted({0, n - 1} | set(rs.choice(n, size=min(args.gate_rows, n), replace=False).tolist()))
            for i in rows:
                want, s = oracle_row(script, data[i])
                assert bytes(out[i]) == want, (script_name, n, form, mode, i)
                assert bytes(dg[i]["state"].tobytes()) == bytes(s.state), (script_name, n, form, mode, i)
                assert s.n_permutes == perms
            for _ in range(3):
                call()                                  # warm-up
            med, mn = time_call(call, reps)
            os.environ.pop("B200G16_DUPLEX_WARP", None)
            rec = {"kind": "duplex", "script": script_name, "n": n, "form": {None: "auto", "0": "thread",
                                                                              "1": "warp"}[form],
                   "mode": mode, "perms_per_sponge": perms, "reps": reps, "median_ms": round(med, 4),
                   "min_ms": round(mn, 4), "gperm_s": round(n * perms / med * 1e-6, 3), "gated_rows": len(rows)}
            emit(rec)
            return rec

        # throughput: the thread form at 2^20 against the raw permutation on 2^20 states, same call
        st = torch.from_numpy(rs.integers(0, 1 << 63, size=(args.big, 25), dtype=np.uint64).view(np.int64)).cuda()
        ref = st[:4].cpu().numpy().view(np.uint64)
        ctx.keccak_f_batch_dev(st.data_ptr(), args.big)
        torch.cuda.synchronize()
        got = st[:4].cpu().numpy().view(np.uint64)
        for i in range(4):
            assert [int(v) for v in got[i]] == ok.keccak_f([int(v) for v in ref[i]])
        for _ in range(3):
            ctx.keccak_f_batch_dev(st.data_ptr(), args.big)
        med, mn = time_call(lambda: ctx.keccak_f_batch_dev(st.data_ptr(), args.big), args.reps)
        emit({"kind": "keccak_f_batch", "n": args.big, "reps": args.reps, "median_ms": round(med, 4),
              "min_ms": round(mn, 4), "gperm_s": round(args.big / med * 1e-6, 3), "gated_rows": 4})
        del st
        for name in ("rate_aligned", "transcript"):
            for mode in ("tag", "continue"):
                run_case(name, args.big, "0", mode, args.reps)
        torch.cuda.empty_cache()
        # latency: both forms forced, transcript script, device path
        for n in [int(x) for x in args.small.split(",")]:
            for form in ("0", "1"):
                run_case("transcript", n, form, "tag", args.reps)
            run_case("transcript", n, None, "continue", args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
