"""Batch proving against a loop of single proofs (tp_prove_batch vs tp_prove_inputs), one JSON line per case.

    python tools/prove_batch_bench.py [--cases 10:1,8,64;12:1,8,64;16:1,8,64;20:1,4,16] [--reps 3] [--out FILE]

Circuit: the mul_chain of BASELINE.json at 2^log_n rows; the batch cycles through `--distinct` witnesses (different
start values and blinders).  Per case, the batch and the loop alternate in one process after one warm-up call each:
  batch_ms, loop_ms               wall time of prove_batch / of K x prove_inputs (median of --reps; *_all: every rep)
  batch_per_proof_ms, loop_...    the same over K
  ratio                           batch_per_proof / loop_per_proof (< 1: the batch is faster)
  wave                            tp_ctx_get_stat("prove_batch_wave")
  batch_phases_ms, loop_phases_ms the library's phase timers (tp_prof_*) over one extra call of each
Every batch is checked byte for byte against the loop.  The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="10:1,8,64;12:1,8,64;16:1,8,64;20:1,4,16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from typlonk_b200 import field as F, synthetic
    from typlonk_b200.ffi import Context
    from oracle.pyoracle import rng

    info = gpu_info()
    ctx = Context(0)
    lines = []
    for case in args.cases.split(";"):
        log_n, counts = case.split(":")
        log_n = int(log_n)
        n = 1 << log_n
        circuit = synthetic.mul_chain_direct(ctx, log_n)
        h = circuit.handle
        wits = []
        for k in range(args.distinct):
            cols = synthetic.mul_chain_witness(n - 3, n, x0=3 + k, blind=rng.fr_rand_stream(700 + k, 9))
            wits.append([F.fr_vec_to_bytes(c) for c in cols])
        for K in [int(x) for x in counts.split(",")]:
            adv = [wits[k % len(wits)] for k in range(K)]
            pis = [b""] * K

            def batch():
                return h.prove_batch(adv, pis)

            def loop():
                return [h.prove_inputs(a, b"") for a in adv]
            fixed, status = batch()
            assert status == [0] * K and fixed == loop()    # warm-up, and the bytes
            bw, lw = [], []
            for _ in range(args.reps):
                t = time.perf_counter()
                batch()
                bw.append((time.perf_counter() - t) * 1e3)
                t = time.perf_counter()
                loop()
                lw.append((time.perf_counter() - t) * 1e3)
            wave = ctx.get_stat("prove_batch_wave")
            phases = {}
            for name, fn in (("batch", batch), ("loop", loop)):
                ctx.prof_enable(True)
                ctx.prof_reset()
                fn()
                phases[name] = {p: round(v[0], 3) for p, v in ctx.prof_get().items() if v[0]}
                ctx.prof_enable(False)
            b, lp = statistics.median(bw), statistics.median(lw)
            rec = dict(info, log_n=log_n, K=K, distinct_witnesses=len(wits), reps=args.reps, wave=int(wave),
                       batch_ms=round(b, 3), batch_ms_all=[round(x, 3) for x in bw],
                       loop_ms=round(lp, 3), loop_ms_all=[round(x, 3) for x in lw],
                       batch_per_proof_ms=round(b / K, 4), loop_per_proof_ms=round(lp / K, 4),
                       ratio=round(b / lp, 3), batch_phases_ms=phases["batch"], loop_phases_ms=phases["loop"])
            line = json.dumps(rec)
            print(line, flush=True)
            lines.append(line)
        h.destroy()
        circuit.srs.handle.destroy()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
