"""Proof format v2 against v1 on the device, one JSON line per size (written to --out, profiles/prove_v2_b200.jsonl
by default).

    python tools/prove_v2_bench.py [--logs 16,20,22] [--reps 5] [--out FILE]

Circuit: the mul_chain of BASELINE.json at 2^log_n rows, no public inputs.  tp_prove and tp_prove_v2 run alternately
in one process on the same witness (host columns), after one warm-up each; the line holds the median wall time of
each, their per-phase device timers (tp_prof, summed over the timed calls and divided by --reps), and tp_verify_v2
(host only) against tp_vk_verify per proof.  The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from verify_batch_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,20,22")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "prove_v2_b200.jsonl"))
    args = ap.parse_args()

    from typlonk_b200 import field as F, synthetic
    from typlonk_b200.ffi import PHASES, Context

    info = gpu_info()
    lines = []
    for log_n in [int(x) for x in args.logs.split(",")]:
        ctx = Context(0)
        n = 1 << log_n
        circuit = synthetic.mul_chain_direct(ctx, log_n)
        cols = [F.fr_vec_to_bytes(c) for c in synthetic.mul_chain_witness(n - 3, n)]
        vk1 = circuit.handle.verifying_key()
        vk2 = circuit.handle.verifying_key_v2(0)
        run = {"v1": lambda: circuit.handle.prove_inputs(cols, b""),
               "v2": lambda: circuit.handle.prove_v2(vk2, cols, 0)[0]}
        proofs = {k: fn() for k, fn in run.items()}   # warm-up
        walls = {k: [] for k in run}
        phases = {k: [0.0] * len(PHASES) for k in run}
        for _ in range(args.reps):
            for k, fn in run.items():
                ctx.prof_enable(True)
                ctx.prof_reset()
                t = time.perf_counter()
                out = fn()
                walls[k].append((time.perf_counter() - t) * 1e3)
                ms = ctx.prof_get()
                ctx.prof_enable(False)
                phases[k] = [a + ms[p][0] for a, p in zip(phases[k], PHASES)]
                assert out == proofs[k], "%s proof bytes changed between calls" % k
        assert vk2.verify(proofs["v2"], b"")
        ver = {}
        for k, fn in (("tp_vk_verify", lambda: vk1.verify(proofs["v1"], bytes(32 * n))),
                      ("tp_verify_v2", lambda: vk2.verify(proofs["v2"], b""))):
            assert fn()
            ts = []
            for _ in range(args.reps):
                t = time.perf_counter()
                fn()
                ts.append((time.perf_counter() - t) * 1e3)
            ver[k] = statistics.median(ts)
        line = {"case": "prove_v2", "log_n": log_n, **info, "reps": args.reps,
                "tp_prove_ms": statistics.median(walls["v1"]), "tp_prove_v2_ms": statistics.median(walls["v2"]),
                "tp_prove_ms_all": walls["v1"], "tp_prove_v2_ms_all": walls["v2"],
                "phases_v1_ms": dict(zip(PHASES, [p / args.reps for p in phases["v1"]])),
                "phases_v2_ms": dict(zip(PHASES, [p / args.reps for p in phases["v2"]])),
                "verify_ms": ver, "proof_bytes": {"v1": len(proofs["v1"]), "v2": len(proofs["v2"])}}
        print(json.dumps(line), flush=True)
        lines.append(line)
        vk1.destroy()
        circuit.handle.destroy()
        ctx.close()
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
