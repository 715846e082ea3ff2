"""Batch verification against one-at-a-time verification (tp_verify_batch vs tp_verify), one JSON line per case.

    python tools/verify_batch_bench.py [--logs 16,20] [--counts 1,16,256,4096] [--reps 3] [--out FILE]

Circuit: the mul_chain of BASELINE.json at 2^log_n rows; the batch cycles through `--distinct` honest proofs.  Per case:
  batch_ms / per_proof_us          wall time of verify_batch (median of --reps, after one warm-up call)
  single_ms_total                   K x tp_verify, measured for K <= 256 (`single_extrapolated`: from the K = 256 run)
  eval_kernel_ms, subgroup_ms       k_multi_eval (+ its range sum) and k_subgroup_flags, torch.profiler, own run
  msm_ms                            the MSM phase timer of the library (tp_prof_*), own run
  host_ms                           batch_ms - the three above: parsing, hashing, scalars, pairing, copies
  eval_roof_frac                    2 K n Fr products x 112 wide products each / tp_measure_imad_peak, over eval_kernel_ms
The GPU name and power limit are read in the same run and written into every line.
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

WIDE_PER_FR_MUL = 112   # DESIGN.md section 4: wide products per Montgomery Fr multiplication


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers stay meaningful with the name from torch
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def kernel_ms(fn, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k in names:
            if k in ev.key:
                out[k] += ev.device_time_total / 1000.0 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,20")
    ap.add_argument("--counts", default="1,16,256,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--distinct", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch  # noqa: F401  (CUDA context for the profiler)
    from typlonk_b200 import field as F, synthetic
    from typlonk_b200.ffi import Context
    from oracle.pyoracle import rng

    info = gpu_info()
    ctx = Context(0)
    _, wide_per_s = ctx.measure_imad_peak()
    lines = []
    for log_n in [int(x) for x in args.logs.split(",")]:
        n = 1 << log_n
        circuit = synthetic.mul_chain_direct(ctx, log_n)
        proofs = []
        for k in range(args.distinct):
            cols = synthetic.mul_chain_witness(n - 3, n, x0=3 + k, blind=rng.fr_rand_stream(500 + k, 9))
            proofs.append(circuit.handle.prove([F.fr_vec_to_bytes(c) for c in cols], bytes(32 * n)))
        h = circuit.handle
        assert h.verify(proofs[0], bytes(32))
        single_per_proof = None
        for K in [int(x) for x in args.counts.split(",")]:
            batch = [proofs[k % len(proofs)] for k in range(K)]
            pis = [bytes(32)] * K
            assert h.verify_batch(batch, pis) == (True, [True] * K)   # warm-up (and the verdict)
            walls = []
            for _ in range(args.reps):
                t = time.perf_counter()
                h.verify_batch(batch, pis)
                walls.append((time.perf_counter() - t) * 1e3)
            batch_ms = statistics.median(walls)
            extrapolated = K > 256
            if not extrapolated:
                t = time.perf_counter()
                for p in batch:
                    h.verify(p, bytes(32))
                single_total = (time.perf_counter() - t) * 1e3
                single_per_proof = single_total / K
            else:
                single_total = single_per_proof * K
            ctx.prof_enable(True)
            ctx.prof_reset()
            h.verify_batch(batch, pis)
            ph = ctx.prof_get()
            ctx.prof_enable(False)
            msm_ms = ph["msm_total"][0]
            ks = kernel_ms(lambda: h.verify_batch(batch, pis), ["k_multi_eval", "k_subgroup_flags"])
            eval_ms, sub_ms = ks["k_multi_eval"], ks["k_subgroup_flags"]
            roof_ms = 2.0 * K * n * WIDE_PER_FR_MUL / wide_per_s * 1e3
            rec = dict(info, log_n=log_n, K=K, distinct_proofs=len(proofs), reps=args.reps,
                       batch_ms=round(batch_ms, 3), batch_ms_all=[round(w, 3) for w in walls],
                       per_proof_us=round(batch_ms / K * 1e3, 2),
                       single_ms_total=round(single_total, 3), single_per_proof_us=round(single_per_proof * 1e3, 2),
                       single_extrapolated=extrapolated,
                       speedup_per_proof=round(single_total / batch_ms, 2),
                       eval_kernel_ms=round(eval_ms, 3), subgroup_ms=round(sub_ms, 3), msm_ms=round(msm_ms, 3),
                       host_ms=round(batch_ms - eval_ms - sub_ms - msm_ms, 3),
                       eval_roof_ms=round(roof_ms, 4), eval_roof_frac=round(roof_ms / eval_ms, 3) if eval_ms else None,
                       wide_products_per_s=wide_per_s)
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
