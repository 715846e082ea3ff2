"""Verification keys on the device, one JSON line per case (written to --out, profiles/verify_key_b200.jsonl by default).

    python tools/verify_key_bench.py [--logs 16,20,22] [--reps 3] [--baseline-tree DIR] [--out FILE]

Cases (circuit: the mul_chain of BASELINE.json at 2^log_n rows):
  key        key bytes, tp_vk_serialize and tp_vk_deserialize wall time at check 1 and 2 (median of --reps)
  single     tp_vk_verify against tp_verify per proof, the mean over 8 honest proofs after a warm-up
  multi_key  4 keys (2^13 .. 2^16) x 64 proofs: tp_vk_verify_batch wall against a loop of tp_vk_verify, and the
             job-table k_multi_eval (+ its range sum) kernel time from torch.profiler with its fraction of the
             multiplier roof (2 K n Fr products x 112 wide products over tp_measure_imad_peak, summed over the keys)
  verify_batch  tp_verify_batch at K = 256, 2^20 through tools/verify_batch_bench.py, run alternately from this tree and
             from --baseline-tree (another checkout with its library built), twice each
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from verify_batch_bench import WIDE_PER_FR_MUL, gpu_info, kernel_ms  # noqa: E402


def median_ms(fn, reps):
    walls = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t) * 1e3)
    return statistics.median(walls), walls


def chain_proofs(circuit, n, count, seed):
    from oracle.pyoracle import rng
    from typlonk_b200 import field as F, synthetic
    cols = [[F.fr_vec_to_bytes(c) for c in synthetic.mul_chain_witness(n - 3, n, x0=3 + k, blind=rng.fr_rand_stream(seed + k, 9))]
            for k in range(count)]
    blocks, status = circuit.handle.prove_batch(cols, [b""] * count)
    assert status == [0] * count
    return blocks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,20,22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "verify_key_b200.jsonl"))
    args = ap.parse_args()

    import torch  # noqa: F401  (CUDA context for the profiler)
    from typlonk_b200 import synthetic
    from typlonk_b200.ffi import Context

    info = gpu_info()
    ctx = Context(0)
    _, wide_per_s = ctx.measure_imad_peak()
    lines = []

    def emit(rec):
        line = json.dumps(dict(info, **rec))
        print(line, flush=True)
        lines.append(line)

    for log_n in [int(x) for x in args.logs.split(",")]:
        n = 1 << log_n
        circuit = synthetic.mul_chain_direct(ctx, log_n)
        h = circuit.handle
        vk = h.verifying_key()
        raw = vk.serialize()
        ser_ms, ser_all = median_ms(vk.serialize, args.reps)
        de = {}
        for check in (1, 2):
            ctx.vk_deserialize(raw, check).destroy()   # warm-up
            keys = []
            de[check] = median_ms(lambda: keys.append(ctx.vk_deserialize(raw, check)), args.reps)
            for k in keys:
                k.destroy()
        emit(dict(case="key", log_n=log_n, key_bytes=len(raw), serialize_ms=round(ser_ms, 3),
                  serialize_ms_all=[round(w, 3) for w in ser_all],
                  deserialize_check1_ms=round(de[1][0], 3), deserialize_check2_ms=round(de[2][0], 3),
                  deserialize_ms_all={str(c): [round(w, 3) for w in de[c][1]] for c in de}))
        if log_n <= 20:
            proofs = chain_proofs(circuit, n, 8, 700)
            z = bytes(32)
            assert h.verify(proofs[0], z) and vk.verify(proofs[0], z)   # warm-up
            t = time.perf_counter()
            assert all(h.verify(p, z) for p in proofs)
            circ_us = (time.perf_counter() - t) * 1e6 / len(proofs)
            t = time.perf_counter()
            assert all(vk.verify(p, z) for p in proofs)
            key_us = (time.perf_counter() - t) * 1e6 / len(proofs)
            emit(dict(case="single", log_n=log_n, proofs=len(proofs), tp_verify_us=round(circ_us, 1),
                      tp_vk_verify_us=round(key_us, 1)))
        vk.destroy()
        h.destroy()
        circuit.srs.handle.destroy()

    # several keys in one batch
    logs = [13, 14, 15, 16]
    per_key = 64
    circuits = [synthetic.mul_chain_direct(ctx, lg) for lg in logs]
    keys = [c.handle.verifying_key() for c in circuits]
    blocks, key_of = [], []
    per = [chain_proofs(c, 1 << lg, per_key, 900 + 100 * j) for j, (c, lg) in enumerate(zip(circuits, logs))]
    for k in range(per_key):
        for j in range(len(logs)):
            blocks.append(per[j][k])
            key_of.append(j)
    pis = [b""] * len(blocks)
    run = lambda: ctx.vk_verify_batch(keys, key_of, blocks, pis)  # noqa: E731
    assert run() == (True, [True] * len(blocks))
    batch_ms, batch_all = median_ms(run, args.reps)
    t = time.perf_counter()
    assert all(keys[j].verify(b, b"") for b, j in zip(blocks, key_of))
    loop_ms = (time.perf_counter() - t) * 1e3
    ks = kernel_ms(run, ["k_multi_eval", "k_subgroup_flags"])
    eval_ms = ks["k_multi_eval"]
    roof_ms = sum(2.0 * per_key * (1 << lg) * WIDE_PER_FR_MUL / wide_per_s * 1e3 for lg in logs)
    emit(dict(case="multi_key", key_logs=logs, proofs_per_key=per_key, proofs=len(blocks),
              batch_ms=round(batch_ms, 3), batch_ms_all=[round(w, 3) for w in batch_all],
              vk_verify_loop_ms=round(loop_ms, 3), speedup=round(loop_ms / batch_ms, 2),
              eval_kernel_ms=round(eval_ms, 3), subgroup_ms=round(ks["k_subgroup_flags"], 3),
              eval_roof_ms=round(roof_ms, 4), eval_roof_frac=round(roof_ms / eval_ms, 3) if eval_ms else None,
              wide_products_per_s=wide_per_s))
    for k in keys:
        k.destroy()
    for c in circuits:
        c.handle.destroy()
        c.srs.handle.destroy()
    ctx.close()

    # tp_verify_batch at K = 256, 2^20: this tree and the baseline tree, alternately, each in its own process
    trees = [("this", ROOT)] + ([("baseline", os.path.abspath(args.baseline_tree))] if args.baseline_tree else [])
    for rnd in range(2):
        for label, tree in trees:
            res = subprocess.run([sys.executable, os.path.join(tree, "tools", "verify_batch_bench.py"), "--logs", "20",
                                  "--counts", "256", "--reps", str(args.reps)], capture_output=True, text=True, cwd=tree)
            recs = [json.loads(x) for x in res.stdout.splitlines() if x.startswith("{")]
            if res.returncode != 0 or not recs:
                emit(dict(case="verify_batch", tree=label, round=rnd, error=res.stderr[-2000:]))
                continue
            r = recs[0]
            emit(dict(case="verify_batch", tree=label, round=rnd, log_n=20, K=256, batch_ms=r["batch_ms"],
                      batch_ms_all=r["batch_ms_all"], eval_kernel_ms=r["eval_kernel_ms"],
                      eval_roof_frac=r["eval_roof_frac"]))

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
