"""SRS ceremony timings (csrc/srs_ceremony.cu, k_srs_contribute in csrc/srs.cu), one JSON line per case.

    python tools/srs_ceremony_bench.py [--logs 16,20,22,24] [--reps 3] [--out FILE]

Cases, for an SRS of 2^log points:
  contribute  tp_srs_contribute wall time, median of --reps after one warm-up call.  Split: k_srs_contribute and the
              table rebuild (k_srs_next_level) from torch.profiler in a run of their own; host_ms is the wall time of a
              contribution to a 16-point SRS, i.e. the two G2 multiplications, the G2 preparation and the call, which
              run on the host while the device works
  verify      tp_srs_verify wall time, median of --reps after a warm-up.  Split: k_subgroup_flags, k_pow_table and the
              MSM (every other kernel of the call) from torch.profiler; host_ms is the wall time of verifying a 16-point
              SRS, i.e. the G2 subgroup check and the pairing product
  roof        k_srs_contribute against the multiplier roof: Fq products and squares per point counted from the laws in
              ec.cuh (doubling 6M + 3S, mixed addition 8M + 2S; fq_mul_sub2 counted as two products) for the scalar
              bits of the powers used, plus 6M of normalisation, weighted 288 / 222 wide products, over the wide-IMAD
              rate tp_measure_imad_peak measures in the same run
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

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
WIDE_PER_FQ_MUL = 288   # interleaved CIOS, 12 x 32-bit limbs (field.cuh)
WIDE_PER_FQ_SQR = 222   # dedicated square: 78 + 144


def ladder_products(s, count=4096):
    """mean (Fq products, Fq squares) per point over the first `count` powers of s: per scalar bit below the leading
    one a doubling (6M + 3S), per set bit among them a mixed addition (8M + 2S); 6M of affine normalisation"""
    muls = sqrs = 0
    k = 1
    for _ in range(count):
        bits = k.bit_length() - 1
        adds = bin(k).count("1") - 1
        muls += 6 * bits + 8 * adds + 6
        sqrs += 3 * bits + 2 * adds
        k = k * s % R
    return muls / count, sqrs / count


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % type(e).__name__}


def timed(fn, reps):
    fn()   # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), ts


def kernel_ms(fn):
    """device time per kernel name of one call, from torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if t <= 0 or ev.key.startswith("Memcpy") or ev.key.startswith("Memset"):
            continue
        key = ev.key.replace("(anonymous namespace)::", "")
        name = key.split("(")[0].split("<")[0].split("::")[-1].split(" ")[-1]
        out[name] = out.get(name, 0.0) + t / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="16,20,22,24")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    from typlonk_b200 import ffi
    from typlonk_b200.kzg import Srs
    info = gpu_info()
    ctx = ffi.Context(0)
    _, wide_peak = ctx.measure_imad_peak()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        line = json.dumps({**info, **rec})
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    tau = int.from_bytes(os.urandom(31), "little") + 1
    s = ffi.fr_rand_stream(11, 1)
    from typlonk_b200 import field as F
    s_int = F.fr_from_bytes(s)

    def contribute(srs):
        srs.contribute(s_int)[0].handle.destroy()

    small = Srs.from_secret(ctx, tau, 13)
    host_contrib_ms, _ = timed(lambda: contribute(small), args.reps)
    host_verify_ms, _ = timed(small.verify, args.reps)
    muls, sqrs = ladder_products(s_int)
    wide_per_point = muls * WIDE_PER_FQ_MUL + sqrs * WIDE_PER_FQ_SQR
    for log in [int(x) for x in args.logs.split(",") if x]:
        srs = Srs.from_secret(ctx, tau, (1 << log) - 3)
        n = len(srs)
        ms, all_ms = timed(lambda: contribute(srs), args.reps)
        ks = kernel_ms(lambda: contribute(srs))
        kc = ks.get("k_srs_contribute", 0.0)
        emit({"case": "contribute", "points": n, "ms": round(ms, 3), "ms_all": [round(t, 3) for t in all_ms],
              "k_srs_contribute_ms": round(kc, 3), "tables_ms": round(ks.get("k_srs_next_level", 0.0), 3),
              "host_ms": round(host_contrib_ms, 3)})
        roof_ms = n * wide_per_point / wide_peak * 1e3
        emit({"case": "roof", "kernel": "k_srs_contribute", "points": n, "kernel_ms": round(kc, 3),
              "fq_mul_per_point": round(muls, 1), "fq_sqr_per_point": round(sqrs, 1),
              "wide_per_point": round(wide_per_point), "wide_imad_per_s": wide_peak, "roof_ms": round(roof_ms, 3),
              "roof_frac": round(roof_ms / kc, 3) if kc else None})
        assert srs.verify()
        ms, all_ms = timed(srs.verify, args.reps)
        ks = kernel_ms(srs.verify)
        sub, pw = ks.pop("k_subgroup_flags", 0.0), ks.pop("k_pow_table", 0.0)
        emit({"case": "verify", "points": n, "ms": round(ms, 3), "ms_all": [round(t, 3) for t in all_ms],
              "k_subgroup_flags_ms": round(sub, 3), "k_pow_table_ms": round(pw, 3),
              "msm_ms": round(sum(ks.values()), 3), "msm_kernels": sorted(ks), "host_ms": round(host_verify_ms, 3)})
        srs.handle.destroy()
    ctx.close()


if __name__ == "__main__":
    main()
