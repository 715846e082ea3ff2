"""Compressed against uncompressed wire encodings (csrc/wire.cu), one JSON line per case.

    python tools/wire_bench.py [--logs 20,24] [--counts 256,4096] [--reps 3] [--out FILE]

Cases:
  srs        SRS of 2^log + 3 points: serialise and deserialise (check 1 and 2), uncompressed and compressed; wall time
             of the library call, median of --reps after one warm-up call (deserialisation includes the upload and the
             MSM table levels, the same work in both forms)
  kernel     k_g1_from_wire_compressed / k_g1_from_wire at check 1 and 2 from torch.profiler, in a run of their own;
             for the compressed kernel at check 1 also its share of the multiplier roof: points x wide products per
             point (the Fq products of one decompression, counted from the exponent below, x 288 per product and 222
             per square) over tp_measure_imad_peak's wide-IMAD rate
  proofs     tp_proofs_decompress of K compressed proof blocks against a host loop of tp_proof_decompress
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

Q = 0x1A0111EA397FE69A4B1BA7B6434BACD764774B84F38512BF6730D2A0F6B0F6241EABFFFEB153FFFFB9FEFFFFFFFFAAAB
WIDE_PER_FQ_MUL = 288   # interleaved CIOS, 12 x 32-bit limbs (field.cuh)
WIDE_PER_FQ_SQR = 222   # dedicated square: 78 + 144


def decompress_products():
    """(Fq products, Fq squares) of one record in k_g1_from_wire_compressed at check 1: to Montgomery, x^3, the
    4-bit-window power (14 table products, 4 squares per window, one product per non-zero digit), the root check,
    out of Montgomery for the sign"""
    e = (Q + 1) // 4
    digits = [(e >> (4 * w)) & 15 for w in range(94)]
    muls = 1 + 1 + 14 + sum(1 for d in digits if d) + 1
    sqrs = 1 + 4 * 94 + 1
    return muls, sqrs


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers stay meaningful with the name from torch
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


def kernel_ms(fn, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k in names:
            if k + "(" in ev.key or ev.key == k:
                out[k] += ev.device_time_total / 1000.0 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logs", default="20,24")
    ap.add_argument("--counts", default="256,4096")
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
    muls, sqrs = decompress_products()
    wide_per_point = muls * WIDE_PER_FQ_MUL + sqrs * WIDE_PER_FQ_SQR
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        line = json.dumps({**info, **rec})
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    tau = ffi.fr_rand_stream(1, 1)
    from typlonk_b200 import field as F
    for log in [int(x) for x in args.logs.split(",") if x]:
        srs = Srs.from_secret(ctx, F.fr_from_bytes(tau), 1 << log)
        npts = len(srs)
        raws = {}
        for comp in (False, True):
            # the handle's calls return bytearrays, which cross ctypes without a copy
            ser = srs.handle.serialize_compressed if comp else srs.handle.serialize
            ms, all_ms = timed(ser, args.reps)
            raws[comp] = ser()
            emit({"case": "srs_serialize", "points": npts, "compressed": comp, "bytes": len(raws[comp]),
                  "ms": round(ms, 3), "ms_all": [round(t, 3) for t in all_ms]})
        for check in (1, 2):
            for comp in (False, True):
                def load():
                    Srs.from_bytes(ctx, raws[comp], check, compressed=comp).handle.destroy()
                ms, all_ms = timed(load, args.reps)
                emit({"case": "srs_deserialize", "points": npts, "compressed": comp, "check": check,
                      "bytes": len(raws[comp]), "ms": round(ms, 3), "ms_all": [round(t, 3) for t in all_ms]})
        # kernel times, profiler on, separate calls
        for check in (1, 2):
            for comp in (False, True):
                name = "k_g1_from_wire_compressed" if comp else "k_g1_from_wire"
                k = kernel_ms(lambda: Srs.from_bytes(ctx, raws[comp], check, compressed=comp).handle.destroy(), [name])[name]
                rec = {"case": "kernel", "kernel": name, "points": npts, "check": check, "kernel_ms": round(k, 3)}
                if comp and check == 1:
                    roof_ms = npts * wide_per_point / wide_peak * 1e3
                    rec.update({"fq_mul_per_point": muls, "fq_sqr_per_point": sqrs, "wide_per_point": wide_per_point,
                                "wide_imad_per_s": wide_peak, "roof_ms": round(roof_ms, 3),
                                "roof_frac": round(roof_ms / k, 3) if k else None})
                emit(rec)
        for comp in (False, True):
            name = "k_g1_to_wire_compressed" if comp else "k_g1_to_wire"
            k = kernel_ms(srs.handle.serialize_compressed if comp else srs.handle.serialize, [name])[name]
            emit({"case": "kernel", "kernel": name, "points": npts, "kernel_ms": round(k, 3)})
        srs.handle.destroy()
        del raws

    proofs = json.load(open(os.path.join(ROOT, "tests", "golden", "proofs.json")))
    blocks = [ffi.proof_compress(bytes.fromhex(p["proof_hex"])[:ffi.PROOF_FIXED_BYTES]) for p in proofs.values()]
    for count in [int(x) for x in args.counts.split(",") if x]:
        blob = b"".join(blocks[k % len(blocks)] for k in range(count))
        ms, all_ms = timed(lambda: ctx.proofs_decompress(blob, count), args.reps)
        got, status = ctx.proofs_decompress(blob, count)
        assert status == [0] * count
        loop_reps = 1 if count > 256 else args.reps

        def loop():
            return b"".join(ffi.proof_decompress(blob[k * 848:(k + 1) * 848]) for k in range(count))
        lms, lall = timed(loop, loop_reps)
        assert loop() == got
        emit({"case": "proofs_decompress", "K": count, "batch_ms": round(ms, 3), "batch_ms_all": [round(t, 3) for t in all_ms],
              "per_proof_us": round(ms * 1e3 / count, 2), "host_loop_ms": round(lms, 3),
              "host_loop_ms_all": [round(t, 3) for t in lall], "host_per_proof_us": round(lms * 1e3 / count, 2),
              "speedup": round(lms / ms, 2)})
    ctx.close()


if __name__ == "__main__":
    main()
