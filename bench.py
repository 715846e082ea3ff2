#!/usr/bin/env python3
"""Headline benchmark: full PLONK prove of the synthetic mul-chain circuit (BASELINE.json configs[2]: 2^20 rows)
through the reference-facing C ABI (tp_prove_dev / tp_prove_inputs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--log-n L] [--impl reference] [--no-sweep] [--no-north-star]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one complete proof (13 G1 MSMs, 5 iNTT + 20 coset NTT + 4 inverse coset
NTT, grand product, quotient, 6 openings).  `value` = prove ms with the witness resident in HBM; `e2e` = the same
through tp_prove_inputs with pinned HOST buffers (H2D of the 3 witness columns + public inputs and D2H of the proof
inside the timed region).  The proof bytes of every run are compared with the CPU oracle's golden proof of the same
workload (tests/golden/mulchain_big.json, made by tools/make_golden_big.py) -> `parity`.

N > 1 (torchrun, one process per GPU): the library owns the NCCL communicator (tp_ctx_comm_init_rank; the 128-byte id
travels once over torch.distributed before anything is timed).  Every MSM is sharded by bucket with the per-rank
reduction outputs all-gathered and combined on the device, the quotient by coset of the 4n domain, the witness upload
by rows; no Python runs inside a proof.  Strong scaling.

Also in the line: `north_star` -- the 2^22-gate prove of BASELINE.json configs[4] on the same N GPUs, digest-checked;
`standalone` -- G1 MSM Mpts/s and NTT GB/s at the prover's size on these N GPUs; `sweeps` (N = 1) -- MSM 2^16..2^26
incl. the skewed and all-equal cases, NTT / iNTT / coset NTT 2^16..2^24; `cpu_baseline` (N = 1) -- ONE real 2^20 prove
of the oracle's C++ port on all host threads, no extrapolation.

`--impl reference` times the CPU oracle port (oracle/c, all host threads) on the SAME 2^20 workload: full proves, as
many of the K requested as fit in ~150 s (at least one); `steps` in its line is the number actually timed.

`--dump-outputs DIR` (rank 0) writes what the last timed step returned to its caller, for the GPU prover and for
`--impl reference` alike, so that two builds, or the GPU and the CPU port, can be compared output for output on the same
seeded inputs: DIR/proof.npy, the 1472-byte proof block (TP_PROOF_FIXED_BYTES: 13 G1
points of 96 B and 7 Fr of 32 B) as float64 values 0..255, so that any changed byte differs by at least 1.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "prove_ms"
UNIT = "ms"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: an NVML polling thread (20 ms period;
    the main thread sits in ctypes / CUDA calls that release the GIL), nvidia-smi -lms as the fallback."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.thread = None
        self.proc = None
        self.lines = []

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            bits = {N.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                    N.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                    N.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                    N.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}

            def poll():
                while not self.stop_flag.is_set():
                    try:
                        self.sm.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                        r = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                        for bit, name in bits.items():
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:  # noqa: BLE001
                        pass
                    self.stop_flag.wait(0.02)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:  # noqa: BLE001
            self.thread = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None and self.thread is not None:      # NVML path
            self.stop_flag.set()
            self.thread.join(timeout=2)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


def _golden(log_n):
    try:
        with open(os.path.join(ROOT, "tests", "golden", "mulchain_big.json")) as f:
            return json.load(f).get("2^%d" % log_n)
    except Exception:  # noqa: BLE001
        return None


def _parity(proof: bytes, log_n: int):
    import hashlib
    digest = hashlib.sha256(proof).hexdigest()
    g = _golden(log_n)
    if g is None:
        return {"digest_ok": None, "vs": "no golden proof committed for n=2^%d" % log_n, "sha256": digest}
    return {"digest_ok": digest == g["sha256"] and proof.hex() == g["proof_hex"], "sha256": digest,
            "vs": "c-oracle golden (tests/golden/mulchain_big.json, all 1472 proof bytes)"}


def _dump(args, proof: bytes):
    """--dump-proof / --dump-outputs: the proof of the last timed step, whichever implementation was timed."""
    if args.dump_proof:
        with open(args.dump_proof, "wb") as f:
            f.write(proof)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "proof.npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float64))


def _cpu_prove(log_n, budget_s, max_steps):
    """Full proves of the oracle's C++ port on all host threads: (ms per prove, proves timed, threads, proof)."""
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)   # torchrun exports OMP_NUM_THREADS=1
    from oracle import coracle  # the only product-side place allowed to execute oracle/
    tau, sel, perm, cols, pi = coracle.mul_chain_inputs(log_n)
    c = coracle.Circuit(tau, sel, perm, 1 << log_n)
    times, proof = [], None
    t_start = time.perf_counter()
    while len(times) < max(max_steps, 1):
        t0 = time.perf_counter()
        proof = c.prove(cols, pi)
        times.append((time.perf_counter() - t0) * 1e3)
        spent = time.perf_counter() - t_start
        if spent + times[-1] / 1e3 > budget_s:   # the next one would not fit
            break
    c.close()
    return sum(times) / len(times), len(times), coracle.threads(), proof


def _b0_as_written(log_n):
    """BASELINE.md B0: the reference's OWN algorithms (kzg/src/lib.rs:46-53 per-point double-and-add + affine conversion;
    plonk/src/proof.rs:317-359 `naive_mul`), timed small on one core by the oracle's C++ statement of them and
    EXTRAPOLATED to n = 2^log_n by their n and n^2 laws: 13 commitments of n points + ~19 n^2 schoolbook multiply-adds."""
    from oracle import coracle
    m = 1 << 10
    tau, sel, perm, cols, pi = coracle.mul_chain_inputs(10)
    c = coracle.Circuit(tau, sel, perm, m)
    coeffs = coracle.fr_rand_stream(3, m)
    t0 = time.perf_counter()
    c.commit_as_written(coeffs)
    t_point = (time.perf_counter() - t0) / m
    c.close()
    k = 1 << 11
    a = coracle.fr_rand_stream(4, k)
    t0 = time.perf_counter()
    coracle.naive_mul(a, a)
    t_pair = (time.perf_counter() - t0) / (k * k)
    n = float(1 << log_n)
    commit_s, quotient_s = 13 * n * t_point, 19 * n * n * t_pair
    return {"value": (commit_s + quotient_s) * 1e3, "unit": UNIT, "cores": 1, "kind": "reference algorithm, EXTRAPOLATED",
            "commit_us_per_point": round(t_point * 1e6, 2), "naive_mul_ns_per_coefficient_pair": round(t_pair * 1e9, 3),
            "commit_s": round(commit_s, 1), "quotient_s": round(quotient_s, 1),
            "sample": "measured: one as-written commit of 2^10 points and one 2^11 x 2^11 naive_mul on one core; "
                      "extrapolated by 13 n and 19 n^2 to n=2^%d (never run at that size: it would take days)" % log_n}


def run_reference(args):
    """CPU arm: the oracle's C++ port of the reference prover on the host cores, on the bench's own workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ms, done, threads, proof = _cpu_prove(args.log_n, args.ref_budget_s, args.steps)
    sample = "%d full prove(s) at n=2^%d, %.0f ms each, %d host threads (requested %d steps; bounded to ~%d s)" % (
        done, args.log_n, ms, threads, args.steps, args.ref_budget_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": ms, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": 0, "ms_per_step": ms, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64-limb Montgomery Fr/Fq (integer)", "data": "synthetic",
        "config": {"workload": "mulchain_prove_n=2^%d" % args.log_n, "gates": (1 << args.log_n) - 3},
        "cpu_baseline": {"value": ms, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": ms, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "parity": _parity(proof, args.log_n),
        "timed_region_s": round(ms * done / 1e3, 1),
    }
    _dump(args, proof)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--impl", default="typlonk_b200")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="--impl reference: stop starting proves after this long")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the MSM / NTT size sweeps (N = 1)")
    ap.add_argument("--no-north-star", action="store_true", help="skip the 2^22-gate prove")
    ap.add_argument("--north-star-log-n", type=int, default=22)
    ap.add_argument("--ab", action="append", default=[], metavar="OPT=VAL[,OPT=VAL]",
                    help="also time the resident prove with these tp_ctx_set_option settings (repeatable); reported under "
                         "'ab', never as the headline value")
    ap.add_argument("--dump-proof", default=None, help="write the proof bytes of the last timed step to this file (rank 0)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the output of the last timed step as DIR/proof.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from typlonk_b200 import field as F, synthetic
    from typlonk_b200.ffi import Context, PHASES

    # a non-default torch stream: its handle is what the library launches on, so torch.cuda.Event
    # timings bracket the library's kernels (the legacy default stream has handle 0 = "make your own")
    # ($TP_BENCH_STREAM_PRIORITY=-1 puts it above the lowest-priority stream the library's optional MSM pipe
    # accumulates on; the default stays an ordinary stream)
    tstream = torch.cuda.Stream(device=dev, priority=int(os.environ.get("TP_BENCH_STREAM_PRIORITY", "0")))
    torch.cuda.set_stream(tstream)
    ctx = Context(local_rank, tstream.cuda_stream)

    if world > 1:
        # The library owns its NCCL communicator.  The one thing it needs from the host language is rank 0's 128-byte id,
        # handed over here, once, before anything is timed; no Python runs inside a proof afterwards.
        from typlonk_b200 import ffi as _ffi
        idt = torch.zeros(_ffi.COMM_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(_ffi.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, src=0)
        torch.cuda.synchronize()
        ctx.comm_init_rank(rank, world, bytes(idt.cpu().numpy().tobytes()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    def to_tensor(b):
        return torch.frombuffer(bytearray(b), dtype=torch.uint8)

    def workload(log_n):
        """Circuit + device-resident witness + pinned host witness of the 2^log_n mul chain."""
        n = 1 << log_n
        t0 = time.time()
        circuit = synthetic.mul_chain_direct(ctx, log_n)
        cols = synthetic.mul_chain_witness(n - 3, n)
        host = [to_tensor(F.fr_vec_to_bytes(c)).pin_memory() for c in cols] + [torch.zeros(32 * n, dtype=torch.uint8).pin_memory()]
        devt = [h.to(dev) for h in host]
        torch.cuda.synchronize()
        return circuit, host, devt, time.time() - t0

    log_n = args.log_n
    n = 1 << log_n
    circuit, host, devt, setup_s = workload(log_n)

    def step_resident():
        return circuit.handle.prove_dev([t.data_ptr() for t in devt[:3]], devt[3].data_ptr())

    # the public-input vector as the reference's caller passes it: `circuit.prove(inputs, vec![0])` (README.md:29,
    # builder/test.rs:28) -- one element; the library zero-fills the other n - 1 rows on the device (proof.rs:52-53)
    host_pi = torch.zeros(32, dtype=torch.uint8).pin_memory()

    def step_e2e():
        return circuit.handle.prove_inputs([h.data_ptr() for h in host[:3]], host_pi.numpy())

    for _ in range(args.warmup):
        proof = step_resident()
    l2_flush = "inputs+tables (%.1f GiB working set) exceed the 126 MB L2" % ((13 * 4 + 30) * n * 32 / 2**30) \
        if log_n >= 18 else "working set may fit L2 at this size"

    sampler = ClockSampler(local_rank)
    if rank == 0:   # one poller per job: the line carries rank 0's clocks, and NVML queries take a driver lock
        sampler.start()
    ctx.prof_reset()
    ctx.prof_enable(True)
    l0 = ctx.launch_count()
    ms_total, proof = timed(step_resident, args.steps)
    launches = ctx.launch_count() - l0
    prof = ctx.prof_get()
    msms, entries = ctx.get_stat("msm_calls"), ctx.get_stat("msm_entries")   # of the K timed steps only
    ctx.prof_enable(False)
    for _ in range(args.warmup):   # the first sharded uploads also set up their NCCL transfers
        step_e2e()
    e2e_wall = []

    def step_e2e_logged():   # host wall clock per step (the call returns with the proof): shows outliers, adds no barrier
        t1 = time.perf_counter()
        out = step_e2e()
        e2e_wall.append(round((time.perf_counter() - t1) * 1e3, 3))
        return out
    ms_e2e, proof_e2e = timed(step_e2e_logged, args.steps)
    clocks = sampler.stop()
    e2e_sample = [round(timed(step_e2e, 1)[0], 3) for _ in range(3)]   # three more, each timed alone (diagnostic)
    assert proof == proof_e2e, "resident and host-buffer proofs differ"
    parity = _parity(proof, log_n)
    if world > 1:   # every rank must hold the same bytes
        import hashlib
        dg = torch.frombuffer(bytearray(hashlib.sha256(proof).digest()), dtype=torch.uint8).to(dev)
        alld = [torch.empty_like(dg) for _ in range(world)]
        dist.all_gather(alld, dg)
        parity["ranks_agree"] = all(bool((x == dg).all().item()) for x in alld)
    # the proof just timed goes through the product verifier (device: PI / sigma evaluations, circuit commitments on the
    # first call; host: pairings).  Outside the timed region; wall clock because the pairing half is host work.
    tv = []
    for _ in range(3):
        t1 = time.perf_counter()
        ok = circuit.handle.verify(proof, bytes(32))
        tv.append((time.perf_counter() - t1) * 1e3)
        assert ok, "tp_verify rejects the proof the bench just produced"
    bad = bytearray(proof)
    bad[192] ^= 1
    assert not circuit.handle.verify(bytes(bad), bytes(32)), "tp_verify accepts a corrupted proof"
    verify = {"first_call_ms": round(tv[0], 2), "ms": round(min(tv[1:]), 2), "accepted": True,
              "note": "first call includes the 8 circuit-commitment MSMs, cached afterwards"}

    # library tunables A/B-ed in this very process (same box, same clocks, same circuit): each variant is warmed up,
    # timed like the headline, byte-checked, and the defaults are restored
    DEFAULTS = {"ntt_radix_log": 2, "msm_pipeline": 0, "msm_acc_staged": 0, "msm_reduce_l1": 0, "quotient_all_cosets": 0}
    ab = []
    for spec in args.ab:
        opts = {k: int(v) for k, v in (kv.split("=") for kv in spec.split(","))}
        for k, v in opts.items():
            ctx.set_option(k, v)
        for _ in range(2):
            step_resident()
        ctx.prof_reset()
        ctx.prof_enable(True)
        ms_ab, proof_ab = timed(step_resident, args.steps)
        prof_ab = ctx.prof_get()
        ctx.prof_enable(False)
        for k in opts:
            ctx.set_option(k, DEFAULTS.get(k, 0))
        ab.append({"options": opts, "prove_ms": round(ms_ab / args.steps, 3), "same_bytes": proof_ab == proof,
                   "phases_ms_per_step": {p_: round(prof_ab[p_][0] / args.steps, 3) for p_ in PHASES}})

    # BASELINE.json's metric names two more numbers next to the prove time: G1 MSM Mpts/s and NTT GB/s (algorithmic
    # 64 * N bytes per transform, SURVEY.md 8(d)), "at 1/2/4/8 B200".  Measured here on the prover's own SRS and a witness
    # column, device resident, after the timed region: the MSM sharded over the N GPUs like the prover's (every rank
    # calls it), the NTT on one GPU (a single transform is not split; the prover shards NTTs by coset).
    def per_call(fn, reps=5):
        fn()
        ms, _ = timed(fn, reps)
        return ms / reps
    scal = devt[2].clone()
    msm_ms = per_call(lambda: ctx.commit_dev(circuit.srs.handle, scal.data_ptr(), n))
    ntt_ms = per_call(lambda: ctx.ntt_dev(scal.data_ptr(), log_n))
    intt_ms = per_call(lambda: ctx.ntt_dev(scal.data_ptr(), log_n, inverse=True))
    cos_ms = per_call(lambda: ctx.ntt_dev(scal.data_ptr(), log_n, coset_mont=F.fr_to_bytes(7)))
    standalone = {"log_n": log_n, "n_gpus": world,
                  "msm_ms": round(msm_ms, 4), "msm_mpts_per_s": round(n / msm_ms / 1e3, 1),
                  "ntt_ms": round(ntt_ms, 4), "ntt_gb_per_s": round(64.0 * n / ntt_ms / 1e6, 1),
                  "intt_ms": round(intt_ms, 4), "coset_ntt_ms": round(cos_ms, 4),
                  "ntt_hbm_frac": round(64.0 * n / ntt_ms / 1e6 / _peaks()[0], 4),
                  "note": "msm: one commitment sharded over n_gpus; ntt: one transform on one GPU"}
    del scal

    ms_step = ms_total / args.steps
    hbm_peak, peak_kind = _peaks()
    # dominant kernel: MSM bucket accumulation.  Algorithmic bytes per MSM = 128 B / point
    # (96 B base + 32 B scalar, SURVEY.md 8(d)); a launch processes this rank's share of every
    # MSM in its batch (13 MSMs per proof go out as batches of 3 + 1 + 9 = 3 launches).
    acc_ms, acc_launches = prof["msm_accum"]
    acc_launch_ms = acc_ms / max(acc_launches, 1)
    pts_per_launch = (n / world) * msms / max(acc_launches, 1)
    achieved = (128.0 * pts_per_launch) / (acc_launch_ms * 1e-3) / 1e9 if acc_ms > 0 else None
    affine = bool(int(os.environ.get("TP_MSM_AFFINE", "0")))
    kernel = "k_msm_accumulate_affine" if affine else "k_msm_accumulate"
    # DRAM bytes per bucket addition of that kernel, from the committed `ncu --set full` capture
    # (profiles/traffic.json; dram__bytes_read.sum + dram__bytes_write.sum over the additions of the launch)
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)[kernel]["dram_bytes_per_addition"] * entries / max(acc_launches, 1)
    except Exception:  # noqa: BLE001
        pass
    imad, imad_wide = ctx.measure_imad_peak()
    roofline = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": hbm_peak,
                "unit": "GB/s", "frac": (achieved / hbm_peak) if achieved else None, "traffic": traffic,
                "peak_kind": peak_kind,
                "note": "381-bit Montgomery arithmetic makes this kernel integer-pipe bound (SURVEY 8d): see roofline_int; "
                        "traffic exceeds the 128 B/point figure by design: every point is read once per window from "
                        "its fixed-base table level"}
    # integer roofline of the same kernel: wide multiply-adds (IMAD.WIDE.U32.X) retired per second against the
    # measured peak of that instruction (tp_measure_imad_peak, carry-chain form).  Per bucket addition:
    # XYZZ mixed = 8 x 288 + 2 x 222; affine chain = 5 x 288 + 222 + (3.9e3 + 288)/16 for the shared inversion.
    per_add = (5 * 288 + 222 + (3900 + 288) / 16.0) if affine else (8 * 288 + 2 * 222)
    prod_rate = entries * per_add / (acc_ms * 1e-3) if acc_ms > 0 else None
    roofline_int = {"bound": "fma-heavy pipe (IMAD.WIDE.U32.X)", "kernel": kernel, "achieved": prod_rate,
                    "peak": imad_wide, "unit": "wide multiply-adds/s", "frac": (prod_rate / imad_wide) if prod_rate else None,
                    "additions_per_step": entries / args.steps, "wide_products_per_addition": per_add,
                    # algorithmic count (8M + 2S); the kernel executes 2604: Y3 = R (Q - X3) - Y1 PPP shares one reduction
                    "wide_products_executed_per_addition": None if affine else 6 * 288 + 2 * 222 + 432,
                    "window_bits": ctx.get_stat("msm_window_bits"), "windows": ctx.get_stat("msm_windows"),
                    "table_levels": ctx.get_stat("msm_table_levels"),
                    "note": "per rank: additions_per_step counts the bucket additions THIS rank issued"}
    phases = {p: round(prof[p][0] / args.steps, 3) for p in PHASES}
    line = {
        "metric": METRIC, "value": ms_step, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32-limb Montgomery Fr/Fq (integer)", "data": "synthetic",
        "config": {"workload": "mulchain_prove_n=2^%d" % log_n, "gates": n - 3, "srs_points": n + 3,
                   "parallelism": ("msm bucket shard + quotient coset shard + row-sharded upload x%d, library-owned NCCL" % world)
                   if world > 1 else "single GPU", "l2": l2_flush, "setup_s": round(setup_s, 1)},
        "e2e": {"value": ms_e2e / args.steps, "unit": UNIT, "h2d_bytes_per_step": 3 * 32 * n + 32 * world,
                "inputs": "3 witness columns of n Fr + the 1-element public-input vector, pinned host memory"
                          + (" (each rank uploads its 1/%d row slice; slices exchanged over NVLink)" % world if world > 1 else ""),
                "d2h_bytes_per_step": 1472, "single_step_sample_ms": e2e_sample, "step_wall_ms": e2e_wall,
                "median_step_wall_ms": sorted(e2e_wall)[len(e2e_wall) // 2] if e2e_wall else None},
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": parity,
        "roofline": roofline,
        "roofline_int": roofline_int,
        "phases_ms_per_step": phases,
        "imad_peak_per_s": imad_wide,
        "proof_sha256": parity["sha256"][:16],
        "verify": verify,
        "standalone": standalone,
        "ab": ab or None,
        "north_star": None,
        "sweeps": None,
        "cpu_baseline": None,
        "b0_as_written": None,
    }

    # ---- BASELINE.json configs[4] / the north-star target: the 2^22-gate circuit on these N GPUs, bytes checked -------
    if not args.no_north_star and args.north_star_log_n != log_n:
        try:
            circuit.handle.destroy()
            circuit.srs.handle.destroy()
            del devt, host
            torch.cuda.empty_cache()
            lg = args.north_star_log_n
            big, bhost, bdev, bsetup = workload(lg)
            f_res = lambda: big.handle.prove_dev([t.data_ptr() for t in bdev[:3]], bdev[3].data_ptr())  # noqa: E731
            f_e2e = lambda: big.handle.prove_inputs([h.data_ptr() for h in bhost[:3]], host_pi.numpy())  # noqa: E731
            f_res()
            f_res()
            ctx.prof_reset()
            ctx.prof_enable(True)
            ns_steps = args.steps
            # every step timed on its own (barrier + events), so that a single stalled upload shows as an outlier in
            # `*_per_step` instead of silently inflating the mean
            res_ms, e2e_ms, pr, pr2 = [], [], None, None
            for _ in range(ns_steps):
                t_ms, pr = timed(f_res, 1)
                res_ms.append(round(t_ms, 3))
            ns_prof = ctx.prof_get()
            ctx.prof_enable(False)
            f_e2e()
            f_e2e()   # two warm-ups: the first sharded upload of a new size also sets up its NCCL transfers
            for _ in range(ns_steps):
                t_ms, pr2 = timed(f_e2e, 1)
                e2e_ms.append(round(t_ms, 3))
            ns_ab = []
            for spec in args.ab:
                opts = {k: int(v) for k, v in (kv.split("=") for kv in spec.split(","))}
                for k, v in opts.items():
                    ctx.set_option(k, v)
                f_res()
                t_ms, pr_ab = timed(f_res, ns_steps)
                for k in opts:
                    ctx.set_option(k, DEFAULTS.get(k, 0))
                ns_ab.append({"options": opts, "prove_ms": round(t_ms / ns_steps, 3), "same_bytes": pr_ab == pr})
            line["north_star"] = {"workload": "mulchain_prove_n=2^%d" % lg, "gates": (1 << lg) - 3, "n_gpus": world,
                                  "prove_ms": round(sum(res_ms) / ns_steps, 3), "e2e_ms": round(sum(e2e_ms) / ns_steps, 3),
                                  "prove_ms_per_step": res_ms, "e2e_ms_per_step": e2e_ms,
                                  "steps": ns_steps, "warmup": 2, "parity": _parity(pr, lg), "e2e_same_bytes": pr == pr2,
                                  "phases_ms_per_step": {p: round(ns_prof[p][0] / ns_steps, 3) for p in PHASES},
                                  "ab": ns_ab or None, "setup_s": round(bsetup, 1)}
            big.handle.destroy()
            big.srs.handle.destroy()
            del bdev, bhost
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            line["north_star"] = {"error": repr(e)}
            if world > 1:
                raise
    if world == 1 and not args.no_sweep:
        from typlonk_b200 import sweep
        line["sweeps"] = sweep.run(ctx, torch)
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        try:
            ms_cpu, done, threads, cproof = _cpu_prove(log_n, 1.0, 1)
            line["cpu_baseline"] = {
                "value": ms_cpu, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": "ONE full prove of the same 2^%d workload by oracle/c (C++ port of the reference prover with "
                          "Pippenger + NTTs), %d host threads; no extrapolation" % (log_n, threads),
                "same_bytes_as_gpu": cproof == proof}
            line["b0_as_written"] = _b0_as_written(log_n)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    if rank == 0:
        _dump(args, proof)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
