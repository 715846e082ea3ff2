# Lazy Fq arithmetic in the MSM (option msm_fq_lazy): card / power limit, two same-process A/B bench runs (lazy is the
# default; the second --ab puts lazy back for bench's 2^22 leg, which follows the first A/B's restore to 0), smoke,
# the GPU suite, and the 8-GPU A/B when the box has eight devices.  Usage: bash tools/gpu/run_fq_lazy.sh OUT_DIR
set -x
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/fq_lazy_card.csv
for i in 1 2; do
  timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --no-sweep --no-cpu-baseline \
    --ab msm_fq_lazy=0 --ab msm_fq_lazy=1 > $OUT/fq_lazy_bench_$i.json 2> $OUT/fq_lazy_bench_$i.err
  tail -2 $OUT/fq_lazy_bench_$i.err
  python - $OUT/fq_lazy_bench_$i.json <<'EOF'
import json, sys
d = json.loads(open(sys.argv[1]).read())
ph = d["phases_ms_per_step"]
print("2^20 lazy %.3f  digest_ok %s  accum %.3f reduce %.3f" % (d["value"], d["parity"].get("digest_ok"), ph["msm_accum"], ph["msm_reduce"]))
for a in d["ab"]:
    print("  ab", a["options"], a["prove_ms"], a["same_bytes"], "accum", a["phases_ms_per_step"]["msm_accum"], "reduce", a["phases_ms_per_step"]["msm_reduce"])
ns = d["north_star"] or {}
print("2^22 (after restore: canonical) %s parity %s" % (ns.get("prove_ms"), (ns.get("parity") or {}).get("digest_ok")))
for a in ns.get("ab") or []:
    print("  ab", a["options"], a["prove_ms"], a["same_bytes"])
EOF
done
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
( time timeout 1500 python -m pytest tests -m gpu -q -x --durations=8 ) > $OUT/fq_lazy_gpu_tests.log 2>&1
tail -20 $OUT/fq_lazy_gpu_tests.log
if [ "$(nvidia-smi -L | wc -l)" -ge 8 ]; then
  timeout 900 torchrun --nproc-per-node 8 bench.py --gpus 8 --steps 10 --warmup 3 --no-cpu-baseline --ab msm_fq_lazy=0 \
    > $OUT/fq_lazy_bench_n8.json 2> $OUT/fq_lazy_bench_n8.err
  tail -2 $OUT/fq_lazy_bench_n8.err
  python -c "import json, sys; d=json.load(open(sys.argv[1])); print('n8', d['value'], d['parity'], d['ab'])" $OUT/fq_lazy_bench_n8.json
fi
