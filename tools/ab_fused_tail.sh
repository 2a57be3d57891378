#!/bin/bash
# Merged ModDown + Rescale tail (default) against the two-pass tail (LGPU_FZ_RESCALE=0) on the headline step: card and power limit, the GPU
# suite, smoke, identical --dump-outputs for both settings, then bench.py alternated between the two settings (3 runs each) and one
# bootstrap run each (3 timed steps: two-step runs can stall on the host at the start of the first one).
# Usage: tools/ab_fused_tail.sh OUTDIR -- logs, bench JSON lines and the A/B table land in OUTDIR/fz_*.
O=${1:?usage: $0 OUTDIR}
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/fz_card.txt
python -m pytest tests -q -m gpu > $O/fz_pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $O/fz_pytest_gpu.log; tail -3 $O/fz_pytest_gpu.log
python __graft_entry__.py smoke > $O/fz_smoke.log 2>&1; echo "smoke rc=$?"
for v in 1 0; do
  LGPU_FZ_RESCALE=$v timeout 600 python bench.py --steps 2 --warmup 1 --no-e2e --no-cpu-baseline --dump-outputs $O/fz_dump_$v > /dev/null 2> $O/fz_dump_$v.err
done
if diff -r -q $O/fz_dump_1 $O/fz_dump_0; then echo "dump-outputs identical"; else echo "dump-outputs DIFFER"; fi
rm -rf $O/fz_dump_1 $O/fz_dump_0
for run in 1 2 3; do
  for v in 1 0; do
    LGPU_FZ_RESCALE=$v timeout 600 python bench.py --steps 5 --warmup 3 > $O/fz_bench_${v}_$run.json 2> $O/fz_bench_${v}_$run.err
    python - "$O/fz_bench_${v}_$run.json" "LGPU_FZ_RESCALE=$v run $run" <<'EOF'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
c = d["roofline"]["classes"]
print(sys.argv[2], "ct/s", round(d["value"], 1), "ms/step", round(d["ms_per_step"], 3),
      {k: round(c[k]["ms"], 2) for k in ("fused", "epilogue", "ntt_inv") if k in c}, "e2e.matches_device_path", d.get("e2e", {}).get("matches_device_path"))
EOF
  done
done | tee $O/fz_ab.txt
for v in 1 0; do
  LGPU_FZ_RESCALE=$v timeout 600 python bench.py --workload bootstrap --preset BOOT_N16QP1767 --batch 64 --steps 3 --warmup 1 > $O/fz_boot_$v.json 2>/dev/null
  python -c "
import json
d=json.loads(open('$O/fz_boot_$v.json').read().strip().splitlines()[-1]); print('bootstrap LGPU_FZ_RESCALE=$v', round(d['value'],2), round(d['ms_per_step'],1), d.get('phase_ms_per_step'))"
done | tee -a $O/fz_ab.txt
