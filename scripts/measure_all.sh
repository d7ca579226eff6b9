#!/usr/bin/env bash
# One GPU: every single-GPU bench line of profiles/ plus the ncu launch list and the --set full capture of one pass.
# Usage (on the GPU box, from the repo root): bash scripts/measure_all.sh [tag]      -> gpurun_out/
tag=${1:-r02_v3}
out=gpurun_out
mkdir -p $out
python bench.py --workload cm --steps 200 > $out/bench_r02_cm.json 2> $out/cm.err
python bench.py --workload pass --steps 30 --warmup 5 > $out/bench_r02_pass_n1.json 2> $out/pass.err
python bench.py --workload market --steps 30 --warmup 5 > $out/bench_r02_market_n1.json 2> $out/market.err
python bench.py --workload hard --steps 30 --warmup 5 > $out/bench_r02_hard_n1.json 2> $out/hard.err
python bench.py --workload scale100k --steps 10 --warmup 3 --no-e2e > $out/bench_r02_scale100k_n1.json 2> $out/s100.err
# ncu only after the same command has run plain and exited 0
if python scripts/prof_pass.py 32621 1041 3 > $out/plain_$tag.log 2>&1; then
  ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
      --log-file $out/${tag}_launches.csv python scripts/prof_pass.py 32621 1041 3 > $out/ncu_l_$tag.log 2>&1
  ncu --profile-from-start off --set full --clock-control none --import-source on -o $out/prof_$tag -f \
      python scripts/prof_pass.py 32621 1041 1 > $out/ncu_f_$tag.log 2>&1
fi
for f in cm pass_n1 market_n1 hard_n1 scale100k_n1; do
  python -c "
import json; d=json.loads(open('$out/bench_r02_$f.json').read().strip().splitlines()[-1])
print('$f', d['ms_per_step'], (d.get('e2e') or {}).get('value'), d.get('stage_ms'))"
done
