#!/bin/bash
# A/B runs of the B=256 humanoid-9 update under environment settings: bash tools/ab_update.sh "NAME=VAL ..." "..." (one quoted group per run)
# prints ms/step (device-timed) and end-to-end samples/s per run.  usage (GPU box), two builds alternated:
#   bash tools/ab_update.sh "" "SGRL_LIB=/path/to/other/libsgrl_b200.so" "" "SGRL_LIB=/path/to/other/libsgrl_b200.so"
cd "$(dirname "$0")/.."
for envs in "$@"; do
  out=$(env $envs timeout 300 python bench.py --steps ${AB_STEPS:-60} --warmup 6 --no-cpu-baseline --no-rollout --no-bf16 2>/dev/null | tail -1)
  echo "$out" | python -c "
import sys, json
d = json.loads(sys.stdin.read())
print('%-60s ms/step %.3f  e2e %.0f  launches %.1f' % ('''$envs''' or '(default)', d['ms_per_step'], d['e2e']['value'], d['gpu_launches']))" 2>&1 | tail -1
done
