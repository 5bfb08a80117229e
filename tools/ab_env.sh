#!/bin/bash
# A/B of environment switches on the SAME box: per-kernel times of one configs[2] step (TIK_PLAN_TRACE) and the
# bench value, alternating the settings, three rounds each.
#   tools/ab_env.sh "TIK_SERPENTINE=0" "TIK_SERPENTINE=1" ...
mkdir -p gpurun_out
for r in 1 2 3; do
  for setting in "$@"; do
    env $setting TIK_PLAN_TRACE=1 timeout 200 python bench.py --steps 2 --warmup 3 --no-cpu --no-hbm --no-c3 2>&1 >/dev/null | grep "tik trace" | tail -17 |
      awk -v w="$setting" -v r=$r '{printf "%s ", $(NF-1); s+=$(NF-1)} END {printf " | sum %.1f us  [%s] round %s\n", s, w, r}'
    env $setting timeout 200 python bench.py --steps 20 --warmup 5 --no-cpu --no-hbm --no-c3 2>/dev/null |
      python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('   bench', round(d['value']/1e6,2), 'M frames/s', d['ms_per_step_min_median_max_rank0'], d['clocks']['sm_mhz'])"
  done
done 2>&1 | tee gpurun_out/ab_env.log
