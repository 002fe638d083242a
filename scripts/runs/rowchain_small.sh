#!/bin/bash
# Hanabi-Small on the row-block executor: card + power limit, parity / stamps / stream timings (exp_rowchain.py NET=small),
# then the pipelined search (bench.py --config 1 --quick) at each "trees:in-flight" point of POINTS, library and rows
# alternated, REPS rounds.  --steps 400: a timed window of 0.1-0.5 s (20 steps is 7 ms at 512 trees).
O=${OUT:-/tmp/rowchain_small}; mkdir -p $O   # where the logs and bench lines go (OUT=dir to choose)
POINTS=${POINTS:-"512:8 512:20 1024:8 1024:20 4096:8 4096:20"}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv | tee $O/card.csv
if [ -z "$NO_EXP" ]; then
  NET=small N=4096 D=8 timeout 300 python scripts/exp_rowchain.py > $O/exp_small.log 2>&1; echo "exp small rc=$?"
  grep -v "max|rows" $O/exp_small.log | tail -n 24
fi
show() { python - "$1" "$2" <<'P'
import json, sys
try:
    d = json.load(open(sys.argv[1]))
    print("%s: value %.2fM in-flight %s executor %s window %.0f ms" % (sys.argv[2], d["value"] / 1e6, d["setup"]["searches_in_flight"], d["setup"].get("network_executor"), d["ms_per_step"] * d["steps"]))
except Exception as e:
    print("no bench line", sys.argv[1], e)
P
}
for rep in $(seq 1 ${REPS:-1}); do
  for pt in $POINTS; do
    trees=${pt%:*}; fl=${pt#*:}
    for ex in library rows; do
      f=$O/bench_c1_${trees}_${fl}_${ex}_r${rep}
      timeout 300 python bench.py --config 1 --trees $trees --in-flight $fl --executor $ex --steps 400 --warmup 20 --quick --no-cpu-baseline > $f.json 2> $f.err
      echo "rc=$?"; show $f.json "c1 $trees x $fl $ex r$rep"
    done
  done
done
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a $O/card.csv
