#!/bin/bash
# Search waves against one search per ticket (scripts/exp_wave.py): card + power limit, then (a) wave=1 depth=20 and
# (b) wave=4096/n depth=8 alternated at n = 512, 1024, 2048, pinned-host and Hanabi-Small points, and a torch.profiler
# trace of each at n = 512.  Everything lands in $OUT.
O=${OUT:-/tmp/wave}; mkdir -p $O   # where the log, the jsonl and the trace go (OUT=dir to choose)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/card.csv
OUT=$O timeout 1500 python scripts/exp_wave.py > $O/exp_wave.log 2>&1; echo "exp_wave rc=$?"
grep -v '^{' $O/exp_wave.log | head -n 80
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee -a $O/card.csv
