#!/bin/bash
# Recorded self-play on the byte frame ring: its GPU tests, then scripts/exp_selfplay_record.py (card + power limit in its output).
O=${OUT:-/tmp/selfplay_record}; mkdir -p $O   # where the logs, the jsonl and the report go (OUT=dir to choose)
python -m hanabizero_b200.build > $O/build.log 2>&1; echo "build rc=$?"
timeout 1500 python -m pytest tests/test_selfplay_record_gpu.py -m gpu -q > $O/pytest_record.log 2>&1; echo "pytest record rc=$?"
grep -E "passed|failed|Error|assert" $O/pytest_record.log | tail -n 30
OUT=$O timeout 1500 python scripts/exp_selfplay_record.py > $O/r05_selfplay_record_exp.log 2>&1; echo "exp_selfplay_record rc=$?"
grep -v '^{' $O/r05_selfplay_record_exp.log | tail -n 40
