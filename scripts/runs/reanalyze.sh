#!/bin/bash
# Reanalyze pipeline: its GPU tests, then scripts/exp_reanalyze.py (card + power limit in its output).
O=${OUT:-/tmp/reanalyze}; mkdir -p $O   # where the logs, the jsonl and the report go (OUT=dir to choose)
python -m hanabizero_b200.build > $O/build.log 2>&1; echo "build rc=$?"
timeout 1200 python -m pytest tests/test_reanalyze_pipeline_gpu.py -m gpu -q > $O/pytest_reanalyze.log 2>&1; echo "pytest reanalyze rc=$?"
grep -E "passed|failed|Error|assert" $O/pytest_reanalyze.log | tail -n 30
OUT=$O timeout 1200 python scripts/exp_reanalyze.py > $O/exp_reanalyze.log 2>&1; echo "exp_reanalyze rc=$?"
grep -v '^{' $O/exp_reanalyze.log | tail -n 40
