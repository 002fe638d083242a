#!/bin/bash
# Episode store: its GPU tests, then scripts/exp_reanalyze_store.py (card + power limit in its output).
O=${OUT:-/tmp/reanalyze_store}; mkdir -p $O   # where the logs, the jsonl and the report go (OUT=dir to choose)
python -m hanabizero_b200.build > $O/build.log 2>&1; echo "build rc=$?"
timeout 1200 python -m pytest tests/test_episode_store_gpu.py -m gpu -q > $O/pytest_episode_store.log 2>&1; echo "pytest episode store rc=$?"
grep -E "passed|failed|Error|assert" $O/pytest_episode_store.log | tail -n 30
OUT=$O timeout 1200 python scripts/exp_reanalyze_store.py > $O/exp_reanalyze_store.log 2>&1; echo "exp_reanalyze_store rc=$?"
grep -v '^{' $O/exp_reanalyze_store.log | tail -n 40
