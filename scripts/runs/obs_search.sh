#!/bin/bash
# Observation tickets: their GPU tests, then scripts/exp_obs_search.py (card + power limit in its output).
O=${OUT:-/tmp/obs_search}; mkdir -p $O   # where the logs, the jsonl and the report go (OUT=dir to choose)
python -m hanabizero_b200.build > $O/build.log 2>&1; echo "build rc=$?"
timeout 1200 python -m pytest tests/test_search_obs_gpu.py -m gpu -q > $O/pytest_obs.log 2>&1; echo "pytest obs rc=$?"
grep -E "passed|failed|Error|assert" $O/pytest_obs.log | tail -n 30
OUT=$O timeout 900 python scripts/exp_obs_search.py > $O/exp_obs_search.log 2>&1; echo "exp_obs_search rc=$?"
grep -v '^{' $O/exp_obs_search.log | tail -n 40
