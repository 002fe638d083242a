#!/bin/bash
# the whole GPU-marked suite, the smoke entry and one bench line
O=${OUT:-/tmp/r04_final}; mkdir -p $O   # where the logs and the bench line go (OUT=dir to choose)
python -c "import __graft_entry__ as g; g.build()" > $O/build.log 2>&1; echo "build rc=$?"
timeout 2400 python -m pytest tests -m gpu -q > $O/pytest.log 2>&1; echo "pytest rc=$?"; grep -E "passed|failed" $O/pytest.log | tail -n 20
timeout 600 python __graft_entry__.py --smoke > $O/smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/smoke.log
timeout 1200 python bench.py --gpus 1 --steps 20 --warmup 5 > $O/bench.json 2> $O/bench.err; echo "bench rc=$?"
python -c "
import json; d=json.loads(open('$O/bench.json').read().strip().splitlines()[-1])
print('value %.2fM' % (d['value']/1e6), 'e2e %.2fM' % (d['e2e']['value']/1e6))"
