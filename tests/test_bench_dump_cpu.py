"""CPU: bench.py --dump-outputs' writer: arrays stored as float32 .npy as given, and above the size limit a fixed
seeded sample of rows (the same in every run) with their indices, within the limit."""
import os
import subprocess
import sys

import numpy as np

from helpers import ROOT

CODE = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import bench
bench.DUMP_LIMIT_BYTES = int(sys.argv[3])
rng = np.random.default_rng(5)
bench.dump_outputs(sys.argv[2], {"root_visits": rng.integers(0, 50, (4096, 20)).astype(np.float32),
                                 "root_values": rng.standard_normal(4096).astype(np.float32)})
"""


def _dump(path, limit):
    subprocess.run([sys.executable, "-c", CODE, ROOT, str(path), str(limit)], check=True)
    return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}, \
        sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def test_dump_outputs_writes_the_arrays_or_a_fixed_sample_within_the_limit(tmp_path):
    rng = np.random.default_rng(5)
    visits = rng.integers(0, 50, (4096, 20)).astype(np.float32)
    values = rng.standard_normal(4096).astype(np.float32)
    full, _ = _dump(tmp_path / "full", 64 << 20)
    assert sorted(full) == ["root_values", "root_visits"]
    assert full["root_visits"].dtype == np.float32 and np.array_equal(full["root_visits"], visits)
    assert np.array_equal(full["root_values"], values)
    limit = 100_000
    a, size_a = _dump(tmp_path / "a", limit)
    b, _ = _dump(tmp_path / "b", limit)
    assert size_a <= limit and sorted(a) == ["root_values", "root_visits", "rows"]
    rows = a["rows"].astype(np.int64)
    assert len(rows) > 0 and np.array_equal(a["root_visits"], visits[rows]) and np.array_equal(a["root_values"], values[rows])
    for k in a:
        assert np.array_equal(a[k], b[k]), k
