"""bench.py --dump-outputs: what the timed Q1 path returned in its last step, one float64 array per result column, equals
the oracle's Q1 over the same generated lineitem, and the JSON line reports the number of timed steps asked for."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    import bench
    from datagen import tpch
    from sail_b200 import plans
    from tests.util import oracle_op
    got_dir, want_dir = tmp_path / "got", tmp_path / "want"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--sf", "0.01", "--chunk-sf", "0.01", "--steps", "2", "--warmup", "1",
                        "--skip-cpu", "--skip-e2e", "--skip-joins", "--skip-suites", "--dump-outputs", str(got_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    want = plans.execute(plans.q1(), {"lineitem": tpch.lineitem(0.01, bench.Q1_COLS)}, oracle_op)
    bench.dump_outputs(want, str(want_dir))
    assert sorted(os.listdir(got_dir)) == sorted(f"{n}.npy" for n in want.column_names)
    for name in want.column_names:
        g, w = np.load(got_dir / f"{name}.npy"), np.load(want_dir / f"{name}.npy")
        assert g.dtype == np.float64 and np.array_equal(g, w), (name, g, w)
