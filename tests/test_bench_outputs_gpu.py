"""-m gpu: bench.py --dump-outputs writes what the timed path decoded in its last step, and those arrays equal the CPU
oracle's decode of the same seeded inputs."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from draco_sharp_b200.decoder import NP_DTYPES
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_equal_the_oracle(tmp_path):
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "3", "--warmup", "1",
                        "--e2e-steps", "0", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
    files = sorted(os.listdir(out))
    assert files and sum(os.path.getsize(out / f) for f in files) <= 64 << 20
    import bench
    arena, offs, lens, _, _, _ = bench.make_workload("tiny", 0, 2048)
    decoded = {}
    for f in files:
        k, a = map(int, re.fullmatch(r"buf(\d+)_attr(\d+)\.npy", f).groups())
        got = np.load(out / f)
        assert got.dtype in (np.float32, np.float64)
        if k not in decoded:
            decoded[k] = O.decode(arena[int(offs[k]): int(offs[k] + lens[k])])
        oa = decoded[k].attrs[a]
        want = oa.out.view(NP_DTYPES[oa.data_type]).reshape(oa.n_entries, oa.nc)
        assert got.shape == want.shape and np.array_equal(got, want.astype(got.dtype)), f
