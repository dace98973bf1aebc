"""bench.py --dump-outputs: what the last timed step returned, as float32 / float64 .npy files, the same from run to run
with the same arguments, and changed by --steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "hmc_iso_gaussian_1024x100_L10", "--steps", str(steps),
           "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == steps
    return {f.name: np.load(f) for f in out_dir.glob("*.npy")}


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_bit_for_bit(tmp_path):
    a, b, c = _bench_dump(tmp_path / "a", 2), _bench_dump(tmp_path / "b", 2), _bench_dump(tmp_path / "c", 3)
    assert {"position.npy", "logdensity.npy", "logdensity_grad.npy", "acceptance_rate.npy", "is_accepted.npy",
            "energy.npy", "chain_index.npy"} <= set(a)
    assert set(a) == set(b) == set(c)
    assert a["position.npy"].shape == (1024, 100)             # all chains of this workload fit the size cap
    assert sum(os.path.getsize(f) for f in (tmp_path / "a").glob("*.npy")) <= 64 * 10 ** 6
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["position.npy"], c["position.npy"])   # one more timed step, other draws
