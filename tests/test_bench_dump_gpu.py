"""bench.py --dump-outputs: the file holds what the timed path returned, for the seeded inputs bench.py times."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import c_oracle, cspn_numpy as onp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    import bench
    from cspn_b200.synth import make_inputs
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '0', '--e2e-steps', '1',
           '--no-other-configs', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)]
    lines = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(lines) == 1 and json.loads(lines[0])['steps'] == 2
    assert os.listdir(tmp_path) == ['out.npy']
    out = np.load(tmp_path / 'out.npy')
    assert out.shape == (bench.B_PER_GPU, 1, bench.H, bench.W) and out.dtype == np.float32
    g, d, s = make_inputs(0, bench.B_PER_GPU, 1, bench.H, bench.W)      # rank 0's inputs; the oracle checks the first image
    ref = c_oracle.cspn2d(g[:1].numpy(), d[:1].numpy(), s[:1].numpy(), bench.ITERS, bench.NORM)
    ok, ratio, normwise = onp.parity_ok(out[:1], ref, 1e-4)
    assert ok, (ratio, normwise)
