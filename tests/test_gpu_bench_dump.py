"""GPU tier: bench.py --steps K times K steps, and --dump-outputs writes a sample of the pairings the last timed step
computed, which the C oracle recomputes from bench.py's seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import bn254_py as o
from oracle import c_oracle as c
from tests import wire as w

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_pairings(tmp_path):
    log2n, steps = 16, 2  # 2^16 > the 2^15 dumped rows, so the dump is a sample
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                          "--warmup", "1", "--log2n", str(log2n), "--verify-log2n", "0", "--extras", "0",
                          "--cpu-seconds", "0.2", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == steps
    n = 1 << log2n
    gt = np.load(tmp_path / "pairing_batch.npy")
    rows = np.load(tmp_path / "pairing_batch_rows.npy")
    assert gt.dtype == rows.dtype == np.float64
    assert gt.shape == (1 << 15, 12, 8) and rows.shape == (1 << 15,)
    idx = rows.astype(np.int64)
    assert (idx == rows).all() and (np.diff(idx) > 0).all() and 0 <= idx[0] and idx[-1] < n

    # bench.py's inputs: P_i = a_i G1gen, Q_i = b_i G2gen, a then b drawn from RandomState(1), top byte masked
    rs = np.random.RandomState(1)
    a = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 31] &= 0x1F
    b = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    b[:, 31] &= 0x1F
    sel = np.linspace(0, len(idx) - 1, 256).astype(np.int64)
    m = len(sel)
    p, _ = c.g1_mul_batch(np.tile(np.frombuffer(w.g1_b(o.G1_GEN), np.uint8), (m, 1)), a[idx[sel]])
    q, _ = c.g2_mul_batch(np.tile(np.frombuffer(w.g2_b(o.G2_GEN), np.uint8), (m, 1)), b[idx[sel]])
    exp = c.pairing_batch(p, q).view("<u4").reshape(m, 12, 8)
    assert (gt[sel] == exp).all()
