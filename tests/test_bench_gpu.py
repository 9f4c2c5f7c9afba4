"""bench.py on the GPU: --steps is the number of timed steps and --dump-outputs writes what the last of them returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_holds_the_results_of_the_timed_step(tmp_path):
    import bench
    from oracle import qagnn_oracle as O
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=1200,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    B, n, D = bench.CFG["graphs"], bench.CFG["n"], bench.CFG["D"]
    assert sorted(os.listdir(tmp_path)) == ["gnn_out.npy", "logits.npy", "pool_attn.npy"]
    got = {name: np.load(tmp_path / f"{name}.npy") for name in ("logits", "pool_attn", "gnn_out")}
    assert got["logits"].shape == (B, 1) and got["pool_attn"].shape == (2 * B, n) and got["gnn_out"].shape == (B, n, D)
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_LIMIT
    # the node output is the message passing of the benchmark's seeded batch: its first graphs against the CPU oracle
    inp = bench.synth_step_inputs(0)
    sd = O.random_state_dict(bench.CFG["k"], D, bench.CFG["T"], bench.CFG["R"], "prod", seed=0)
    ref = bench.oracle_slice(inp, sd, 0, 2).numpy()
    assert (np.abs(got["gnn_out"][:2] - ref) <= 1e-4 + 1e-4 * np.abs(ref)).all()
