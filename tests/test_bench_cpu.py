"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-graphs", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_traffic_artefact_belongs_to_the_current_kernel_source():
    """bench.py reports roofline.traffic only from profiles/mp_traffic.json and only while its sha matches mp_headtile.cu:
    the committed artefact must be the capture of the committed kernel (else the field silently becomes null)."""
    import bench
    sha = bench.mp_kernel_sha()
    traffic = bench.mp_traffic_from_profile(sha)
    assert traffic is not None and 150e6 < traffic < 260e6, "re-capture profiles/mp_traffic.json after changing mp_headtile.cu"
    assert bench.mp_traffic_from_profile("0" * 16) is None


def test_oracle_slice_equals_the_full_batch_rows():
    """The parity gate of bench.py evaluates the oracle on a slice of the batch; sub-graphs are independent, so the slice must
    reproduce the corresponding rows of a full-batch oracle run (small shape)."""
    import bench
    from oracle import qagnn_oracle as O
    saved = dict(bench.CFG)
    try:
        bench.CFG.update(graphs=6, n=20, e=40, D=16, k=2, H=4)
        inp = O.synth_graph_batch(6, 20, 40, 16, bench.CFG["R"], seed=1)
        sd = O.random_state_dict(2, 16, bench.CFG["T"], bench.CFG["R"], "peaky", seed=1)
        full = O.message_passing_forward(sd, inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"], 2,
                                         bench.CFG["T"], bench.CFG["R"], 4)
        part = bench.oracle_slice(inp, sd, 2, 3)
        assert torch.allclose(part, full[2:5], atol=1e-6, rtol=1e-6)
    finally:
        bench.CFG.clear(); bench.CFG.update(saved)


def _bench_lines(path):
    import json
    return [json.loads(l) for l in open(path) if l.strip().startswith("{")]


@pytest.mark.parametrize("name", ["r2_final_bench.json", "r2_bench_n2.json", "r2_bench_n4.json", "r2_bench_n8.json"])
def test_committed_bench_lines_are_self_consistent(name):
    """The arithmetic a reader redoes on a bench line (DESIGN.md §6): throughput from ms_per_step, roofline from B_alg."""
    path = os.path.join(ROOT, "profiles", name)
    lines = _bench_lines(path)
    assert lines, path
    d = lines[-1]
    k, D = 5, 200
    N, E, G = d["config"]["N"], d["config"]["E"], d["n_gpus"]
    assert d["metric"] == "GNN edges/sec" and d["scaling"] == "weak" and d["dtype"] == "f32" and d["vs_baseline"] is None
    assert d["value"] == pytest.approx(G * k * E / (d["ms_per_step"] * 1e-3), rel=1e-6)
    assert d["e2e"]["value"] == pytest.approx(G * k * E / (d["e2e"]["ms_per_step"] * 1e-3), rel=1e-6)
    assert d["e2e"]["value"] < d["value"] and d["e2e"]["h2d_bytes_per_step"] > 8 * 2 * E and d["e2e"]["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["algorithmic_bytes_per_launch"] == 16 * N * D + 24 * E + 8 * N == 212992000     # SURVEY.md §8d
    assert r["achieved"] == pytest.approx(r["algorithmic_bytes_per_launch"] / (r["avg_launch_ms"] * 1e-3) / 1e9, rel=1e-6)
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-9) and r["bound"] == "hbm"
    assert r["traffic"] is None or 0.5 * r["algorithmic_bytes_per_launch"] < r["traffic"] < 1.5 * r["algorithmic_bytes_per_launch"]
    assert k * r["avg_launch_ms"] < d["ms_per_step"]                                        # the kernel fits k times in the step
    st = d["stages"]
    assert st["message_passing"]["ms_per_step"] == pytest.approx(k * r["avg_launch_ms"], rel=1e-3)
    assert sum(s["ms_per_step"] for s in st.values()) < d["ms_per_step_per_kernel_launches"]
    gm = d["roofline_gemm"]
    assert gm["frac"] == pytest.approx(gm["achieved"] / gm["peak"], rel=1e-9)
    if "flops_per_launch" in gm:  # the 8-GPU line predates this key
        assert gm["flops_per_launch"] == 3 * 2 * N * (D + D // 2) * 624                      # three bf16 passes, padded 3*H*DP columns
        assert gm["achieved"] == pytest.approx(gm["flops_per_launch"] / (gm["avg_launch_ms"] * 1e-3) / 1e12, rel=1e-6)
    assert d["gpu_launches"] > 0 and d["parity_gate"]["max_abs_err"] < 1e-4
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if G > 1:
        assert d["parity_gate"]["multi_rank_logits_vs_single_gpu_max_abs_err"] < 1e-5


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bad_arguments_are_refused(extra):
    """--steps is the number of timed steps (at least one); --dump-outputs belongs to the CUDA arm, whose inputs are seeded."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                         cwd=ROOT)
    assert out.returncode == 2 and "error:" in out.stderr
    assert not os.path.exists(os.path.join(ROOT, "unused"))


def test_dump_outputs_writes_float32_npy_within_the_limit(tmp_path):
    import numpy as np
    import bench
    bench.dump_outputs(str(tmp_path / "d"), {"a": np.arange(6.0).reshape(2, 3)})
    got = np.load(tmp_path / "d" / "a.npy")
    assert got.dtype == np.float32 and got.tolist() == [[0, 1, 2], [3, 4, 5]]
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "e"), {"big": np.zeros(bench.DUMP_LIMIT // 4 + 1, np.float32)})
    assert not (tmp_path / "e").exists()
