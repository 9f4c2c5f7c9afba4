#!/usr/bin/env python
"""bench.py — the QA-GNN message-passing hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores
    python bench.py --gpus 1 --steps K --dump-outputs bench_outputs  # + the last timed step's results as .npy files

One "step" = one QAGNN_Message_Passing.forward (k=5 GATConvE layers, modeling_qagnn.py:53-95) over one
synthetic batch of BASELINE.json configs[1]: 64x5 = 320 sub-graphs of 200 nodes / 1000 edges per GPU,
hidden 200, 4 heads, 38 relation types.  Metric: GNN edges/sec = k * E / t ("edge-layers per second",
E = real directed edges, self loops excluded; SURVEY.md §8d).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(graphs=320, n=200, e=1000, D=200, k=5, H=4, T=4, R=38)
SENT_DIM = 1024  # RoBERTa-large sentence vector (modeling_encoder.py)
METRIC = "GNN edges/sec"
UNIT = "edge-layers/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample-graphs", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true", help="launch the ~60 kernels of a step one by one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (logits, pool_attn, gnn_out of "
                         "rank 0) as DIR/<name>.npy in float32; the inputs are seeded, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm times a sample sized to the host)")
    return args


DUMP_LIMIT = 64 << 20  # bytes, all dumped arrays together


def dump_outputs(dirname, arrays):
    """Writes {name: float32 ndarray} as dirname/<name>.npy."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: the outputs take {total} bytes, more than the {DUMP_LIMIT} of --dump-outputs")
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def workload_name():
    return (f"cfg2: {CFG['graphs']} graphs/GPU (64x5 choices) x {CFG['n']} nodes x {CFG['e']} edges, hidden {CFG['D']}, "
            f"{CFG['k']} layers, {CFG['H']} heads, {CFG['R']} edge types (17 merged relations -> (17+2)*2)")


def b_alg_per_layer(N, E, D):
    """SURVEY.md §8d: compulsory bytes of the message-passing kernel per layer (read Q,Kx,Mx + write aggr,
    int64 src/tgt/etype, int64 node_type)."""
    return 16 * N * D + 24 * E + 8 * N


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm (oracle/qagnn_oracle.py), all host threads
# ------------------------------------------------------------------------------------------------
CPU_THREADS = 32  # pinned intra-op pool of the CPU arm (torch's pool degrades when oversubscribed on many-core hosts;
#                   16-32 threads were the fastest sizes of every probe on the 128-cpu GPU boxes, round 1 and 2)


def cpu_reference_run(steps, warmup, sample_graphs, seed=0, budget_s=None, full_batch_once=False):
    """Times the CPU restatement on `sample_graphs` graphs of the workload with a PINNED thread-pool size.  With `budget_s`
    the sample is shrunk (never below 4 graphs) so that warmup+steps forwards fit the budget; steps and warmup are always
    honoured.  full_batch_once: additionally one timed forward over all 320 graphs of the workload."""
    from oracle import qagnn_oracle as O
    ncpu = os.cpu_count() or 1
    cores = min(CPU_THREADS, ncpu)
    torch.set_num_threads(cores)
    sd = O.random_state_dict(CFG["k"], CFG["D"], CFG["T"], CFG["R"], "prod", seed)
    probe = O.synth_graph_batch(8, CFG["n"], CFG["e"], CFG["D"], CFG["R"], seed)

    def fwd(inp, k):
        return O.message_passing_forward(sd, inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"], k,
                                         CFG["T"], CFG["R"], CFG["H"])
    fwd(probe, 1)  # warms the pool and the allocator
    t0 = time.perf_counter()
    fwd(probe, 1)
    per_graph = (time.perf_counter() - t0) / 8 * CFG["k"]  # seconds per graph and forward
    if budget_s is not None:
        sample_graphs = int(max(4, min(sample_graphs, budget_s / ((steps + warmup) * per_graph))))
    inp = O.synth_graph_batch(sample_graphs, CFG["n"], CFG["e"], CFG["D"], CFG["R"], seed)
    E = inp["edge_index"].size(1)
    for _ in range(warmup):
        fwd(inp, CFG["k"])
    t0 = time.perf_counter()
    for _ in range(steps):
        fwd(inp, CFG["k"])
    dt = (time.perf_counter() - t0) / steps
    res = {"value": CFG["k"] * E / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{sample_graphs} of the {CFG['graphs']} graphs of the workload ({E} edges), {steps} timed "
                     f"forwards of the op-for-op oracle port (torch CPU fp32, {cores} threads pinned, {ncpu}-cpu host), "
                     f"{dt * 1e3:.1f} ms each",
           "ms_per_step": dt * 1e3}
    if full_batch_once:
        full = O.synth_graph_batch(CFG["graphs"], CFG["n"], CFG["e"], CFG["D"], CFG["R"], seed)
        t0 = time.perf_counter()
        fwd(full, CFG["k"])
        dtf = time.perf_counter() - t0
        Ef = full["edge_index"].size(1)
        res["full_batch"] = {"value": CFG["k"] * Ef / dtf, "unit": UNIT, "ms": dtf * 1e3,
                             "sample": f"all {CFG['graphs']} graphs ({Ef} edges), one timed forward, {cores} threads"}
    return res


def oracle_slice(inp, sd, g0, count):
    """CPU oracle output for graphs [g0, g0+count) of a workload batch (sub-graphs are independent)."""
    from oracle import qagnn_oracle as O
    n = CFG["n"]
    ei, et = inp["edge_index"], inp["edge_type"]
    sel = (ei[0] >= g0 * n) & (ei[0] < (g0 + count) * n)
    return O.message_passing_forward(sd, inp["H"][g0:g0 + count], ei[:, sel] - g0 * n, et[sel], inp["node_type"][g0:g0 + count],
                                     inp["node_score"][g0:g0 + count], CFG["k"], CFG["T"], CFG["R"], CFG["H"])


def gemm_roofline(N, D, H, avg_launch_ms, peaks):
    """Tensor roofline of the projection GEMM as the forward runs it since round 2: [N, D + D/2] x [D + D/2, 3*H*DP]
    ([x | score_emb] against the head-major padded Q|Kx|Mx weights; the type-embedding half of node_feature_extra is a
    per-type bias row), three bf16 passes (hi*hi, hi*lo, lo*hi) per launch."""
    peak = peaks.get("bf16_tflops", 1590.0)
    K = D + D // 2
    ncols = 3 * H * ((D // H + 3) // 4 * 4)
    flops = 3 * 2 * N * K * ncols
    achieved = flops / (avg_launch_ms * 1e-3) / 1e12 if avg_launch_ms > 0 else 0.0
    return {"kernel": "gemm_tc_kernel (projection Q|Kx|Mx, K = D + D/2)", "bound": "tensor", "achieved": achieved, "peak": peak,
            "unit": "TFLOP/s", "frac": achieved / peak, "avg_launch_ms": avg_launch_ms, "flops_per_launch": flops,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if "bf16_tflops" in peaks else "fallback 1590 TFLOP/s"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    r = cpu_reference_run(steps, warm, args.cpu_sample_graphs, budget_s=100.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(), "bounded_sample": r["sample"]},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's torch-geometric/torch-scatter wheels cannot be installed offline; this arm times the "
                "op-for-op CPU restatement of the reference path (oracle/), pinned against goldens minted from the "
                "reference's own modules",
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()  # exact child we started
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower() == "active" for r in self.rows)]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def mp_traffic_from_profile(kernel_sha):
    """dram bytes (read + write) of one mp_headtile launch from the committed ncu artefact that was captured with the SAME
    kernel source (profiles/mp_traffic.json: {"mp_headtile_sha16": ..., "dram_bytes": ...}); None when the artefact is
    missing or belongs to another version of the kernel — never a hard-coded literal."""
    try:
        art = json.load(open(os.path.join(ROOT, "profiles", "mp_traffic.json")))
        return art["dram_bytes"] if art.get("mp_headtile_sha16") == kernel_sha else None
    except Exception:  # noqa: BLE001
        return None


def mp_kernel_sha():
    import hashlib
    return hashlib.sha256(open(os.path.join(ROOT, "qagnn_b200", "csrc", "mp_headtile.cu"), "rb").read()).hexdigest()[:16]


def build_decoder_tail(D, sent_dim, dev):
    """The pooling layer and answer MLP of the QAGNN decoder around the message passing (modeling_qagnn.py:121-125 with the
    scripts' defaults: 2 pooling heads, fc_layer_num 0 -> one Linear(2D+sent_dim -> 1); random init, seed 1)."""
    from qagnn_b200.layers import MLP, MultiheadAttPoolLayer
    torch.manual_seed(1)
    pooler = MultiheadAttPoolLayer(2, sent_dim, D).eval().to(dev)
    fc = MLP(D + sent_dim + D, D, 1, 0, 0.2, layer_norm=True).eval().to(dev)
    return pooler, fc


def synth_step_inputs(rank):
    """One rank's shard of the workload: the cfg2 graph batch + sentence vectors and graph sizes for the pooling tail."""
    from oracle import qagnn_oracle as O  # input generator only (shared with the tests)
    B, n, e, D = CFG["graphs"], CFG["n"], CFG["e"], CFG["D"]
    inp = O.synth_graph_batch(B, n, e, D, CFG["R"], seed=100 + rank)
    g = torch.Generator().manual_seed(7000 + rank)
    inp["sent_vecs"] = torch.randn(B, SENT_DIM, generator=g) * 0.5
    if "adj_lengths" not in inp or inp["adj_lengths"] is None:
        inp["adj_lengths"] = torch.full((B,), n, dtype=torch.long)
    # the batch is packed graph by graph, as LM_QAGNN.batch_graph / qagnn_b200.data.PackedAdjBatchGenerator deliver it
    cnt = torch.bincount(inp["edge_index"][0] // n, minlength=B)
    inp["graph_ptr"] = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(cnt, 0)])
    return inp


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import torch.distributed as dist
    import qagnn_b200
    from qagnn_b200 import _lib
    from qagnn_b200 import distributed as QD
    from qagnn_b200.pipeline import DecoderStep, StreamedRunner
    from oracle import qagnn_oracle as O  # weights generator + the parity gate below; never inside a timed region

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = QD.bind_to_gpu_numa_node(local)  # before any pinned allocation: first touch lands on the GPU's node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    B, n, e, D, k = CFG["graphs"], CFG["n"], CFG["e"], CFG["D"], CFG["k"]
    inp = synth_step_inputs(rank)
    sd = O.random_state_dict(k, D, CFG["T"], CFG["R"], "prod", seed=0)
    mod = qagnn_b200.QAGNN_Message_Passing(None, k, CFG["T"], CFG["R"], D, D, D).eval()
    mod.load_state_dict(sd)
    mod = mod.to(dev)
    pooler, fc = build_decoder_tail(D, SENT_DIM, dev)
    N, E = B * n, inp["edge_index"].size(1)

    host = {k_: inp[k_].pin_memory() for k_ in DecoderStep.PACKED_FIELDS}
    max_edges = int((inp["graph_ptr"][1:] - inp["graph_ptr"][:-1]).max())
    d = {k_: v.to(dev, non_blocking=True) for k_, v in host.items()}
    torch.cuda.synchronize()

    # parity gate: what is about to be timed must match the CPU oracle (first and last 4 graphs of this rank's batch)
    # within the 1e-4 bar, otherwise the run aborts before any number is produced
    first = mod(d["H"], (d["edge_index"], d["edge_type"]), d["node_type"], d["node_score"]).cpu()
    parity_err = 0.0
    for g0 in (0, B - 4):
        ref = oracle_slice(inp, sd, g0, 4)
        err = (first[g0:g0 + 4] - ref).abs()
        if not bool((err <= 1e-4 + 1e-4 * ref.abs()).all()):
            raise SystemExit(f"bench.py: output of graphs {g0}..{g0 + 3} differs from the oracle (max |err| {err.max().item():.3e})")
        parity_err = max(parity_err, err.max().item())

    # resident arm: the whole step — graph prep, 5 layers, Vh/Vx, pooling, the all-gather of the pooled features (N > 1)
    # and the answer MLP — replayed as ONE CUDA graph on static device buffers
    group = dist.group.WORLD if world > 1 else None
    try:
        step = DecoderStep(mod, pooler, fc, d, world, group, use_cuda_graph=not args.no_cuda_graph, max_edges=max_edges)
    except Exception as exc:  # noqa: BLE001  capture unavailable (e.g. a NCCL build that cannot be captured): per-kernel launches
        if args.no_cuda_graph:
            raise
        step = DecoderStep(mod, pooler, fc, d, world, group, use_cuda_graph=False, max_edges=max_edges)
        step.mode = f"per-kernel launches (CUDA graph capture failed: {type(exc).__name__})"
    launch_mode = step.mode if step.graph is not None or args.no_cuda_graph else step.mode

    # multi-rank check: every rank must hold the logits a single GPU computes for all N shards (rank 0 recomputes them)
    logits_err = None
    if world > 1:
        got = step.run()[0].clone()
        torch.cuda.synchronize()
        if rank == 0:
            refs = []
            for r in range(world):
                ri = synth_step_inputs(r)
                rd = {k_: ri[k_].to(dev) for k_ in DecoderStep.PACKED_FIELDS}
                refs.append(DecoderStep(mod, pooler, fc, rd, 1, None, use_cuda_graph=False,
                                        max_edges=int((ri["graph_ptr"][1:] - ri["graph_ptr"][:-1]).max())).run()[0])
            ref = torch.cat(refs)
            logits_err = (got - ref).abs().max().item()
            if logits_err > 1e-5 + 1e-5 * ref.abs().max().item():
                raise SystemExit(f"bench.py: {world}-rank logits differ from the single-GPU logits by {logits_err:.3e}")

    def step_resident():
        step.run()

    # e2e arm: the public streaming API (qagnn_b200.pipeline.StreamedRunner) around the same step: every step uploads its
    # inputs from pinned host memory and downloads the step's results (logits of the whole job + this rank's pooling
    # attention); copies run on their own streams, double-buffered (one captured graph per buffer set)
    def make_step(dev_inputs):
        return DecoderStep(mod, pooler, fc, dev_inputs, world, group, use_cuda_graph=step.graph is not None, max_edges=max_edges)
    runner = StreamedRunner(mod, host, dev, depth=2, make_step=make_step, fields=DecoderStep.PACKED_FIELDS, download=(0, 1))
    # second e2e figure, round 1's definition: bare QAGNN_Message_Passing.forward, [B,n,D] node output downloaded
    mod.use_cuda_graph = not args.no_cuda_graph
    runner_nodes = StreamedRunner(mod, host, dev, depth=2)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False):
        barrier()
        if profile:
            lib.qagnn_profile_enable(1)
        l0 = lib.qagnn_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        launches = lib.qagnn_launch_count() - l0
        prof = _lib.profile_read() if profile else None
        if profile:
            lib.qagnn_profile_enable(0)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), launches, prof

    def timed_e2e(r, steps):
        for _ in range(4):
            r.submit(host)
        r.drain()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for s_ in (r.h2d, r.compute, r.d2h):
            s_.wait_event(ev0)
        for _ in range(steps):
            r.submit(host)
        r.drain()
        ev1.record()
        barrier()
        t_ = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return t_.item()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, _, _ = timed(step_resident, args.steps)
    # the results of the last timed step, (logits, pool_attn, gnn_out) as DecoderStep.run returns them; the passes below
    # run the same model on other buffers
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = {name: t.detach().float().cpu().numpy()
                  for name, t in zip(("logits", "pool_attn", "gnn_out"), (step.logits, step.pool_attn, step.gnn_out))}
    ms_e2e = timed_e2e(runner, args.steps)
    ms_e2e_nodes = timed_e2e(runner_nodes, args.steps) if world == 1 else None
    # kernel-level pass: the same K steps launched kernel by kernel with the library's CUDA-event stage timers on the
    # launching stream (events cannot be timed inside a replayed graph); feeds `roofline`, `stages`, `gpu_launches`
    mod.use_cuda_graph = False
    eager = DecoderStep(mod, pooler, fc, d, world, group, use_cuda_graph=False, max_edges=max_edges)
    eager.run()
    ms_eager, launches, prof = timed(eager.run, args.steps, profile=True)
    clocks = sampler.stop() if rank == 0 else None

    ms_step = ms_total / args.steps
    value = world * k * E / (ms_step * 1e-3)
    e2e_value = world * k * E / (ms_e2e / args.steps * 1e-3)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = peaks.get("hbm_gbs", 6650.0)
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    mp_ms, mp_cnt = prof["message_passing"]
    mp_avg_ms = mp_ms / max(mp_cnt, 1)
    balg = b_alg_per_layer(N, E, D)
    achieved = balg / (mp_avg_ms * 1e-3) / 1e9 if mp_avg_ms > 0 else 0.0
    stages = {s: {"ms_per_step": v[0] / args.steps, "intervals_per_step": v[1] / args.steps} for s, v in prof.items()}
    stage_total = sum(v["ms_per_step"] for v in stages.values()) or 1.0
    for v in stages.values():
        v["share"] = v["ms_per_step"] / stage_total

    def finish():
        """Leaves the job without tearing NCCL down: the captured CUDA graphs hold NCCL kernels, and destroying the
        communicator under them hung the 2-GPU run at exit (profiles/README.md).  Everybody meets at a last barrier, then
        each process exits on its own."""
        sys.stdout.flush()
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)

    if rank != 0:
        finish()
        return
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(), "graphs_per_gpu": B, "N": N, "E": E, "parallelism": f"dp{world} (sub-graph "
                   "shards; ONE NCCL all_gather_into_tensor of the pooled features [B, 2D+sent_dim] per step, inside the step's "
                   "CUDA graph, then the answer MLP on the whole job's batch)" if world > 1 else "single GPU",
                   "l2": f"no flush: a step streams the {lib.qagnn_forward_workspace_bytes(_lib.C.byref(mod._shape(N, E, n))) / 1e6:.0f} MB "
                         "workspace + 51 MB inputs, > 126 MB L2", "step": "graph prep (packed batch: one launch) + 5 x (projection, message passing, "
                   "node MLP) + Vh/Vx epilogue + attention pooling + (all-gather) + answer MLP, inputs resident in HBM",
                   "launch": launch_mode, "numa_node_bound": numa},
        "qa_pairs_per_s": world * B / (ms_step * 1e-3),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": runner.h2d_bytes(), "d2h_bytes_per_step": runner.d2h_bytes(),
                "ms_per_step": ms_e2e / args.steps,
                "api": "qagnn_b200.pipeline.StreamedRunner around qagnn_b200.pipeline.DecoderStep: per step H2D of H/edge_index/"
                       "edge_type/node_type/node_score/sent_vecs/adj_lengths/graph_ptr from pinned host memory, the step, D2H of its results "
                       "(logits of the whole job + pooling attention) into pinned memory; copies on separate streams, "
                       "double-buffered, so they overlap the neighbouring steps' kernels"},
        "gpu_launches": int(launches),
        "gpu_launches_note": "kernels of libqagnn_b200.so enqueued by the K steps of the kernel-level pass (the CUDA graph "
                             "of the headline pass replays the same kernel nodes)",
        "ms_per_step_per_kernel_launches": ms_eager / args.steps,
        "roofline": {"kernel": "mp_headtile_kernel (fused logits + per-source softmax + out-degree rescale + per-target sum), one GATConvE layer",
                     "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": balg, "avg_launch_ms": mp_avg_ms,
                     "launches_timed": int(mp_cnt),
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch from the ncu capture of THIS kernel source
                     "traffic": mp_traffic_from_profile(mp_kernel_sha()) if world == 1 else None},
        # second-largest kernel: the tcgen05 projection GEMM, three bf16 passes (hi*hi, hi*lo, lo*hi)
        "roofline_gemm": gemm_roofline(N, D, CFG["H"], prof["projection"][0] / max(prof["projection"][1], 1), peaks),
        "stages": stages,
        "parity_gate": {"checked": "graphs 0-3 and %d-%d of the timed batch vs the CPU oracle before timing" % (B - 4, B - 1),
                        "max_abs_err": parity_err, "bar": "1e-4 + 1e-4*|ref|",
                        "multi_rank_logits_vs_single_gpu_max_abs_err": logits_err},
        "clocks": clocks,
    }
    if ms_e2e_nodes is not None:
        line["e2e_node_output"] = {"value": k * E / (ms_e2e_nodes / args.steps * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e_nodes / args.steps,
                                   "h2d_bytes_per_step": runner_nodes.h2d_bytes(), "d2h_bytes_per_step": runner_nodes.d2h_bytes(),
                                   "api": "round 1's definition: StreamedRunner around the bare QAGNN_Message_Passing.forward, the "
                                          "[B,n,D] node output downloaded every step"}
    if not args.no_cpu_baseline and world == 1:  # the CPU arm is reported at N=1 only
        r = cpu_reference_run(3, 1, args.cpu_sample_graphs, full_batch_once=True)
        line["cpu_baseline"] = {k_: r[k_] for k_ in ("value", "unit", "cores", "kind", "sample", "full_batch")}
    print(json.dumps(line))
    finish()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
