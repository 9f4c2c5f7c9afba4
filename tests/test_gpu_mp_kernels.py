"""The message-passing kernels alone, forward and backward, at every head count and head width the library compiles for,
against fp64 references.  Needs a GPU.

* `training._MPCore` (qagnn_mp_core_forward / qagnn_mp_core_backward: mp_scores / mp_aggregate, mp_bwd_source / _target /
  _table) against autograd through `helpers.mp_core_reference` in fp64 — aggr, alpha and the gradients of qkm, Ke, Me
  compared directly, not through the dense layers around them.  The (H, D) rows reach every CH instance of the kernels
  (D <= 128 / 256 / 512 / 1024), a CH = 8 instance with masked lanes (D = 520) and float4 chunks that straddle heads
  (d = 50, 17, 5, 3, 1); the graphs reach hub segments of ~2000 edges, no edges, one node, duplicate edges, one combo
  spanning many 64-edge runs of the table kernel, E + N on both sides of a multiple of 64, and saturated softmaxes.
* `GATConvE(..., head_count=H).eval()` against the oracle's per-edge layer in fp64, through the column-sliced kernels
  (every slice width) and the basic CSR kernels.
* Shapes no message-passing path can run raise QagnnError in .eval() and .train() instead of returning numbers.
"""
import functools

import numpy as np
import pytest
import torch

import qagnn_b200
from oracle import qagnn_oracle as O
from qagnn_b200 import _lib
from qagnn_b200.modeling_qagnn import GraphPrep
from qagnn_b200.training import _MPCore
from tests import helpers as Hh

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F64 = torch.float64


def _grad_close(got, ref, what):
    # the project's gradient bar: 1e-4 of the tensor's own largest value, plus 1e-4 relative
    scale = max(float(ref.abs().max()), 1e-6)
    Hh.assert_close(got, ref, what, atol=1e-4 * scale, rtol=1e-4)


def _rand_edges(g, N, E):
    return torch.randint(0, N, (2, E), generator=g)


@functools.lru_cache(maxsize=None)
def _graph(kind):
    """(edge_index [2,E], edge_type [E], node_type [N], T, R), each kind from its own fixed seed."""
    seeds = ["random", "hub", "empty", "single", "dup", "t1r1", "mod64", "mod64p1", "peaky"]
    g = torch.Generator().manual_seed(100 + seeds.index(kind))
    T, R = 4, 38
    if kind in ("random", "peaky"):
        N, ei = 300, _rand_edges(g, 300, 1500)
    elif kind == "hub":
        # node 5 is the source of 2000 edges, node 9 the target of 2000 more: one warp loops over each segment
        N, deg = 300, 2000
        ei = _rand_edges(g, N, 2 * deg + 500)
        ei[0, :deg] = 5
        ei[1, deg:2 * deg] = 9
        ei = ei[:, torch.randperm(ei.size(1), generator=g)]
    elif kind == "empty":
        N, ei = 50, torch.zeros(2, 0, dtype=torch.long)
    elif kind == "single":
        N, ei = 1, torch.zeros(2, 0, dtype=torch.long)
    elif kind == "dup":
        # 300 distinct (src, tgt, type) triples, each repeated 1..6 times
        N, base = 200, _rand_edges(g, 200, 300)
        et0 = torch.randint(0, R, (300,), generator=g)
        rep = torch.randint(1, 7, (300,), generator=g)
        ei, et = base.repeat_interleave(rep, dim=1), et0.repeat_interleave(rep)
        nt = torch.randint(0, T, (N,), generator=g)
        return ei, et, nt, T, R
    elif kind == "t1r1":
        # one node type, one relation: every real edge has combo 0, so the table kernel flushes the same row from ~24 runs
        T, R = 1, 1
        N, ei = 300, _rand_edges(g, 300, 1500)
    elif kind == "mod64":
        N, ei = 100, _rand_edges(g, 100, 1180)      # E + N = 20 * 64
    elif kind == "mod64p1":
        N, ei = 100, _rand_edges(g, 100, 1181)      # E + N = 20 * 64 + 1
    else:
        raise ValueError(kind)
    et = torch.randint(0, R, (ei.size(1),), generator=g)
    nt = torch.randint(0, T, (N,), generator=g)
    return ei, et, nt, T, R


def _core_inputs(kind, N, D, H, C, seed):
    """Random fp32 qkm [N, 3D], ke / me [C, D] and upstream gradient G [N, D].  Q carries the layer's 1/sqrt(d), so logits
    are O(1); for `peaky` Q is rescaled until the largest |logit| is 30 and most per-source softmaxes saturate."""
    d = D // H
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(N, D, generator=g) / d ** 0.5
    kx = torch.randn(N, D, generator=g)
    mx = torch.randn(N, D, generator=g) * 0.1
    ke = torch.randn(C, D, generator=g) * 0.5
    me = torch.randn(C, D, generator=g) * 0.1
    G = torch.randn(N, D, generator=g)
    qkm = torch.cat([q, kx, mx], dim=1)
    return qkm, ke, me, G


# (H, D): D <= 128 / 256 / 512 / 1024 selects CH = 1 / 2 / 4 / 8 (float4 chunks per lane); D = 520 runs CH = 8 with the
# last 126 chunk slots masked; d = 50, 17, 5, 3, 1 put head boundaries inside float4 chunks
SHAPES = [(1, 4), (1, 1024), (2, 100), (2, 520), (4, 12), (4, 200), (4, 1024), (8, 8), (8, 40), (8, 1024),
          (16, 16), (16, 272), (16, 1024)]
OTHER_GRAPHS = ["empty", "single", "dup", "t1r1", "mod64", "mod64p1", "peaky"]
CORE_CASES = ([(kind, H, D) for (H, D) in SHAPES for kind in ("random", "hub")]
              + [(kind, H, D) for kind in OTHER_GRAPHS for (H, D) in ((16, 272), (8, 1024), (2, 520), (8, 40))])


def _run_core(kind, H, D):
    ei, et, nt, T, R = _graph(kind)
    N, E = nt.numel(), ei.size(1)
    C = R * T * T + T
    qkm, ke, me, G = _core_inputs(kind, N, D, H, C, seed=7 + H * 4096 + D)
    prep_o = O.graph_prep_oracle(ei, et, nt, T, R)
    if kind == "peaky":
        src, tgt, combo = (torch.from_numpy(prep_o[k]) for k in ("src", "tgt", "combo"))
        q, k = qkm[:, :D].double()[src], (qkm[:, D:2 * D].double()[tgt] + ke.double()[combo])
        s = (q * k).view(-1, H, D // H).sum(-1)
        qkm[:, :D] *= 30.0 / float(s.abs().max())
    # fp64 reference and its gradients
    q64, k64, m64 = (t.double().requires_grad_(True) for t in (qkm, ke, me))
    ref_aggr, ref_alpha = Hh.mp_core_reference(q64, k64, m64, prep_o, H)
    ref_dq, ref_dk, ref_dm = torch.autograd.grad(ref_aggr, (q64, k64, m64), G.double())
    # device
    prep = GraphPrep(ei.to(DEV), et.to(DEV), nt.to(DEV), T, R, 0)
    qd, kd, md = (t.to(DEV).requires_grad_(True) for t in (qkm, ke, me))
    aggr, alpha = _MPCore.apply(qd, kd, md, prep, (N, E, D, H, T, R), True)
    got = torch.autograd.grad(aggr, (qd, kd, md), G.to(DEV), retain_graph=True)
    return dict(prep_o=prep_o, C=C, ref=(ref_aggr, ref_alpha, ref_dq, ref_dk, ref_dm), aggr=aggr, alpha=alpha, got=got,
                dev=(qd, kd, md, G))


@pytest.mark.parametrize("kind,H,D", CORE_CASES)
def test_mp_core_forward_and_backward_against_fp64_autograd(kind, H, D):
    r = _run_core(kind, H, D)
    ref_aggr, ref_alpha, ref_dq, ref_dk, ref_dm = r["ref"]
    if kind == "peaky":  # softmaxes over several edges saturate
        multi = torch.from_numpy(r["prep_o"]["outdeg"][r["prep_o"]["src"]] > 1)
        a = ref_alpha.detach()[multi]
        assert float(a.max()) > 0.999 and float(a.min()) < 1e-6
    Hh.assert_close(r["alpha"], ref_alpha, "alpha")
    Hh.assert_close(r["aggr"], ref_aggr, "aggr")
    d_qkm, d_ke, d_me = r["got"]
    _grad_close(d_qkm[:, :D], ref_dq[:, :D], "dQ")
    _grad_close(d_qkm[:, D:2 * D], ref_dq[:, D:2 * D], "dKx")
    _grad_close(d_qkm[:, 2 * D:], ref_dq[:, 2 * D:], "dMx")
    _grad_close(d_ke, ref_dk, "dKe")
    _grad_close(d_me, ref_dm, "dMe")
    # combos no edge uses: their gradient rows are exactly zero (nothing flushed into them)
    unused = torch.from_numpy(np.bincount(r["prep_o"]["combo"], minlength=r["C"]) == 0)
    assert torch.equal(d_ke.cpu()[unused], torch.zeros(int(unused.sum()), D))
    assert torch.equal(d_me.cpu()[unused], torch.zeros(int(unused.sum()), D))
    # d_qkm has no atomics: a second backward gives the same bits (d_ke / d_me accumulate atomically: tolerance only)
    qd, kd, md, G = r["dev"]
    again = torch.autograd.grad(r["aggr"], (qd, kd, md), G.to(DEV))
    assert torch.equal(again[0], d_qkm), "d_qkm differs between two backward calls"
    _grad_close(again[1], ref_dk, "dKe (second backward)")
    _grad_close(again[2], ref_dm, "dMe (second backward)")


@pytest.mark.parametrize("H,D", [(1, 4), (16, 272), (8, 1024)])
def test_mp_core_backward_of_a_sum_takes_a_stride_zero_gradient(H, D):
    """aggr.sum().backward() hands the backward an expanded (stride-0) upstream gradient of ones."""
    ei, et, nt, T, R = _graph("random")
    N, E = nt.numel(), ei.size(1)
    C = R * T * T + T
    qkm, ke, me, _ = _core_inputs("random", N, D, H, C, seed=3)
    prep_o = O.graph_prep_oracle(ei, et, nt, T, R)
    q64, k64, m64 = (t.double().requires_grad_(True) for t in (qkm, ke, me))
    Hh.mp_core_reference(q64, k64, m64, prep_o, H)[0].sum().backward()
    prep = GraphPrep(ei.to(DEV), et.to(DEV), nt.to(DEV), T, R, 0)
    qd, kd, md = (t.to(DEV).requires_grad_(True) for t in (qkm, ke, me))
    aggr, _ = _MPCore.apply(qd, kd, md, prep, (N, E, D, H, T, R), False)
    aggr.sum().backward()
    _grad_close(qd.grad, q64.grad, "d_qkm")
    _grad_close(kd.grad, k64.grad, "d_ke")
    _grad_close(md.grad, m64.grad, "d_me")


# ---- GATConvE.eval() at every head count, default path and basic CSR kernels ----------------------------------------
def _layer_graph(kind):
    """Eval-layer graphs: E stays below ~5k so the per-edge fp64 oracle is quick at D = 1024."""
    g = torch.Generator().manual_seed(200 + (kind == "hub"))
    N = 300
    if kind == "random":
        ei = _rand_edges(g, N, 1500)
    else:
        ei = _rand_edges(g, N, 4000)
        ei[0, :1500] = 7
        ei[1, 1500:3000] = 11
    et = torch.randint(0, 38, (ei.size(1),), generator=g)
    nt = torch.randint(0, 4, (N,), generator=g)
    return ei, et, nt


@functools.lru_cache(maxsize=None)
def _layer_case(kind, H, D):
    ei, et, nt = _layer_graph(kind)
    N = nt.numel()
    g = torch.Generator().manual_seed(300 + H * 4096 + D)
    x = torch.randn(N, D, generator=g) * 0.5
    extra = torch.randn(N, D, generator=g) * 0.5
    sd = O.random_state_dict(1, D, 4, 38, "peaky", seed=H * 4096 + D)
    ref = O.gatconve_forward(sd, "gnn_layers.0", x, ei, et, nt, extra, 4, 38, head_count=H, dtype=F64)
    return ei, et, nt, x, extra, sd, ref


def _layer(sd, D, H, n_ntype=4, n_etype=38):
    enc = torch.nn.Sequential(torch.nn.Linear(n_etype + 1 + 2 * n_ntype, D), torch.nn.BatchNorm1d(D), torch.nn.ReLU(),
                              torch.nn.Linear(D, D))
    layer = qagnn_b200.GATConvE(None, D, n_ntype, n_etype, enc, head_count=H).eval()
    layer.load_state_dict({k_[len("gnn_layers.0."):]: v for k_, v in sd.items() if k_.startswith("gnn_layers.0.")})
    return layer.to(DEV)


# the default path's kernel per row (make_slice_plan): column slices of SL = 16 / 32 / 64 columns, one or two per head;
# d = 5 and d = 3 have no slice plan and run the basic CSR kernels (D = 12 also runs the FFMA GEMMs: D % 8 != 0)
EVAL_SHAPES = [(16, 256), (2, 64), (2, 128), (16, 1024), (1, 128), (8, 40), (4, 12)]


@pytest.mark.parametrize("path", ["default", "basic"])
@pytest.mark.parametrize("kind", ["random", "hub"])
@pytest.mark.parametrize("H,D", EVAL_SHAPES)
def test_gatconve_eval_at_every_head_count_against_fp64_oracle(H, D, kind, path, monkeypatch):
    if path == "basic":
        monkeypatch.setenv("QAGNN_MP_PATH", "basic")
    ei, et, nt, x, extra, sd, (ref_out, ref_ei, ref_alpha, ref_aggr) = _layer_case(kind, H, D)
    layer = _layer(sd, D, H)
    (out, (ei_g, alpha)), aggr = layer(x.to(DEV), ei.to(DEV), et.to(DEV), nt.to(DEV), extra.to(DEV),
                                       return_attention_weights=True, return_aggr=True)
    assert torch.equal(ei_g.cpu(), ref_ei)
    Hh.assert_close(alpha, ref_alpha, f"alpha H={H} D={D} {kind} {path}")
    Hh.assert_close(aggr, ref_aggr, f"aggr H={H} D={D} {kind} {path}")
    # hub: the softmax of the 1500-edge source saturates, so a' = a * outdeg reaches ~1500 and aggr ~5e2; the node MLP in
    # fp32 then rounds at ~1e-5 of the output's scale, above 1e-4 absolute on its small entries (aggr itself meets the bar)
    atol = 2e-5 * float(ref_out.abs().max()) if kind == "hub" else Hh.ATOL
    Hh.assert_close(out, ref_out, f"out H={H} D={D} {kind} {path}", atol=atol)


# ---- shapes no message-passing path takes ---------------------------------------------------------------------------
# D % 4 != 0 (float4 columns) with no slice plan, H outside {1, 2, 4, 8, 16} (H = 3), and D > 1024 with no slice plan
@pytest.mark.parametrize("D,H", [(50, 2), (18, 1), (48, 3), (1040, 8)])
def test_shapes_without_a_message_passing_path_raise_in_eval_and_train(D, H):
    ei, et, nt = _layer_graph("random")
    N = nt.numel()
    g = torch.Generator().manual_seed(D)
    x, extra = torch.randn(N, D, generator=g).to(DEV), torch.randn(N, D, generator=g).to(DEV)
    sd = O.random_state_dict(1, D, 4, 38, "peaky", seed=1)
    layer = _layer(sd, D, H)
    args = (x, ei.to(DEV), et.to(DEV), nt.to(DEV), extra)
    with pytest.raises(_lib.QagnnError, match="unsupported"):
        layer.eval()(*args)
    with pytest.raises(_lib.QagnnError, match="unsupported"):
        layer.train()(*args).sum().backward()


def test_head_tiled_kernel_takes_a_width_the_csr_kernels_refuse():
    """D = 50 (d = 25) has no CSR path, but the head-tiled kernel pads heads to 28 columns and runs it when the caller passes
    a per-graph prep: the refusal is per path, not per shape.  The training path has only the CSR kernels and refuses."""
    D, H, n, B = 50, 2, 60, 5
    inp = O.synth_graph_batch(B, n, 200, D, 38, seed=17)
    sd = O.random_state_dict(1, D, 4, 38, "peaky", seed=17)
    x = inp["H"].view(-1, D)
    extra = torch.randn(x.shape, generator=torch.Generator().manual_seed(2)) * 0.5
    nt = inp["node_type"].view(-1)
    ref_out, _, ref_alpha, ref_aggr = O.gatconve_forward(sd, "gnn_layers.0", x, inp["edge_index"], inp["edge_type"], nt, extra,
                                                         4, 38, head_count=H, dtype=F64)
    layer = _layer(sd, D, H)
    ntd = nt.to(DEV)
    prep = GraphPrep(inp["edge_index"].to(DEV), inp["edge_type"].to(DEV), ntd, 4, 38, n_per_graph=n)
    (out, (_, alpha)), aggr = layer(x.to(DEV), None, None, ntd, extra.to(DEV), return_attention_weights=True, prep=prep,
                                    return_aggr=True)
    Hh.assert_close(alpha, ref_alpha, "alpha (head-tiled, d = 25)")
    Hh.assert_close(aggr, ref_aggr, "aggr (head-tiled, d = 25)")
    Hh.assert_close(out, ref_out, "out (head-tiled, d = 25)")
    with pytest.raises(_lib.QagnnError, match="unsupported"):
        layer.train()(x.to(DEV), None, None, ntd, extra.to(DEV), prep=prep)
