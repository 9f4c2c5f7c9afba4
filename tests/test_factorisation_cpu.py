"""CPU checks of the algebra the CUDA path relies on (DESIGN.md §2), independent of any GPU.

The kernels do not evaluate the reference's per-edge form: they project Q | Kx | Mx once per NODE, look the edge-encoder
term up in a table with one row per distinct one-hot feature ("combo"), fold the type-embedding half of `extra` into one bias
row per node type, fold BatchNorm into the preceding linear, and run the per-source softmax over CSR segments.  This file
restates that factorised evaluation in fp64 torch ops (test-local, nothing of the product is imported) and requires it to
agree with the oracle's per-edge restatement of modeling_qagnn.py:411-484 to 1e-10 — so a parity failure on the GPU can only
be a kernel bug, not an algebra bug.  It also pins on the oracle itself the size-independent properties the full-size GPU
tests use (edge-order invariance, sub-batch independence, attention normalisation).
"""
import math

import numpy as np
import pytest
import torch

from oracle import qagnn_oracle as O

F64 = torch.float64


def _combo_features(T, R):
    """[C, R+1+2T] one-hot rows in graph-prep's combo numbering (graph_prep_oracle)."""
    C = R * T * T + T
    tab = torch.zeros(C, R + 1 + 2 * T, dtype=F64)
    for c in range(C):
        if c < R * T * T:
            et, ts, tt = c // (T * T), (c // T) % T, c % T
        else:
            et, ts, tt = R, c - R * T * T, c - R * T * T
        tab[c, et] = 1
        tab[c, R + 1 + ts] = 1
        tab[c, R + 1 + T + tt] = 1
    return tab


def _fold_bn(sd, lin, bn):
    """Linear followed by eval BatchNorm as one linear: W' = s*W, b' = s*(b - mean) + beta."""
    s = sd[bn + ".weight"].to(F64) / torch.sqrt(sd[bn + ".running_var"].to(F64) + O.BN_EPS)
    W = sd[lin + ".weight"].to(F64) * s[:, None]
    b = (sd[lin + ".bias"].to(F64) - sd[bn + ".running_mean"].to(F64)) * s + sd[bn + ".bias"].to(F64)
    return W, b


def _factorised_layer(sd, prefix, x, score_emb, type_emb_rows, nt, prep, T, R, H):
    """One GATConvE layer the way qagnn_mp_forward evaluates it.  x [N,D], score_emb [N,D/2], type_emb_rows [T,D/2]."""
    N, D = x.shape
    d = D // H
    wq, bq = sd[prefix + ".linear_query.weight"].to(F64), sd[prefix + ".linear_query.bias"].to(F64)
    wk, bk = sd[prefix + ".linear_key.weight"].to(F64), sd[prefix + ".linear_key.bias"].to(F64)
    wm, bm = sd[prefix + ".linear_msg.weight"].to(F64), sd[prefix + ".linear_msg.bias"].to(F64)
    # edge table: the shared edge encoder (BatchNorm folded) on the C distinct one-hot rows, then the edge halves of key / msg
    W0, b0 = _fold_bn(sd, "edge_encoder.0", "edge_encoder.1")
    tab = torch.relu(_combo_features(T, R) @ W0.t() + b0) @ sd["edge_encoder.3.weight"].to(F64).t() + sd["edge_encoder.3.bias"].to(F64)
    Ke = tab @ wk[:, 2 * D:].t() + bk
    Me = tab @ wm[:, 2 * D:].t() + bm
    # node projection [x | type_emb | score_emb] -> Q|Kx|Mx with the type_emb columns folded into a per-type bias row
    Wp = torch.cat([wq / math.sqrt(d), wk[:, :2 * D], wm[:, :2 * D]], dim=0)                      # [3D, 2D]
    bp = torch.cat([bq / math.sqrt(d), torch.zeros(2 * D, dtype=F64)])
    Ws = torch.cat([Wp[:, :D], Wp[:, D + D // 2:]], dim=1)                                        # K = D + D/2
    tbias = bp[None, :] + type_emb_rows @ Wp[:, D:D + D // 2].t()                                 # [T, 3D]
    qkm = torch.cat([x, score_emb], dim=1) @ Ws.t() + tbias[nt]
    Q, Kx, Mx = qkm[:, :D].view(N, H, d), qkm[:, D:2 * D].view(N, H, d), qkm[:, 2 * D:].view(N, H, d)
    src, tgt, combo = (torch.from_numpy(prep[k]) for k in ("src", "tgt", "combo"))
    s = (Q[src] * (Kx[tgt] + Ke[combo].view(-1, H, d))).sum(-1)                                   # [E', H]
    # per-SOURCE softmax over CSR segments (stable order by source), then the out-degree rescale
    a = torch.empty_like(s)
    perm, rp = prep["perm_src"], prep["rowptr_src"]
    for v in range(N):
        seg = torch.from_numpy(perm[rp[v]:rp[v + 1]])
        if seg.numel():
            e = torch.exp(s[seg] - s[seg].max(0).values)
            a[seg] = e / (e.sum(0) + 1e-16)
    a_scaled = a * torch.from_numpy(prep["outdeg"])[src].to(F64)[:, None]
    aggr = torch.zeros(N, H, d, dtype=F64).index_add_(0, tgt, a_scaled[:, :, None] * (Mx[src] + Me[combo].view(-1, H, d)))
    aggr = aggr.view(N, D)
    W1, b1 = _fold_bn(sd, prefix + ".mlp.0", prefix + ".mlp.1")
    out = torch.relu(aggr @ W1.t() + b1) @ sd[prefix + ".mlp.3.weight"].to(F64).t() + sd[prefix + ".mlp.3.bias"].to(F64)
    return out, a, aggr, (qkm, Ke, Me)


def _factorised_forward(sd, b, k, T, R, H):
    Bn, n, D = b["H"].shape
    nt = b["node_type"].reshape(-1)
    prep = O.graph_prep_oracle(b["edge_index"], b["edge_type"], nt, T, R)
    type_emb_rows = O.gelu_tanh(torch.eye(T, dtype=F64) @ sd["emb_node_type.weight"].to(F64).t() + sd["emb_node_type.bias"].to(F64))
    js = torch.pow(1.1, torch.arange(D // 2).float())                         # fp32, as modeling_qagnn.py:70-71
    basis = torch.sin((js[None, :] * b["node_score"].reshape(-1, 1).float()).to(F64))
    score_emb = O.gelu_tanh(basis @ sd["emb_score.weight"].to(F64).t() + sd["emb_score.bias"].to(F64))
    X = b["H"].to(F64).reshape(-1, D)
    layers = []
    for l in range(k):
        X, a, aggr, proj = _factorised_layer(sd, f"gnn_layers.{l}", X, score_emb, type_emb_rows, nt, prep, T, R, H)
        X = O.gelu_tanh(X)
        layers.append({"x": X, "alpha": a, "aggr": aggr, "proj": proj})
    Vcat = torch.cat([sd["Vh.weight"], sd["Vx.weight"]], dim=1).to(F64)     # one GEMM over [H | X]
    out = O.gelu_tanh(torch.cat([b["H"].to(F64).reshape(-1, D), X], dim=1) @ Vcat.t() + (sd["Vh.bias"].to(F64) + sd["Vx.bias"].to(F64)))
    return out.view(Bn, n, D), layers, prep


_FACTORISATION_CASES = [
    ("peaky", False, 3, 12, 40, 16, 4, 2, 38),
    ("prod", True, 4, 20, 60, 24, 4, 3, 38),
    ("peaky", True, 2, 9, 0, 16, 2, 1, 6),       # no real edges: self loops only
    ("peaky", False, 1, 1, 3, 8, 2, 2, 5),       # one node, three i->i edges
]


@pytest.mark.parametrize("regime,realistic,B,n,e,D,H,k,R", _FACTORISATION_CASES)
def test_node_level_factorisation_equals_the_per_edge_form(regime, realistic, B, n, e, D, H, k, R):
    T = 4
    b = O.synth_graph_batch(B, n, e, D, n_etype=R, seed=11, realistic=realistic)
    sd = O.random_state_dict(k, D, T, R, regime=regime, seed=3)
    want, _, want_layers = O.message_passing_forward(sd, b["H"], b["edge_index"], b["edge_type"], b["node_type"], b["node_score"],
                                                    k, T, R, head_count=H, dtype=F64, return_layers=True)
    got, got_layers, _ = _factorised_forward(sd, b, k, T, R, H)
    for g, w in zip(got_layers, want_layers):
        assert torch.allclose(g["alpha"], w["alpha"], rtol=0, atol=1e-12)
        assert torch.allclose(g["aggr"], w["aggr"], rtol=1e-10, atol=1e-10)
        assert torch.allclose(g["x"], w["x"], rtol=1e-10, atol=1e-10)
    assert torch.allclose(got, want, rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("regime,realistic,B,n,e,D,H,k,R", _FACTORISATION_CASES)
def test_mp_core_reference_on_factorised_projections_equals_the_per_edge_form(regime, realistic, B, n, e, D, H, k, R):
    """tests/helpers.mp_core_reference — the fp64 reference the GPU kernel tests compare _MPCore with — fed the factorised
    Q|Kx|Mx, Ke, Me of every layer gives the oracle's per-edge alpha and aggr."""
    from tests import helpers as Hh
    T = 4
    b = O.synth_graph_batch(B, n, e, D, n_etype=R, seed=11, realistic=realistic)
    sd = O.random_state_dict(k, D, T, R, regime=regime, seed=3)
    _, _, want_layers = O.message_passing_forward(sd, b["H"], b["edge_index"], b["edge_type"], b["node_type"], b["node_score"],
                                                  k, T, R, head_count=H, dtype=F64, return_layers=True)
    _, got_layers, prep = _factorised_forward(sd, b, k, T, R, H)
    for g, w in zip(got_layers, want_layers):
        qkm, Ke, Me = g["proj"]
        aggr, alpha = Hh.mp_core_reference(qkm, Ke, Me, prep, H)
        assert torch.allclose(alpha, w["alpha"], rtol=1e-10, atol=1e-10)
        assert torch.allclose(aggr, w["aggr"], rtol=1e-10, atol=1e-10)


def _mp(sd, b, k, R, H=4, **kw):
    return O.message_passing_forward(sd, b["H"], b["edge_index"], b["edge_type"], b["node_type"], b["node_score"], k, 4, R,
                                     head_count=H, dtype=F64, **kw)


def test_oracle_is_invariant_to_edge_order_and_batches_are_independent():
    B, n, e, D, k, R = 5, 14, 50, 16, 2, 38
    b = O.synth_graph_batch(B, n, e, D, n_etype=R, seed=4)
    sd = O.random_state_dict(k, D, 4, R, regime="peaky", seed=1)
    full = _mp(sd, b, k, R)
    perm = torch.randperm(b["edge_type"].numel(), generator=torch.Generator().manual_seed(0))
    shuffled = dict(b, edge_index=b["edge_index"][:, perm].contiguous(), edge_type=b["edge_type"][perm])
    assert torch.allclose(_mp(sd, shuffled, k, R), full, rtol=1e-11, atol=1e-11)
    for g in (0, 3, 4):   # a graph of the batch computed alone gives the same rows
        m = (b["edge_index"][0] >= g * n) & (b["edge_index"][0] < (g + 1) * n)
        alone = {"H": b["H"][g:g + 1], "edge_index": b["edge_index"][:, m] - g * n, "edge_type": b["edge_type"][m],
                 "node_type": b["node_type"][g:g + 1], "node_score": b["node_score"][g:g + 1]}
        assert torch.allclose(_mp(sd, alone, k, R)[0], full[g], rtol=1e-11, atol=1e-11)


def test_oracle_attention_sums_to_one_per_source_and_rescale_is_the_out_degree():
    B, n, e, D, R = 2, 10, 35, 16, 38
    b = O.synth_graph_batch(B, n, e, D, n_etype=R, seed=9)
    sd = O.random_state_dict(1, D, 4, R, regime="peaky", seed=2)
    _, _, layers = _mp(sd, b, 1, R, return_layers=True)
    alpha = layers[0]["alpha"]
    prep = O.graph_prep_oracle(b["edge_index"], b["edge_type"], b["node_type"].reshape(-1), 4, R)
    src = torch.from_numpy(prep["src"])
    sums = torch.zeros(B * n, alpha.size(1), dtype=F64).index_add_(0, src, alpha)
    assert torch.allclose(sums, torch.ones_like(sums), atol=1e-12)     # every node has at least its self loop
    assert int(prep["outdeg"].min()) >= 1 and int(prep["outdeg"].sum()) == e * B + B * n
    # duplicated edges are separate softmax entries with equal weight
    ei, et = b["edge_index"], b["edge_type"]
    dup = dict(b, edge_index=torch.cat([ei, ei[:, :1]], 1), edge_type=torch.cat([et, et[:1]]))
    _, _, l2 = _mp(sd, dup, 1, R, return_layers=True)
    assert torch.allclose(l2[0]["alpha"][0], l2[0]["alpha"][ei.size(1)], atol=0)
    assert np.array_equal(O.graph_prep_oracle(dup["edge_index"], dup["edge_type"], b["node_type"].reshape(-1), 4, R)["outdeg"],
                          prep["outdeg"] + np.bincount([int(ei[0, 0])], minlength=B * n))


def _core_forward(Q, Kx, Mx, Ke, Me, src, tgt, combo, outdeg, N):
    """The graph part of a layer on node-level projections (what qagnn_mp_core_forward evaluates), in autograd-able torch ops."""
    s = (Q[src] * (Kx[tgt] + Ke[combo])).sum(-1)
    a = O.segment_softmax(s, src)
    a_scaled = a * outdeg[src][:, None]
    aggr = torch.zeros(N, *Q.shape[1:], dtype=F64).index_add_(0, tgt, a_scaled[:, :, None] * (Mx[src] + Me[combo]))
    return aggr, a, a_scaled


@pytest.mark.parametrize("seed,B,n,e", [(0, 3, 9, 30), (1, 2, 6, 0), (2, 1, 1, 4)])
def test_backward_formulas_of_the_graph_part_equal_autograd(seed, B, n, e):
    """DESIGN.md §2b: da' = G[tgt]·(Mx[src]+Me[c]); ds = a(da − Σ_src a·da) with da = outdeg·da'; dQ / dKx / dKe from ds,
    dMx / dMe from a'·G — the closed forms mp_bwd_source / _target / _table_kernel implement, against autograd."""
    T, R, H, d = 4, 7, 2, 5
    b = O.synth_graph_batch(B, n, e, H * d, n_etype=R, seed=seed)
    N = B * n
    prep = O.graph_prep_oracle(b["edge_index"], b["edge_type"], b["node_type"].reshape(-1), T, R)
    src, tgt, combo = (torch.from_numpy(prep[k]) for k in ("src", "tgt", "combo"))
    outdeg = torch.from_numpy(prep["outdeg"]).to(F64)
    g = torch.Generator().manual_seed(seed)
    C = R * T * T + T
    Q, Kx, Mx = (torch.randn(N, H, d, dtype=F64, generator=g, requires_grad=True) for _ in range(3))
    Ke, Me = (torch.randn(C, H, d, dtype=F64, generator=g, requires_grad=True) for _ in range(2))
    G = torch.randn(N, H, d, dtype=F64, generator=g)
    aggr, a, a_scaled = _core_forward(Q, Kx, Mx, Ke, Me, src, tgt, combo, outdeg, N)
    want = torch.autograd.grad(aggr, (Q, Kx, Mx, Ke, Me), G)
    with torch.no_grad():
        da_scaled = (G[tgt] * (Mx[src] + Me[combo])).sum(-1)                     # [E', H]
        da = da_scaled * outdeg[src][:, None]
        dot = torch.zeros(N, H, dtype=F64).index_add_(0, src, a * da)            # Σ over the edges of one source
        ds = a * (da - dot[src])
        zeros = lambda rows: torch.zeros(rows, H, d, dtype=F64)                  # noqa: E731
        dQ = zeros(N).index_add_(0, src, ds[:, :, None] * (Kx[tgt] + Ke[combo]))
        dKx = zeros(N).index_add_(0, tgt, ds[:, :, None] * Q[src])
        dKe = zeros(C).index_add_(0, combo, ds[:, :, None] * Q[src])
        dMx = zeros(N).index_add_(0, src, a_scaled[:, :, None] * G[tgt])
        dMe = zeros(C).index_add_(0, combo, a_scaled[:, :, None] * G[tgt])
    for name, got, w in zip(("dQ", "dKx", "dMx", "dKe", "dMe"), (dQ, dKx, dMx, dKe, dMe), want):
        assert torch.allclose(got, w, rtol=1e-9, atol=1e-9), name
