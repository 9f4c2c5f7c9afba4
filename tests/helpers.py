"""Shared helpers for the parity tests (tests only)."""
import glob
import os

import torch

from oracle import make_goldens as MG
from oracle import qagnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# "within 1e-4 fp32" (BASELINE.json north_star): |got - ref| <= ATOL + RTOL*|ref| element-wise
ATOL = 1e-4
RTOL = 1e-4


def golden_names(kind):
    names = []
    for p in sorted(glob.glob(os.path.join(GOLDEN, "*.pt"))):
        fx = torch.load(p, weights_only=False)
        if fx["kind"] == kind:
            names.append(os.path.basename(p)[:-3])
    return names


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)


def assert_close(got, ref, what="", atol=ATOL, rtol=RTOL):
    got = got.detach().cpu().double()
    ref = ref.detach().cpu().double()
    assert got.shape == ref.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    err = (got - ref).abs()
    bound = atol + rtol * ref.abs()
    worst = (err - bound).max().item() if err.numel() else -1.0
    assert worst <= 0, (f"{what}: max|err|={err.max().item():.3e} (ref scale {ref.abs().max().item():.3e}) "
                        f"exceeds {atol}+{rtol}*|ref| by {worst:.3e}")
    return err.max().item() if err.numel() else 0.0


def mp_core_reference(qkm, ke, me, prep, H):
    """The graph part of one GATConvE layer on node-level projections — what `training._MPCore` computes — restated in
    vectorised torch ops in the dtype of the inputs (fp64 in the tests), differentiable by autograd:

        s[e,h]  = Q[src] . (Kx[tgt] + Ke[combo])       per head, over the d = D/H columns of head h
        a       = softmax of s over the edges that share SRC          a' = a * outdeg(src)
        aggr[v] = sum_{e: tgt = v} a'[e,h] (Mx[src] + Me[combo])

    qkm [N, 3D] = Q | Kx | Mx; ke, me [C, D]; `prep` = O.graph_prep_oracle(...) (edges then self loops).
    Returns (aggr [N, D], alpha [E+N, H]) with alpha before the out-degree rescale, in edge_index' order."""
    N, D = qkm.size(0), qkm.size(1) // 3
    d = D // H
    src, tgt, combo = (torch.from_numpy(prep[k]) for k in ("src", "tgt", "combo"))
    outdeg = torch.from_numpy(prep["outdeg"]).to(qkm.dtype)
    Q, Kx, Mx = (qkm[:, i * D:(i + 1) * D].reshape(N, H, d) for i in range(3))
    Ke, Me = ke.reshape(-1, H, d), me.reshape(-1, H, d)
    s = (Q[src] * (Kx[tgt] + Ke[combo])).sum(-1)
    a = O.segment_softmax(s, src)
    a_scaled = a * outdeg[src][:, None]
    aggr = O.scatter_sum(a_scaled[:, :, None] * (Mx[src] + Me[combo]), tgt, N)
    return aggr.reshape(N, D), a


def regen_mp_inputs(fx):
    c = fx["case"]
    inp = O.synth_graph_batch(c["B"], c["n"], c["e"], c["D"], fx["n_etype"], c["seed"], c["realistic"])
    sd = O.random_state_dict(c["k"], c["D"], fx["n_ntype"], fx["n_etype"], c["regime"], c["seed"])
    fp = MG.fingerprint(inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"])
    assert fp == fx["input_fp"], "regenerated inputs differ from the ones the golden was minted on"
    wfp = MG.fingerprint(*[sd[k] for k in sorted(sd) if sd[k].dtype.is_floating_point])
    assert wfp == fx["weight_fp"], "regenerated weights differ from the ones the golden was minted on"
    return inp, sd


def regen_layer_inputs(fx):
    c = fx["case"]
    x, extra, node_type, ei, et = MG.build_layer_inputs(c, fx["n_ntype"], fx["n_etype"])
    assert MG.fingerprint(x, extra, node_type, ei, et) == fx["input_fp"]
    sd = MG.layer_state_dict(c, fx["n_ntype"], fx["n_etype"])
    return x, extra, node_type, ei, et, sd
