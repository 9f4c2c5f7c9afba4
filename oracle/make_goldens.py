"""TEST INFRASTRUCTURE — mints tests/golden/*.pt from the reference's OWN modules.

Needs the reference tree (oracle/ref_shim.py, QAGNN_REFERENCE_ROOT):

    python -m oracle.make_goldens            # writes tests/golden/*.pt
    python -m oracle.make_goldens --check    # re-mints in memory, compares with the committed files, writes nothing
    python -m oracle.make_goldens --fuzz 24  # reference vs oracle on 24 random cases that are not committed as fixtures
    python -m oracle.make_goldens --record   # stores what the reference produced where the tests compare against it
                                             # (tests/golden/reference_digests.json, fuzz_mp_sampled.pt)

Every fixture is produced by the unmodified `GATConvE` / `QAGNN_Message_Passing` / `QAGNN`
classes of /root/reference/modeling/modeling_qagnn.py (imported through oracle/ref_shim.py),
in eval mode, fp32, on CPU.  Inputs and weights are regenerated deterministically from seeds by
`oracle.qagnn_oracle.synth_graph_batch` / `random_state_dict`, so the fixtures only store the
case description, a fingerprint of the regenerated inputs, and the reference outputs.
"""
import hashlib
import json
import os
import sys

import torch

from oracle import qagnn_oracle as O
from oracle.ref_shim import load_reference

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def fingerprint(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


# ---------------------------------------------------------------------------------------------
# case table (shared with the tests through the saved 'case' dict)
# ---------------------------------------------------------------------------------------------
MP_CASES = [
    # name, B, n, e/graph, D, k, regime, realistic, seed
    dict(name="cfg1_prod", B=4, n=50, e=200, D=64, k=1, regime="prod", realistic=False, seed=0),
    dict(name="cfg1_peaky_k2", B=4, n=50, e=200, D=64, k=2, regime="peaky", realistic=False, seed=1),
    dict(name="cfg2small_prod", B=3, n=200, e=1000, D=200, k=5, regime="prod", realistic=False, seed=0),
    dict(name="cfg2small_peaky", B=3, n=200, e=1000, D=200, k=5, regime="peaky", realistic=False, seed=2),
    dict(name="cfg2small_realistic", B=5, n=200, e=1000, D=200, k=5, regime="peaky", realistic=True, seed=3),
    dict(name="tiny_realistic_d100", B=6, n=24, e=60, D=100, k=3, regime="peaky", realistic=True, seed=4),
    dict(name="no_edges", B=3, n=10, e=0, D=64, k=2, regime="peaky", realistic=False, seed=5),
]

# single-layer GATConvE cases (hand-built graphs and non-default head counts)
LAYER_CASES = [
    dict(name="layer_h8_d1024", N=40, E=300, D=1024, H=8, regime="peaky", seed=10, kind="random"),
    dict(name="layer_h8_d64", N=30, E=200, D=64, H=8, regime="peaky", seed=11, kind="random"),
    dict(name="layer_h4_d200_prod", N=200, E=1000, D=200, H=4, regime="prod", seed=12, kind="random"),
    dict(name="layer_multi_dup", N=12, E=0, D=64, H=4, regime="peaky", seed=13, kind="multi_dup"),
    dict(name="layer_src_only_tgt_only", N=9, E=0, D=64, H=4, regime="peaky", seed=14, kind="bipartite"),
    dict(name="layer_hub", N=300, E=0, D=64, H=4, regime="peaky", seed=15, kind="hub"),
    dict(name="layer_single_node", N=1, E=0, D=64, H=4, regime="peaky", seed=16, kind="random"),
]


def build_layer_inputs(case, n_ntype=4, n_etype=38):
    g = torch.Generator().manual_seed(500 + case["seed"])
    N, D = case["N"], case["D"]
    x = torch.randn(N, D, generator=g) * 0.5
    extra = torch.randn(N, D, generator=g) * 0.5
    node_type = torch.randint(0, n_ntype, (N,), generator=g)
    kind = case["kind"]
    if kind == "random":
        E = case["E"]
        ei = torch.randint(0, N, (2, E), generator=g)
        et = torch.randint(0, n_etype, (E,), generator=g)
    elif kind == "multi_dup":
        # parallel multi-edges of different type between the same pair, exact duplicates, explicit i->i
        pairs = [(0, 1, 3), (0, 1, 7), (0, 1, 7), (0, 1, 7), (1, 0, 22), (2, 2, 5), (2, 2, 5), (3, 4, 0),
                 (3, 4, 37), (4, 3, 19), (5, 6, 1), (5, 6, 1), (11, 0, 9), (11, 0, 9), (11, 0, 10)]
        ei = torch.tensor([[p[0] for p in pairs], [p[1] for p in pairs]])
        et = torch.tensor([p[2] for p in pairs])
    elif kind == "bipartite":
        # nodes 0-3 only ever sources, 4-7 only ever targets, node 8 isolated (self loop only)
        s = torch.tensor([0, 0, 1, 2, 3, 3, 3, 1])
        t = torch.tensor([4, 5, 5, 6, 7, 4, 5, 7])
        ei = torch.stack([s, t])
        et = torch.randint(0, n_etype, (s.numel(),), generator=g)
    elif kind == "hub":
        # node 0 points at everybody (out-degree N) and half of them point back (in-degree N/2)
        s = torch.cat([torch.zeros(N - 1, dtype=torch.long), torch.arange(1, N, 2)])
        t = torch.cat([torch.arange(1, N), torch.zeros(len(range(1, N, 2)), dtype=torch.long)])
        ei = torch.stack([s, t])
        et = torch.randint(0, n_etype, (s.numel(),), generator=g)
    else:
        raise ValueError(kind)
    return x, extra, node_type, ei.long().contiguous(), et.long().contiguous()


def layer_state_dict(case, n_ntype=4, n_etype=38):
    full = O.random_state_dict(1, case["D"], n_ntype, n_etype, case["regime"], case["seed"])
    return full


@torch.no_grad()
def mint_mp_case(ref, case, n_ntype=4, n_etype=38):
    inp = O.synth_graph_batch(case["B"], case["n"], case["e"], case["D"], n_etype, case["seed"], case["realistic"])
    sd = O.random_state_dict(case["k"], case["D"], n_ntype, n_etype, case["regime"], case["seed"])
    mod = ref.QAGNN_Message_Passing(None, k=case["k"], n_ntype=n_ntype, n_etype=n_etype, input_size=case["D"],
                                    hidden_size=case["D"], output_size=case["D"], dropout=0.2)
    missing = mod.load_state_dict(sd, strict=True)
    mod.eval()
    adj = (inp["edge_index"], inp["edge_type"])
    out = mod(inp["H"], adj, inp["node_type"], inp["node_score"])
    # per-layer trace through the reference's own layers (same code path as mp_helper :45-50)
    T = ref.make_one_hot(inp["node_type"].view(-1), n_ntype).view(case["B"], case["n"], n_ntype)
    type_emb = mod.activation(mod.emb_node_type(T))
    js = torch.pow(1.1, torch.arange(case["D"] // 2).unsqueeze(0).unsqueeze(0).float())
    score_emb = mod.activation(mod.emb_score(torch.sin(js * inp["node_score"])))
    extra = torch.cat([type_emb, score_emb], dim=2).view(case["B"] * case["n"], -1).contiguous()
    X = inp["H"].view(-1, case["D"]).contiguous()
    nt = inp["node_type"].view(-1)
    layers = []
    for l in range(case["k"]):
        X, (ei2, alpha) = mod.gnn_layers[l](X, inp["edge_index"], inp["edge_type"], nt, extra,
                                            return_attention_weights=True)
        X = mod.activation(X)
        layers.append({"x": X.clone(), "alpha": alpha.clone()})
    keep = [0, case["k"] - 1] if case["k"] > 1 else [0]
    fx = {
        "kind": "mp", "case": case, "n_ntype": n_ntype, "n_etype": n_etype,
        "input_fp": fingerprint(inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"]),
        "weight_fp": fingerprint(*[sd[k_] for k_ in sorted(sd) if sd[k_].dtype.is_floating_point]),
        "out": out.clone(), "extra": extra.clone(), "edge_index_prime": ei2.clone(),
        "layers": {l: layers[l] for l in keep},
        "state_dict_keys": sorted(mod.state_dict().keys()),
    }
    return fx


@torch.no_grad()
def mint_layer_case(ref, case, n_ntype=4, n_etype=38):
    x, extra, node_type, ei, et = build_layer_inputs(case, n_ntype, n_etype)
    sd = layer_state_dict(case, n_ntype, n_etype)
    D = case["D"]
    enc = torch.nn.Sequential(torch.nn.Linear(n_etype + 1 + n_ntype * 2, D), torch.nn.BatchNorm1d(D),
                              torch.nn.ReLU(), torch.nn.Linear(D, D))
    layer = ref.GATConvE(None, D, n_ntype, n_etype, enc, head_count=case["H"])
    lsd = {k_[len("gnn_layers.0."):]: v for k_, v in sd.items() if k_.startswith("gnn_layers.0.")}
    layer.load_state_dict(lsd, strict=True)
    layer.eval()
    out, (ei2, alpha) = layer(x, ei, et, node_type, extra, return_attention_weights=True)
    return {"kind": "layer", "case": case, "n_ntype": n_ntype, "n_etype": n_etype,
            "input_fp": fingerprint(x, extra, node_type, ei, et),
            "out": out.clone(), "alpha": alpha.clone(), "edge_index_prime": ei2.clone()}


DEC_CASES = [
    dict(name="decoder_small", B=6, n=30, e=80, D=64, k=2, sent_dim=48, n_concept=500, concept_in_dim=32,
         n_head=2, n_fc_layer=0, regime="peaky", seed=20),
    dict(name="decoder_fc1", B=4, n=20, e=50, D=100, k=2, sent_dim=64, n_concept=300, concept_in_dim=100,
         n_head=2, n_fc_layer=1, regime="peaky", seed=21),
]


def build_decoder_inputs(case, n_etype=38):
    inp = O.synth_graph_batch(case["B"], case["n"], case["e"], case["D"], n_etype, case["seed"], realistic=True)
    g = torch.Generator().manual_seed(700 + case["seed"])
    sent_vecs = torch.randn(case["B"], case["sent_dim"], generator=g)
    concept_ids = torch.randint(1, case["n_concept"] + 1, (case["B"], case["n"]), generator=g)
    concept_ids[:, 0] = 0
    for b in range(case["B"]):
        concept_ids[b, int(inp["adj_lengths"][b]):] = 1
    return inp, sent_vecs, concept_ids


def decoder_state_dict(ref_module, case):
    """Random (seeded) values for every tensor of the reference decoder, 'peaky' style."""
    g = torch.Generator().manual_seed(900 + case["seed"])
    gnn_sd = O.random_state_dict(case["k"], case["D"], 4, 38, case["regime"], case["seed"])
    sd = {}
    for key, v in ref_module.state_dict().items():
        if key.startswith("gnn."):
            sd[key] = gnn_sd[key[4:]].clone()
        elif not v.dtype.is_floating_point:
            sd[key] = v.clone()
        elif key.endswith("running_var"):
            sd[key] = 0.5 + torch.rand(v.shape, generator=g)
        elif v.dim() >= 2:
            sd[key] = torch.randn(v.shape, generator=g) * (1.0 / (v.shape[-1] ** 0.5))
        elif "LayerNorm.weight" in key or key.endswith("1.weight"):
            sd[key] = 1 + 0.3 * torch.randn(v.shape, generator=g)
        else:
            sd[key] = 0.1 * torch.randn(v.shape, generator=g)
    return sd


@torch.no_grad()
def mint_decoder_case(ref, case, n_ntype=4, n_etype=38):
    inp, sent_vecs, concept_ids = build_decoder_inputs(case, n_etype)
    dec = ref.QAGNN(None, case["k"], n_ntype, n_etype, case["sent_dim"], case["n_concept"], case["D"],
                    case["concept_in_dim"], case["n_head"], case["D"], case["n_fc_layer"], 0.2, 0.2, 0.2,
                    pretrained_concept_emb=None, freeze_ent_emb=True, init_range=0.02)
    sd = decoder_state_dict(dec, case)
    dec.load_state_dict(sd, strict=True)
    dec.eval()
    logits, pool_attn = dec(sent_vecs, concept_ids, inp["node_type"], inp["node_score"], inp["adj_lengths"],
                            (inp["edge_index"], inp["edge_type"]))
    return {"kind": "decoder", "case": case, "n_ntype": n_ntype, "n_etype": n_etype,
            "state_dict": {k_: v.clone() for k_, v in sd.items()},
            "logits": logits.clone(), "pool_attn": pool_attn.clone(),
            "input_fp": fingerprint(inp["H"], inp["edge_index"], sent_vecs, concept_ids)}


# training-mode cases (SURVEY.md §8f #3): the reference modules in .train() with dropout 0 (the mask stream of a live
# dropout cannot be reproduced), BatchNorm batch statistics, loss = sum(out * G) for a fixed random G, autograd gradients
TRAIN_CASES = [
    dict(name="train_cfg1_peaky_k2", B=4, n=50, e=200, D=64, k=2, regime="peaky", realistic=False, seed=21),
    dict(name="train_tiny_realistic_d100", B=6, n=24, e=60, D=100, k=3, regime="peaky", realistic=True, seed=22),
    dict(name="train_cfg2tiny_prod", B=2, n=200, e=1000, D=200, k=2, regime="prod", realistic=False, seed=23),
]


def train_loss_weights(case):
    g = torch.Generator().manual_seed(9000 + case["seed"])
    return torch.randn(case["B"], case["n"], case["D"], generator=g)


def mint_train_case(ref, case, n_ntype=4, n_etype=38):
    inp = O.synth_graph_batch(case["B"], case["n"], case["e"], case["D"], n_etype, case["seed"], case["realistic"])
    sd = O.random_state_dict(case["k"], case["D"], n_ntype, n_etype, case["regime"], case["seed"])
    mod = ref.QAGNN_Message_Passing(None, k=case["k"], n_ntype=n_ntype, n_etype=n_etype, input_size=case["D"],
                                    hidden_size=case["D"], output_size=case["D"], dropout=0.0)
    mod.load_state_dict(sd, strict=True)
    mod.train()
    H = inp["H"].clone().requires_grad_(True)
    score = inp["node_score"].clone().requires_grad_(True)
    out = mod(H, (inp["edge_index"], inp["edge_type"]), inp["node_type"], score)
    loss = (out * train_loss_weights(case)).sum()
    loss.backward()
    grads = {}
    seen = set()
    for name, p_ in mod.named_parameters():  # named_parameters de-duplicates the shared edge_encoder
        if id(p_) in seen:
            continue
        seen.add(id(p_))
        grads[name] = p_.grad.detach().clone() if p_.grad is not None else None
    buffers = {name: b.detach().clone() for name, b in mod.named_buffers() if "running" in name or "num_batches" in name}
    return {"kind": "train", "case": case, "n_ntype": n_ntype, "n_etype": n_etype,
            "input_fp": fingerprint(inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"]),
            "weight_fp": fingerprint(*[sd[k_] for k_ in sorted(sd) if sd[k_].dtype.is_floating_point]),
            "out": out.detach().clone(), "loss": float(loss), "grad_H": H.grad.clone(), "grad_score": score.grad.clone(),
            "grads": grads, "buffers_after": buffers}


TRAIN_DEC_CASES = [
    dict(name="train_decoder_small", B=6, n=30, e=80, D=64, k=2, sent_dim=48, n_concept=500, concept_in_dim=32,
         n_head=2, n_fc_layer=1, regime="peaky", seed=24),
]


def mint_train_decoder_case(ref, case, n_ntype=4, n_etype=38):
    """The whole reference decoder (`QAGNN`, modeling_qagnn.py:99-189) in .train(): every nn.Dropout of the instance gets
    p = 0 (a live mask stream cannot be reproduced), BatchNorm batch statistics, loss = sum(logits * g), autograd."""
    inp, sent_vecs, concept_ids = build_decoder_inputs(case, n_etype)
    dec = ref.QAGNN(None, case["k"], n_ntype, n_etype, case["sent_dim"], case["n_concept"], case["D"],
                    case["concept_in_dim"], case["n_head"], case["D"], case["n_fc_layer"], 0.0, 0.0, 0.0,
                    pretrained_concept_emb=None, freeze_ent_emb=True, init_range=0.02)
    sd = decoder_state_dict(dec, case)
    dec.load_state_dict(sd, strict=True)
    dec.train()
    for m in dec.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    dec.gnn.dropout_rate = 0.0
    sv = sent_vecs.clone().requires_grad_(True)
    logits, pool_attn = dec(sv, concept_ids, inp["node_type"], inp["node_score"], inp["adj_lengths"],
                            (inp["edge_index"], inp["edge_type"]))
    g = torch.Generator().manual_seed(9100 + case["seed"])
    w = torch.randn(logits.shape, generator=g)
    loss = (logits * w).sum()
    loss.backward()
    grads, seen = {}, set()
    for name, p_ in dec.named_parameters():
        if id(p_) in seen:
            continue
        seen.add(id(p_))
        grads[name] = p_.grad.detach().clone() if p_.grad is not None else None
    return {"kind": "train_decoder", "case": case, "n_ntype": n_ntype, "n_etype": n_etype,
            "state_dict": {k_: v.clone() for k_, v in sd.items()}, "logits": logits.detach().clone(),
            "pool_attn": pool_attn.detach().clone(), "loss_weights": w, "loss": float(loss.detach()),
            "grad_sent": sv.grad.clone(), "grads": grads,
            "input_fp": fingerprint(inp["H"], inp["edge_index"], sent_vecs, concept_ids)}


def _max_diff(a, b, path=""):
    """Largest absolute difference between two fixtures (nested dicts / lists of tensors and scalars); raises on a
    structural mismatch."""
    if isinstance(a, dict):
        assert isinstance(b, dict) and a.keys() == b.keys(), f"{path}: keys differ"
        return max([_max_diff(a[k_], b[k_], f"{path}.{k_}") for k_ in a] or [0.0])
    if isinstance(a, (list, tuple)):
        assert isinstance(b, (list, tuple)) and len(a) == len(b), f"{path}: lengths differ"
        return max([_max_diff(x, y, f"{path}[{i}]") for i, (x, y) in enumerate(zip(a, b))] or [0.0])
    if torch.is_tensor(a):
        assert torch.is_tensor(b) and a.shape == b.shape and a.dtype == b.dtype, f"{path}: tensor meta differs"
        return float((a.double() - b.double()).abs().max()) if a.numel() else 0.0
    if isinstance(a, float):
        return abs(a - b)
    assert a == b, f"{path}: {a!r} != {b!r}"
    return 0.0


def all_cases():
    return ([(mint_mp_case, c) for c in MP_CASES] + [(mint_layer_case, c) for c in LAYER_CASES] +
            [(mint_train_case, c) for c in TRAIN_CASES] + [(mint_train_decoder_case, c) for c in TRAIN_DEC_CASES] +
            [(mint_decoder_case, c) for c in DEC_CASES])


def check(names=None):
    """Re-mints every fixture (or those in `names`) from the reference in memory and returns {name: max |diff|} against the
    committed file — nothing is written.  0.0 everywhere = the fixtures are what the reference's own modules produce here."""
    torch.set_num_threads(8)
    ref = load_reference()
    out = {}
    for mint, case in all_cases():
        if names is not None and case["name"] not in names:
            continue
        have = torch.load(os.path.join(GOLDEN_DIR, case["name"] + ".pt"), weights_only=False)
        out[case["name"]] = _max_diff(mint(ref, case), have, case["name"])
    return out


FUZZ_TOL = (2e-6, 2e-5)  # abs, rel: the oracle and the reference run the same fp32 op sequence


def fuzz_cases(count):
    """Random small cases outside the fixture table (1-4 graphs, 1-30 nodes, 0-80 edges, D 16-100, k 1-3, 6 / 17 / 38 edge
    types, both weight regimes); the i-th case is the same for every `count`."""
    g = torch.Generator().manual_seed(12345)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))  # noqa: E731
    cases = []
    for i in range(count):
        n = ri(1, 30)
        R = (38, 38, 6, 17)[ri(0, 3)]
        cases.append(dict(name=f"fuzz{i}", B=ri(1, 4), n=n, e=ri(0, 80), D=(16, 32, 64, 100)[ri(0, 3)], k=ri(1, 3),
                          regime=("prod", "peaky")[ri(0, 1)], realistic=bool(ri(0, 1)) and n >= 8 and R >= 6, seed=100 + i,
                          n_etype=R))
    return cases


def _fuzz_compared(fx):
    """The tensors a fuzz case compares, by name: output, node_feature_extra, x and attention of the first / last layer."""
    out = {"out": fx["out"], "extra": fx["extra"]}
    for l, layer in fx["layers"].items():
        out[f"x[{l}]"], out[f"alpha[{l}]"] = layer["x"], layer["alpha"]
    return out


def fuzz_oracle(case):
    """The oracle's side of a fuzz case: (input fingerprint, weight fingerprint, {name: tensor} as _fuzz_compared)."""
    R = case["n_etype"]
    inp = O.synth_graph_batch(case["B"], case["n"], case["e"], case["D"], R, case["seed"], case["realistic"])
    sd = O.random_state_dict(case["k"], case["D"], 4, R, case["regime"], case["seed"])
    out, extra, layers = O.message_passing_forward(sd, inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"],
                                                   inp["node_score"], case["k"], 4, R, return_layers=True)
    keep = [0, case["k"] - 1] if case["k"] > 1 else [0]
    fx = {"out": out, "extra": extra, "layers": {l: layers[l] for l in keep}}
    return (fingerprint(inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"], inp["node_score"]),
            fingerprint(*[sd[k_] for k_ in sorted(sd) if sd[k_].dtype.is_floating_point]), _fuzz_compared(fx))


def _excess(a, b, tol_abs, tol_rel):
    return float(((a - b).abs() - tol_abs - tol_rel * b.abs()).max()) if a.numel() else -tol_abs


def fuzz(count, tol_abs=FUZZ_TOL[0], tol_rel=FUZZ_TOL[1]):
    """The reference's own QAGNN_Message_Passing against the oracle on `count` fuzz cases, every element compared.  Returns
    [(case, worst excess over the tolerance)]; excess <= 0 means inside `tol_abs + tol_rel*|ref|`."""
    torch.set_num_threads(8)
    ref = load_reference()
    results = []
    for case in fuzz_cases(count):
        want = _fuzz_compared(mint_mp_case(ref, case, 4, case["n_etype"]))
        got = fuzz_oracle(case)[2]
        results.append((case, max(_excess(got[k_], want[k_], tol_abs, tol_rel) for k_ in want)))
    return results


# ---------------------------------------------------------------------------------------------
# what the reference produced, stored for the tests (`--record`): content digests where the tests compare bit for bit,
# a seeded sample of every compared tensor where they compare within a tolerance
# ---------------------------------------------------------------------------------------------
DIGEST_FILE = os.path.join(GOLDEN_DIR, "reference_digests.json")
FUZZ_FILE = os.path.join(GOLDEN_DIR, "fuzz_mp_sampled.pt")
FUZZ_COUNT = 24
FUZZ_SAMPLES = 128  # entries kept per compared tensor
LOADER_CASE = dict(n_records=20, seed=4, num_choice=5)
LOADER_FIELDS = ("concept_ids", "node_type_ids", "node_scores", "adj_lengths", "edge_index", "edge_type")


def digest(obj):
    """sha256 over nested dicts / lists / tuples of tensors and scalars.  Equal digests: same structure, and every tensor
    has the same dtype, shape and bits (lists and tuples count as the same)."""
    h = hashlib.sha256()

    def walk(o):
        if isinstance(o, dict):
            h.update(b"{")
            for k_ in sorted(o, key=repr):
                h.update(repr(k_).encode())
                walk(o[k_])
            h.update(b"}")
        elif isinstance(o, (list, tuple)):
            h.update(b"[%d" % len(o))
            for x in o:
                walk(x)
            h.update(b"]")
        elif torch.is_tensor(o):
            t = o.detach().contiguous().cpu()
            h.update(f"T{t.dtype}{tuple(t.shape)}".encode())
            h.update(t.numpy().tobytes())
        else:
            h.update(repr(o).encode())
    walk(obj)
    return h.hexdigest()


def records_digest(records):
    """Digest of the content of `*.graph.adj.pk` records (qagnn_b200.data.synth_adj_pickle)."""
    import numpy as np
    return digest([[torch.from_numpy(r["adj"].row.astype(np.int64)), torch.from_numpy(r["adj"].col.astype(np.int64)),
                    tuple(r["adj"].shape), torch.from_numpy(np.asarray(r["concepts"], dtype=np.int64)),
                    torch.from_numpy(np.asarray(r["qmask"], dtype=bool)), torch.from_numpy(np.asarray(r["amask"], dtype=bool)),
                    sorted(r["cid2score"].items())] for r in records])


def loader_split(path):
    """Writes the synthetic split the loader comparison reads; returns its records."""
    from qagnn_b200 import data as Dt
    return Dt.synth_adj_pickle(path, LOADER_CASE["n_records"], seed=LOADER_CASE["seed"])


def batch_generator_inputs(path):
    """Inputs of the batch-generator comparison: 10 questions x 5 choices of a synthetic split, batch size 4 (a partial last
    batch).  Returns the generator's positional and keyword arguments (adj_data excluded) and the nested adjacency."""
    from qagnn_b200 import data as Dt
    n, nc, bs = 40, 5, 4
    Dt.synth_adj_pickle(path, 50, seed=2, max_nodes=60)
    cids, ntypes, scores, lens, (ei, et) = Dt.load_sparse_adj_data_with_contextnode(path, n, nc, None, use_cache=False,
                                                                                   write_cache=False)
    Q = cids.size(0)
    qids = [f"q{i}" for i in range(Q)]
    labels = torch.arange(Q) % nc
    lm = torch.arange(Q * nc * 7).view(Q, nc, 7)
    indexes = torch.randperm(Q, generator=torch.Generator().manual_seed(0))

    class Args:
        drop_partial_batch = False
        fill_partial_batch = False
    return dict(n=n, bs=bs, Q=Q, args=(Args(), "eval", "cpu", "cpu", bs, indexes, qids, labels),
                kw=dict(tensors0=[lm], tensors1=[cids, ntypes, scores, lens]), ei=ei, et=et)


def batch_generator_input_digest(case):
    return digest([case["args"][5:], case["kw"]["tensors0"], case["kw"]["tensors1"], case["ei"], case["et"]])


def fuzz_sample_index(numel, seed):
    """Flat indices of the entries of a compared tensor that FUZZ_FILE keeps (all of them for small tensors)."""
    if numel <= FUZZ_SAMPLES:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:FUZZ_SAMPLES].sort().values


def fuzz_check_stored(stored, samples, tol_abs=FUZZ_TOL[0], tol_rel=FUZZ_TOL[1]):
    """The oracle against one stored fuzz case (`samples`: FUZZ_FILE's flat tensor of sampled entries): the sampled entries
    within `tol_abs + tol_rel*|ref|`, and every tensor's sum within the sum of those bounds (which the element-wise bound
    implies).  Returns the worst excess; <= 0 passes."""
    in_fp, w_fp, got = fuzz_oracle(stored["case"])
    assert in_fp == stored["input_fp"] and w_fp == stored["weight_fp"], "regenerated fuzz inputs differ from the recorded ones"
    assert sorted(got) == sorted(stored["tensors"]), "compared tensors differ from the recorded ones"
    worst = -tol_abs
    for i, (name, want) in enumerate(sorted(stored["tensors"].items())):
        a = got[name].detach().double()
        assert tuple(a.shape) == want["shape"], name
        idx = fuzz_sample_index(a.numel(), stored["case"]["seed"] * 16 + i)
        sample = samples[want["offset"]:want["offset"] + idx.numel()].double()
        worst = max(worst, _excess(a.reshape(-1)[idx], sample, tol_abs, tol_rel))
        worst = max(worst, abs(float(a.sum()) - want["sum"]) - a.numel() * tol_abs - tol_rel * want["abs_sum"])
    return worst


def record():
    """Runs the reference where the tests compare against it and stores what it produced: DIGEST_FILE (every committed
    fixture re-minted in memory; the reference's adjacency loader and batch generator) and FUZZ_FILE."""
    import pickle
    import tempfile
    from oracle.ref_shim import load_reference_data_utils
    torch.set_num_threads(8)
    ref = load_reference()
    RD = load_reference_data_utils()
    out = {"fixtures": {case["name"]: digest(mint(ref, case)) for mint, case in all_cases()}, "loader": {}}
    with tempfile.TemporaryDirectory() as tmp:
        for max_node_num in (200, 30):
            path = os.path.join(tmp, f"n{max_node_num}", "dev.graph.adj.pk")
            os.makedirs(os.path.dirname(path))
            records = loader_split(path)
            res = RD.load_sparse_adj_data_with_contextnode(path, max_node_num, LOADER_CASE["num_choice"], None)
            with open(path + ".loaded_cache", "rb") as f:
                cache = pickle.load(f)
            entry = {"input": records_digest(records), "cache": digest(cache)}
            entry.update({name: digest(v) for name, v in zip(LOADER_FIELDS, res[:4] + tuple(res[4]))})
            out["loader"][str(max_node_num)] = entry
        case = batch_generator_inputs(os.path.join(tmp, "s.graph.adj.pk"))
        batches = RD.MultiGPUSparseAdjDataBatchGenerator(*case["args"], adj_data=(case["ei"], case["et"]), **case["kw"])
        out["batch_generator"] = {"input": batch_generator_input_digest(case), "batches": [digest(b) for b in batches]}
    with open(DIGEST_FILE, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    cases, samples, offset = [], [], 0
    for case in fuzz_cases(FUZZ_COUNT):
        fx = mint_mp_case(ref, case, 4, case["n_etype"])
        tensors = {}
        for i, (name, t) in enumerate(sorted(_fuzz_compared(fx).items())):
            t = t.detach().double()
            idx = fuzz_sample_index(t.numel(), case["seed"] * 16 + i)
            samples.append(t.reshape(-1)[idx].float())
            tensors[name] = {"shape": tuple(t.shape), "offset": offset, "sum": float(t.sum()), "abs_sum": float(t.abs().sum())}
            offset += idx.numel()
        cases.append({"case": case, "input_fp": fx["input_fp"], "weight_fp": fx["weight_fp"], "tensors": tensors})
    torch.save({"kind": "mp_fuzz", "tol": FUZZ_TOL, "cases": cases, "samples": torch.cat(samples)}, FUZZ_FILE)


def reference_digests():
    with open(DIGEST_FILE) as f:
        return json.load(f)


def main():
    if "--record" in sys.argv[1:]:
        record()
        print("wrote", DIGEST_FILE, "and", FUZZ_FILE)
        return
    if "--fuzz" in sys.argv[1:]:
        count = int(sys.argv[sys.argv.index("--fuzz") + 1])
        bad = 0
        for case, worst in fuzz(count):
            print(f"{case}: {'inside' if worst <= 0 else 'OUTSIDE'} the tolerance (excess {worst:.3g})")
            bad += worst > 0
        sys.exit(1 if bad else 0)
    if "--check" in sys.argv[1:]:
        worst = 0.0
        for name, diff in check().items():
            print(f"{name}: max |re-minted - committed| = {diff:.3g}")
            worst = max(worst, diff)
        sys.exit(0 if worst == 0.0 else 1)
    torch.set_num_threads(8)
    ref = load_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    for mint, case in all_cases():
        fx = mint(ref, case)
        torch.save(fx, os.path.join(GOLDEN_DIR, case["name"] + ".pt"))
        print("minted", case["name"], fx.get("kind"))


if __name__ == "__main__":
    main()
