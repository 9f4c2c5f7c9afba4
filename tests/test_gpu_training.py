"""Training mode of the CUDA path (SURVEY.md §8f #3): forward with BatchNorm batch statistics and the gradients of every
parameter and input against goldens minted from the reference's own modules in .train() with autograd
(oracle/make_goldens.py: mint_train_case; dropout 0 because a live mask stream cannot be reproduced).  Needs a GPU."""
import pytest
import torch

import qagnn_b200
from oracle import make_goldens as MG
from tests import helpers as Hh

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _module(fx, sd, dropout=0.0):
    c = fx["case"]
    mod = qagnn_b200.QAGNN_Message_Passing(None, c["k"], fx["n_ntype"], fx["n_etype"], c["D"], c["D"], c["D"], dropout=dropout)
    mod.load_state_dict(sd, strict=True)
    return mod.to(DEV)


def _grad_close(got, ref, what, floor=0.0):
    # gradients span orders of magnitude across parameters: 1e-4 relative to the tensor's own scale, plus 1e-4 relative.
    # `floor`: a gradient that is mathematically zero (the bias in front of a BatchNorm) is pure rounding noise in both
    # implementations; it is compared on the scale of the largest gradient of the model instead of its own
    scale = max(float(ref.abs().max()), floor, 1e-6)
    Hh.assert_close(got, ref, what, atol=1e-4 * scale, rtol=1e-4)


@pytest.mark.parametrize("name", Hh.golden_names("train"))
def test_training_forward_and_gradients_match_reference(name):
    fx = Hh.load_golden(name)
    c = fx["case"]
    inp, sd = Hh.regen_mp_inputs(fx)
    mod = _module(fx, sd).train()
    H = inp["H"].to(DEV).requires_grad_(True)
    score = inp["node_score"].to(DEV).requires_grad_(True)
    out = mod(H, (inp["edge_index"].to(DEV), inp["edge_type"].to(DEV)), inp["node_type"].to(DEV), score)
    Hh.assert_close(out, fx["out"], "train-mode out")
    loss = (out * MG.train_loss_weights(c).to(DEV)).sum()
    loss.backward()
    assert abs(float(loss) - fx["loss"]) <= 1e-3 + 1e-4 * abs(fx["loss"])
    _grad_close(H.grad, fx["grad_H"], "dL/dH")
    _grad_close(score.grad, fx["grad_score"], "dL/dscore")
    got = dict(mod.named_parameters())
    assert sorted(got) == sorted(fx["grads"]), "parameter names (shared edge_encoder de-duplicated) differ from the reference"
    gmax = max(float(g.abs().max()) for g in fx["grads"].values() if g is not None)
    for pname, ref_g in fx["grads"].items():
        assert got[pname].grad is not None, pname
        _grad_close(got[pname].grad, ref_g, f"dL/d{pname}", floor=1e-2 * gmax)
    bufs = dict(mod.named_buffers())
    for bname, ref_b in fx["buffers_after"].items():
        if "num_batches" in bname:
            assert int(bufs[bname]) == int(ref_b), bname
        else:
            Hh.assert_close(bufs[bname], ref_b, bname, atol=1e-5, rtol=1e-4)


def test_train_then_eval_uses_updated_weights_and_statistics():
    """An optimiser step and the BatchNorm running-statistics update must invalidate the folded eval-mode weights."""
    fx = Hh.load_golden("train_cfg1_peaky_k2")
    inp, sd = Hh.regen_mp_inputs(fx)
    mod = _module(fx, sd)
    d = {k: v.to(DEV) for k, v in inp.items()}
    args = (d["H"], (d["edge_index"], d["edge_type"]), d["node_type"], d["node_score"])
    before = mod.eval()(*args).clone()
    opt = torch.optim.SGD(mod.parameters(), lr=0.05)
    out = mod.train()(*args)
    out.square().mean().backward()
    opt.step()
    after = mod.eval()(*args)
    assert not torch.allclose(before, after, atol=1e-4), "eval output did not change after a training step"
    # the same weights loaded into a fresh module give the same eval output (nothing stale in the folded cache)
    fresh = _module(fx, {k: v.detach().cpu() for k, v in mod.state_dict().items()}).eval()
    Hh.assert_close(after, fresh(*args).cpu(), "eval after step vs fresh module", atol=1e-6, rtol=1e-6)
    # .data edits do not bump the version counter: invalidate() is the documented way
    with torch.no_grad():
        mod.Vh.weight.data.mul_(0.5)
    mod.invalidate()
    fresh2 = _module(fx, {k: v.detach().cpu() for k, v in mod.state_dict().items()}).eval()
    Hh.assert_close(mod(*args), fresh2(*args).cpu(), "eval after .data edit + invalidate()", atol=1e-6, rtol=1e-6)


def test_dropout_is_applied_in_training_mode_only():
    fx = Hh.load_golden("train_cfg1_peaky_k2")
    inp, sd = Hh.regen_mp_inputs(fx)
    mod = _module(fx, sd, dropout=0.5).train()
    d = {k: v.to(DEV) for k, v in inp.items()}
    args = (d["H"], (d["edge_index"], d["edge_type"]), d["node_type"], d["node_score"])
    torch.manual_seed(0)
    a = mod(*args)
    b = mod(*args)
    zero_frac = float((a == 0).float().mean())
    assert 0.4 < zero_frac < 0.6, f"final dropout (modeling_qagnn.py:93) should zero ~half of the outputs, got {zero_frac}"
    assert not torch.equal(a, b), "two training-mode forwards must draw different dropout masks"
    e1, e2 = mod.eval()(*args), mod.eval()(*args)
    assert torch.equal(e1, e2) and float((e1 == 0).float().mean()) < 0.01


def _hub_graph_batch(D, seed):
    """One 200-node graph in which node 3 is the source of 600 edges and node 8 the target of 600 more."""
    g = torch.Generator().manual_seed(seed)
    n = 200
    ei = torch.randint(0, n, (2, 1400), generator=g)
    ei[0, :600] = 3
    ei[1, 600:1200] = 8
    nt = torch.randint(0, 3, (1, n), generator=g)
    nt[0, 0] = 3
    return {"H": torch.randn(1, n, D, generator=g) * 0.5, "edge_index": ei, "edge_type": torch.randint(0, 38, (1400,), generator=g),
            "node_type": nt}


def _single_layer_training_check(D, Hd, graph):
    """GATConvE alone in .train(): out, alpha and the gradients of x / extra / every parameter vs autograd through the CPU
    oracle's op-for-op restatement with batch statistics, evaluated in fp64 (the oracle is differentiable: it is written in
    torch ops)."""
    from oracle import qagnn_oracle as O
    T, R = 4, 38
    inp = O.synth_graph_batch(3, 30, 90, D, R, seed=31) if graph == "random" else _hub_graph_batch(D, seed=31)
    sd = O.random_state_dict(1, D, T, R, "peaky", seed=31)
    x = inp["H"].view(-1, D).clone().requires_grad_(True)
    g0 = torch.Generator().manual_seed(5)
    extra = (torch.randn(x.shape, generator=g0) * 0.5).requires_grad_(True)
    nt = inp["node_type"].view(-1)
    ref_params = {k_[len("gnn_layers.0."):]: v.requires_grad_(True) for k_, v in sd.items()
                  if k_.startswith("gnn_layers.0.") and v.is_floating_point() and "running_" not in k_}
    ref_out, _, ref_alpha, _ = O.gatconve_forward(sd, "gnn_layers.0", x, inp["edge_index"], inp["edge_type"], nt, extra, T, R,
                                                  head_count=Hd, dtype=torch.float64, train=True)
    G = torch.randn(ref_out.shape, generator=g0)
    (ref_out * G.double()).sum().backward()
    enc = torch.nn.Sequential(torch.nn.Linear(R + 1 + 2 * T, D), torch.nn.BatchNorm1d(D), torch.nn.ReLU(), torch.nn.Linear(D, D))
    layer = qagnn_b200.GATConvE(None, D, T, R, enc, head_count=Hd)
    layer.load_state_dict({k_[len("gnn_layers.0."):]: v.detach() for k_, v in sd.items() if k_.startswith("gnn_layers.0.")})
    layer = layer.to(DEV).train()
    xg = x.detach().to(DEV).requires_grad_(True)
    eg = extra.detach().to(DEV).requires_grad_(True)
    out, (_, alpha) = layer(xg, inp["edge_index"].to(DEV), inp["edge_type"].to(DEV), nt.to(DEV), eg, return_attention_weights=True)
    Hh.assert_close(out, ref_out.detach(), "train-mode GATConvE out")
    Hh.assert_close(alpha, ref_alpha.detach(), "alpha")
    (out * G.to(DEV)).sum().backward()
    _grad_close(xg.grad, x.grad, "dL/dx")
    _grad_close(eg.grad, extra.grad, "dL/dextra")
    got = dict(layer.named_parameters())
    assert sorted(got) == sorted(ref_params)
    gmax = max(float(p.grad.abs().max()) for p in ref_params.values())
    for pname, ref_p in ref_params.items():
        # floor: the biases in front of a BatchNorm have a mathematically zero gradient (rounding noise in both)
        _grad_close(got[pname].grad, ref_p.grad, f"dL/d{pname}", floor=1e-2 * gmax)


def test_single_layer_training_gradients_against_autograd_of_the_oracle():
    """D = 64, H = 4 on a batch of three random 30-node graphs."""
    _single_layer_training_check(64, 4, "random")


@pytest.mark.parametrize("D,Hd,graph", [(64, 1, "random"), (128, 2, "random"), (1024, 8, "random"), (256, 16, "random"),
                                        (64, 4, "hub"), (256, 16, "hub")])
def test_single_layer_training_gradients_at_every_head_count(D, Hd, graph):
    """The same check at H = 1, 2, 8, 16 and on a graph with 600-edge source / target hubs: the wiring around the
    message-passing kernels (per-head 1/sqrt(d), the node / edge halves of the key and msg weights) for every head count."""
    _single_layer_training_check(D, Hd, graph)


def test_whole_decoder_training_step_matches_reference():
    """`QAGNN` (input assembly + message passing + pooling + answer MLP, modeling_qagnn.py:99-189) in .train(): logits, loss and
    every gradient against the reference's own decoder run under autograd (oracle/make_goldens.py: mint_train_decoder_case)."""
    fx = Hh.load_golden("train_decoder_small")
    c = fx["case"]
    inp, sent_vecs, concept_ids = MG.build_decoder_inputs(c, fx["n_etype"])
    dec = qagnn_b200.QAGNN(None, c["k"], fx["n_ntype"], fx["n_etype"], c["sent_dim"], c["n_concept"], c["D"], c["concept_in_dim"],
                           c["n_head"], c["D"], c["n_fc_layer"], 0.0, 0.0, 0.0)
    dec.load_state_dict(fx["state_dict"], strict=True)
    dec = dec.to(DEV).train()
    for m in dec.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    dec.gnn.dropout_rate = 0.0
    sv = sent_vecs.to(DEV).requires_grad_(True)
    logits, pool_attn = dec(sv, concept_ids.to(DEV), inp["node_type"].to(DEV), inp["node_score"].to(DEV), inp["adj_lengths"].to(DEV),
                            (inp["edge_index"].to(DEV), inp["edge_type"].to(DEV)))
    Hh.assert_close(logits, fx["logits"], "train-mode logits")
    Hh.assert_close(pool_attn, fx["pool_attn"], "train-mode pool_attn")
    loss = (logits * fx["loss_weights"].to(DEV)).sum()
    loss.backward()
    assert abs(float(loss.detach()) - fx["loss"]) <= 1e-3 + 1e-4 * abs(fx["loss"])
    _grad_close(sv.grad, fx["grad_sent"], "dL/dsent_vecs")
    got = dict(dec.named_parameters())
    assert sorted(got) == sorted(fx["grads"])
    gmax = max(float(g.abs().max()) for g in fx["grads"].values() if g is not None)
    for pname, ref_g in fx["grads"].items():
        if ref_g is None:  # frozen entity embedding (freeze_ent_emb=True)
            assert got[pname].grad is None, pname
            continue
        assert got[pname].grad is not None, pname
        _grad_close(got[pname].grad, ref_g, f"dL/d{pname}", floor=1e-2 * gmax)


def test_training_step_under_fp16_autocast_and_grad_scaler():
    """qagnn.py:91,249-278 with --fp16: forward under autocast, scaled backward, optimiser step.  The CUDA message passing keeps
    fp32 inside (custom_fwd cast), the dense layers run in half: finite loss / gradients, output close to the fp32 forward."""
    fx = Hh.load_golden("train_cfg1_peaky_k2")
    inp, sd = Hh.regen_mp_inputs(fx)
    mod = _module(fx, sd).train()
    d = {k: v.to(DEV) for k, v in inp.items()}
    args = (d["H"], (d["edge_index"], d["edge_type"]), d["node_type"], d["node_score"])
    ref = mod(*args).detach()
    opt = torch.optim.SGD(mod.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda")
    with torch.autocast("cuda", dtype=torch.float16):
        out = mod(*args)
        loss = out.float().square().mean()
    scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    assert torch.isfinite(loss) and all(p.grad is None or torch.isfinite(p.grad).all() for p in mod.parameters())
    assert float((out.float() - ref).abs().max()) < 5e-2 * max(1.0, float(ref.abs().max()))


def test_lm_qagnn_training_step_runs_end_to_end():
    """The whole LM_QAGNN (tiny random-init RoBERTa + decoder) in .train(): cross-entropy over the choices, backward, one
    optimiser step — the loop body of qagnn.py:249-278 with this package's classes."""
    from transformers import RobertaConfig
    torch.manual_seed(0)
    cfg = RobertaConfig(vocab_size=100, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
                        max_position_embeddings=40)
    bs, nc, n, D, k = 2, 5, 20, 64, 2
    model = qagnn_b200.LM_QAGNN(None, "roberta-large", k, 4, 38, n_concept=50, concept_dim=D, concept_in_dim=32, n_attention_head=2,
                                fc_dim=D, n_fc_layer=0, p_emb=0.1, p_gnn=0.1, p_fc=0.1, init_range=0.02,
                                encoder_config={"config": cfg}).to(DEV).train()
    from oracle import qagnn_oracle as O
    g = torch.Generator().manual_seed(1)
    inp = O.synth_graph_batch(bs * nc, n, 40, D, 38, seed=2, realistic=True)
    ei, et = [], []
    for q in range(bs):
        ei.append([]); et.append([])
        for c in range(nc):
            gi = q * nc + c
            sel = (inp["edge_index"][0] >= gi * n) & (inp["edge_index"][0] < (gi + 1) * n)
            ei[-1].append((inp["edge_index"][:, sel] - gi * n).to(DEV)); et[-1].append(inp["edge_type"][sel].to(DEV))
    lm = [torch.randint(3, 90, (bs, nc, 12), generator=g).to(DEV), torch.ones(bs, nc, 12, dtype=torch.long, device=DEV),
          torch.zeros(bs, nc, 12, dtype=torch.long, device=DEV), torch.zeros(bs, nc, 12, dtype=torch.long, device=DEV)]
    concept_ids = torch.randint(1, 51, (bs, nc, n), generator=g)
    concept_ids[..., 0] = 0
    dec = [concept_ids.to(DEV), inp["node_type"].view(bs, nc, n).to(DEV), inp["node_score"].view(bs, nc, n, 1).to(DEV),
           inp["adj_lengths"].view(bs, nc).to(DEV)]
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-3)
    labels = torch.tensor([1, 3], device=DEV)
    before = model.decoder.gnn.gnn_layers[0].linear_key.weight.detach().clone()
    logits, _ = model(*lm, *dec, ei, et)
    assert logits.shape == (bs, nc) and logits.requires_grad
    loss = torch.nn.functional.cross_entropy(logits, labels)
    loss.backward()
    opt.step()
    assert torch.isfinite(loss)
    assert model.decoder.gnn.gnn_layers[0].linear_key.weight.grad is not None
    assert not torch.equal(before, model.decoder.gnn.gnn_layers[0].linear_key.weight.detach())
    with torch.no_grad():  # and the eval path sees the updated weights
        model.eval()
        logits_eval, _ = model(*lm, *dec, ei, et)
    assert torch.isfinite(logits_eval).all()
