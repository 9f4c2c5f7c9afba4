"""Pins oracle/qagnn_oracle.py against every golden vector minted from the reference's own
modules (tests/golden/, made by oracle/make_goldens.py).  CPU only."""
import pytest
import torch

from oracle import qagnn_oracle as O
from tests import helpers as Hh

# the oracle and the reference run the same fp32 op sequence on the same CPU: they agree to
# rounding noise, far inside the 1e-4 parity bar
TIGHT = dict(atol=2e-6, rtol=2e-5)


@pytest.mark.parametrize("name", Hh.golden_names("mp"))
def test_oracle_matches_reference_message_passing(name):
    fx = Hh.load_golden(name)
    c = fx["case"]
    inp, sd = Hh.regen_mp_inputs(fx)
    out, extra, layers = O.message_passing_forward(sd, inp["H"], inp["edge_index"], inp["edge_type"],
                                                   inp["node_type"], inp["node_score"], c["k"], fx["n_ntype"],
                                                   fx["n_etype"], return_layers=True)
    Hh.assert_close(extra, fx["extra"], "node_feature_extra", **TIGHT)
    for l, ref_l in fx["layers"].items():
        Hh.assert_close(layers[l]["alpha"], ref_l["alpha"], f"alpha[{l}]", **TIGHT)
        Hh.assert_close(layers[l]["x"], ref_l["x"], f"x[{l}]", atol=2e-5, rtol=1e-4)
    Hh.assert_close(out, fx["out"], "out", atol=2e-5, rtol=1e-4)
    # integer side: edge_index' (self loops appended after the real edges) is bit-exact
    prep = O.graph_prep_oracle(inp["edge_index"], inp["edge_type"], inp["node_type"], fx["n_ntype"], fx["n_etype"])
    assert torch.equal(torch.from_numpy(prep["src"]), fx["edge_index_prime"][0])
    assert torch.equal(torch.from_numpy(prep["tgt"]), fx["edge_index_prime"][1])


@pytest.mark.parametrize("name", Hh.golden_names("layer"))
def test_oracle_matches_reference_gatconve(name):
    fx = Hh.load_golden(name)
    c = fx["case"]
    x, extra, node_type, ei, et, sd = Hh.regen_layer_inputs(fx)
    out, ei2, alpha, _ = O.gatconve_forward(sd, "gnn_layers.0", x, ei, et, node_type, extra, fx["n_ntype"],
                                            fx["n_etype"], head_count=c["H"])
    assert torch.equal(ei2, fx["edge_index_prime"])
    Hh.assert_close(alpha, fx["alpha"], "alpha", **TIGHT)
    Hh.assert_close(out, fx["out"], "out", atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("name", Hh.golden_names("decoder"))
def test_oracle_matches_reference_decoder(name):
    from oracle import make_goldens as MG
    fx = Hh.load_golden(name)
    c = fx["case"]
    inp, sent_vecs, concept_ids = MG.build_decoder_inputs(c, fx["n_etype"])
    logits, pool_attn, _ = O.qagnn_decoder_forward(fx["state_dict"], sent_vecs, concept_ids, inp["node_type"],
                                                   inp["node_score"], inp["adj_lengths"], inp["edge_index"],
                                                   inp["edge_type"], c["k"], fx["n_ntype"], fx["n_etype"],
                                                   c["n_head"], c["n_fc_layer"])
    Hh.assert_close(pool_attn, fx["pool_attn"], "pool_attn", atol=2e-5, rtol=1e-4)
    Hh.assert_close(logits, fx["logits"], "logits", atol=5e-5, rtol=1e-4)


def test_fp64_oracle_is_the_same_function():
    """fp64 evaluation of the same restatement stays within fp32 noise of the fp32 golden: the
    1e-4 bar is far above the reference's own rounding floor on these cases."""
    fx = Hh.load_golden("cfg2small_peaky")
    c = fx["case"]
    inp, sd = Hh.regen_mp_inputs(fx)
    out64 = O.message_passing_forward(sd, inp["H"], inp["edge_index"], inp["edge_type"], inp["node_type"],
                                      inp["node_score"], c["k"], fx["n_ntype"], fx["n_etype"], dtype=torch.float64)
    Hh.assert_close(out64.float(), fx["out"], "fp64 oracle vs fp32 reference", atol=5e-5, rtol=1e-4)


def test_state_dict_contract():
    """Key names a replacement module must accept (SURVEY.md §8b), incl. the k aliased copies of the
    shared edge encoder."""
    fx = Hh.load_golden("cfg1_peaky_k2")
    keys = fx["state_dict_keys"]
    sd = O.random_state_dict(2, 64)
    assert sorted(sd.keys()) == keys
    assert "gnn_layers.1.edge_encoder.3.weight" in keys and "edge_encoder.3.weight" in keys


def test_committed_goldens_are_what_the_reference_produces_here():
    """Every committed fixture equals, bit for bit, what the reference's own modules produced when it was re-minted in
    memory: tests/golden/reference_digests.json holds one content digest per re-minted fixture
    (`python -m oracle.make_goldens --record`; `--check` redoes the comparison against a reference tree)."""
    import glob
    import os
    from oracle import make_goldens as MG
    want = MG.reference_digests()["fixtures"]
    names = [case["name"] for _, case in MG.all_cases()]
    assert sorted(want) == sorted(names) and len(names) >= 20
    on_disk = {os.path.basename(p)[:-3] for p in glob.glob(os.path.join(Hh.GOLDEN, "*.pt"))}
    assert on_disk == set(names) | {os.path.basename(MG.FUZZ_FILE)[:-3]}
    for name in names:
        assert MG.digest(Hh.load_golden(name)) == want[name], f"{name}: not what the reference produced"


def test_oracle_equals_the_reference_on_uncommitted_random_cases():
    """24 random small cases outside the fixture table (1-4 graphs, 1-30 nodes, 0-80 edges, D 16-100, k 1-3, 6 / 17 / 38 edge
    types, both weight regimes): the oracle against what the reference's own QAGNN_Message_Passing produced, fp32,
    2e-6 + 2e-5 rel, on a seeded sample of every compared tensor and on every tensor's sum — widens the pinned region beyond
    the fixtures (tests/golden/fuzz_mp_sampled.pt from `python -m oracle.make_goldens --record`; `--fuzz 24` compares every
    element against a reference tree)."""
    from oracle import make_goldens as MG
    stored = torch.load(MG.FUZZ_FILE, weights_only=False)
    assert stored["tol"] == MG.FUZZ_TOL and len(stored["cases"]) == MG.FUZZ_COUNT == 24
    assert [c["case"] for c in stored["cases"]] == MG.fuzz_cases(MG.FUZZ_COUNT)
    for c in stored["cases"]:
        worst = MG.fuzz_check_stored(c, stored["samples"])
        assert worst <= 0, f"{c['case']}: outside the tolerance by {worst:.3g}"
