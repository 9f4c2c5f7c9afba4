"""The adjacency loader keeps the reference's input format (utils/data_utils.py:79-197): checked field by field
against what the reference's own loader and batch generator produced (content digests in
tests/golden/reference_digests.json, recorded by `python -m oracle.make_goldens --record`), and against its
structural invariants."""
import pickle

import pytest
import torch

from oracle import make_goldens as MG
from qagnn_b200 import data as Dt


def _equal_nested(a, b):
    return len(a) == len(b) and all(len(x) == len(y) and all(torch.equal(p, q) for p, q in zip(x, y)) for x, y in zip(a, b))


@pytest.mark.parametrize("max_node_num", [200, 30])
def test_loader_matches_reference_loader(tmp_path, max_node_num):
    want = MG.reference_digests()["loader"][str(max_node_num)]
    path = str(tmp_path / "dev.graph.adj.pk")
    records = MG.loader_split(path)
    assert MG.records_digest(records) == want["input"], "the synthetic split differs from the one the reference loaded"
    ours = Dt.load_sparse_adj_data_with_contextnode(path, max_node_num, 5, None, use_cache=False, write_cache=True)
    for name, value in zip(MG.LOADER_FIELDS, ours[:4] + ours[4]):
        assert MG.digest(value) == want[name], name
    # the cache next to the split is the reference's `.loaded_cache`, item for item, and reading it gives the same answer
    with open(path + ".loaded_cache", "rb") as f:
        assert MG.digest(pickle.load(f)) == want["cache"]
    cached = Dt.load_sparse_adj_data_with_contextnode(path, max_node_num, 5, None, use_cache=True)
    for name, value in zip(MG.LOADER_FIELDS, cached[:4] + cached[4]):
        assert MG.digest(value) == want[name], name


def test_loader_invariants_and_packing(tmp_path):
    path = str(tmp_path / "x.graph.adj.pk")
    Dt.synth_adj_pickle(path, 10, seed=1)
    n = 50
    cids, ntypes, scores, lens, (ei, et) = Dt.load_sparse_adj_data_with_contextnode(path, n, 5, None, use_cache=False,
                                                                                   write_cache=False)
    assert cids.shape == (2, 5, n) and ntypes.shape == (2, 5, n) and scores.shape == (2, 5, n, 1) and lens.shape == (2, 5)
    assert (cids[..., 0] == 0).all() and (ntypes[..., 0] == 3).all()
    for q in range(2):
        for c in range(5):
            L = int(lens[q, c]); e, t = ei[q][c], et[q][c]
            assert e.dtype == torch.int64 and e.shape[0] == 2 and e.shape[1] == t.numel() and e.shape[1] % 2 == 0
            assert int(e.max()) < n and (cids[q, c, L:] == 1).all() and (ntypes[q, c, L:] == 2).all()
            half = e.shape[1] // 2  # inverse half = swapped endpoints, relation + 19
            assert torch.equal(e[:, half:], e[:, :half].flip(0)) and torch.equal(t[half:], t[:half] + 19)
    packed = Dt.pack_adj(ei, et, n, pin=False)
    assert packed.edge_index.shape[1] == sum(x.shape[1] for r in ei for x in r)


def _make_split(tmp_path, n_records=30, n=40, nc=5):
    path = str(tmp_path / "s.graph.adj.pk")
    Dt.synth_adj_pickle(path, n_records, seed=2, max_nodes=60)
    return path, Dt.load_sparse_adj_data_with_contextnode(path, n, nc, None, use_cache=False, write_cache=False)


def test_flat_cache_pack_equals_batch_graph_of_the_nested_lists(tmp_path):
    n, nc = 40, 5
    path, (cids, ntypes, scores, lens, (ei, et)) = _make_split(tmp_path, 30, n, nc)
    flat = Dt.FlatAdjCache.from_nested(ei, et, n)
    flat.save(path + ".flat_cache.npz")
    flat2 = Dt.FlatAdjCache.load(path + ".flat_cache.npz")
    for idx in ([0, 1, 2], [5, 1, 3, 3], [4]):
        want = Dt.pack_adj([ei[i] for i in idx], [et[i] for i in idx], n, pin=False)
        for f in (flat, flat2):
            got = f.pack(idx, pin=False)
            assert torch.equal(got.edge_index, want.edge_index) and torch.equal(got.edge_type, want.edge_type)
            assert torch.equal(got.graph_ptr, want.graph_ptr)
            assert got.buf.data_ptr() == got.edge_index.data_ptr()  # one buffer: one host-to-device copy
    # load_flat_adj_cache writes the file once and reuses it
    out = Dt.load_flat_adj_cache(path, n, nc)
    assert isinstance(out[4], Dt.FlatAdjCache) and out[4].n_graphs() == cids.size(0) * nc
    assert torch.equal(out[4].pack([1]).edge_index, Dt.pack_adj([ei[1]], [et[1]], n, pin=False).edge_index)


def test_flat_cache_answers_what_the_reference_dataloader_asks_of_adj_data(tmp_path):
    """LM_QAGNN_DataLoader (modeling_qagnn.py:281-287,307-308) takes len(adj_data[0]) and adj_data[:n_train]."""
    n, nc = 40, 5
    path, (cids, ntypes, scores, lens, (ei, et)) = _make_split(tmp_path, 30, n, nc)
    flat = Dt.FlatAdjCache.from_nested(ei, et, n)
    assert len(flat[0]) == len(ei) == cids.size(0) and len(flat[1]) == len(et)
    head = flat[:4]
    assert head.n_questions() == 4 and len(head[0]) == 4
    for idx in ([0, 3], [2]):
        want = Dt.pack_adj([ei[i] for i in idx], [et[i] for i in idx], n, pin=False)
        got = head.pack(idx, pin=False)
        assert torch.equal(got.edge_index, want.edge_index) and torch.equal(got.edge_type, want.edge_type)
    mid = flat[2:5]
    want = Dt.pack_adj([ei[3]], [et[3]], n, pin=False)
    assert torch.equal(mid.pack([1], pin=False).edge_index, want.edge_index)
    assert flat[6:6].n_questions() == 0
    with pytest.raises(IndexError):
        flat[2]
    with pytest.raises(IndexError):
        flat[::2]


def test_packed_batch_generator_matches_reference_generator(tmp_path):
    want = MG.reference_digests()["batch_generator"]
    case = MG.batch_generator_inputs(str(tmp_path / "s.graph.adj.pk"))
    assert MG.batch_generator_input_digest(case) == want["input"], "the inputs differ from the ones the reference batched"
    n, bs, Q, ei, et = case["n"], case["bs"], case["Q"], case["ei"], case["et"]
    flat = Dt.FlatAdjCache.from_nested(ei, et, n)
    ours = list(Dt.PackedAdjBatchGenerator(*case["args"], adj_data=flat, **case["kw"]))
    nested = list(Dt.PackedAdjBatchGenerator(*case["args"], adj_data=(ei, et), **case["kw"]))
    assert len(ours) == len(nested) == len(want["batches"]) == (Q + bs - 1) // bs
    for bo, bn, wd in zip(ours, nested, want["batches"]):
        assert MG.digest(bn) == wd  # the nested batch is the reference's MultiGPUSparseAdjDataBatchGenerator batch
        assert bo[0] == bn[0] and torch.equal(bo[1], bn[1])
        for x, z in zip(bo[2:-2], bn[2:-2]):
            assert torch.equal(x, z)
        want_packed = Dt.pack_adj(bn[-2], bn[-1], n, pin=False)  # == LM_QAGNN.batch_graph of the reference's nested batch
        assert isinstance(bo[-2], Dt.PackedAdj)
        assert torch.equal(bo[-2].edge_index, want_packed.edge_index) and torch.equal(bo[-1], want_packed.edge_type)


def _batches_equal(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x[0] == y[0]
        for u, v in zip(x[1:-2], y[1:-2]):
            assert torch.equal(u, v)
        if isinstance(x[-2], Dt.PackedAdj):
            assert torch.equal(x[-2].edge_index, y[-2].edge_index) and torch.equal(x[-2].graph_ptr, y[-2].graph_ptr)
            assert torch.equal(x[-1], y[-1])
        else:
            assert _equal_nested(x[-2], y[-2]) and _equal_nested(x[-1], y[-1])


@pytest.mark.parametrize("mode,drop,fill", [("eval", False, False), ("train", True, False), ("train", False, True)])
def test_prefetching_generator_yields_the_same_batches_in_the_same_order(tmp_path, mode, drop, fill):
    import numpy as np
    import threading
    n, nc, bs = 40, 5, 4
    path, (cids, ntypes, scores, lens, (ei, et)) = _make_split(tmp_path, 55, n, nc)  # 11 questions: a partial last batch
    Q = cids.size(0)
    qids = [f"q{i}" for i in range(Q)]
    labels = torch.arange(Q) % nc
    indexes = torch.randperm(Q, generator=torch.Generator().manual_seed(1))

    class Args:
        drop_partial_batch = drop
        fill_partial_batch = fill
    kw = dict(tensors0=[torch.arange(Q * nc).view(Q, nc)], tensors1=[cids, ntypes, scores, lens])
    flat = Dt.FlatAdjCache.from_nested(ei, et, n)
    for adj in (flat, (ei, et)):
        np.random.seed(5)
        plain = list(Dt.PackedAdjBatchGenerator(Args(), mode, "cpu", "cpu", bs, indexes, qids, labels, adj_data=adj, **kw))
        np.random.seed(5)
        ahead = list(Dt.PackedAdjBatchGenerator(Args(), mode, "cpu", "cpu", bs, indexes, qids, labels, adj_data=adj,
                                                prefetch=2, **kw))
        _batches_equal(plain, ahead)
        assert len(plain) == (Q // bs if drop else (Q + bs - 1) // bs)
    # a consumer that stops early does not leave the worker thread behind
    before = threading.active_count()
    it = iter(Dt.PackedAdjBatchGenerator(Args(), "eval", "cpu", "cpu", 2, indexes, qids, labels, adj_data=flat, prefetch=1, **kw))
    next(it)
    it.close()
    assert threading.active_count() == before


def test_prefetching_generator_reraises_worker_errors(tmp_path):
    n, nc = 40, 5
    path, (cids, ntypes, scores, lens, (ei, et)) = _make_split(tmp_path, 20, n, nc)
    Q = cids.size(0)
    bad = torch.tensor([0, 1, Q + 3])  # question Q+3 does not exist

    class Args:
        pass
    gen = Dt.PackedAdjBatchGenerator(Args(), "eval", "cpu", "cpu", 2, bad, [f"q{i}" for i in range(Q + 4)], torch.zeros(Q + 4),
                                     tensors1=[], adj_data=Dt.FlatAdjCache.from_nested(ei, et, n), prefetch=2)
    it = iter(gen)
    next(it)
    with pytest.raises(IndexError):
        next(it)


@pytest.mark.parametrize("seed", range(6))
def test_flat_cache_pack_on_ragged_and_empty_graphs(seed):
    """Random nested adjacency with empty sub-graphs (and, for seed 0, no edges at all): pack == pack_adj of the slice."""
    g = torch.Generator().manual_seed(seed)
    n, nc, Q = 17, 3, 7
    sizes = torch.randint(0, 9, (Q, nc), generator=g)
    if seed == 0:
        sizes.zero_()
    sizes[2] = 0                                            # one question whose choices all have empty graphs
    ei = [[torch.randint(0, n, (2, int(sizes[q, c])), generator=g) for c in range(nc)] for q in range(Q)]
    et = [[torch.randint(0, 38, (int(sizes[q, c]),), generator=g) for c in range(nc)] for q in range(Q)]
    flat = Dt.FlatAdjCache.from_nested(ei, et, n)
    assert flat.n_graphs() == Q * nc and int(flat.graph_ptr[-1]) == int(sizes.sum())
    for idx in ([0], [2], [6, 2, 1], list(range(Q)), [3, 3]):
        want = Dt.pack_adj([ei[i] for i in idx], [et[i] for i in idx], n, pin=False)
        got = flat.pack(idx, pin=False)
        assert torch.equal(got.edge_index, want.edge_index) and torch.equal(got.edge_type, want.edge_type)
        assert torch.equal(got.graph_ptr, want.graph_ptr) and got.edge_index.dtype == torch.long
    sub = flat[1:4]
    assert torch.equal(sub.pack([1], pin=False).graph_ptr, flat.pack([2], pin=False).graph_ptr)
