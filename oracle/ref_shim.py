"""TEST INFRASTRUCTURE — not product code.

Imports the *unmodified* reference modules from /root/reference (only available in the
build container, never on the GPU box) so that golden vectors can be minted from the
reference's own `GATConvE` / `QAGNN_Message_Passing` / `QAGNN` code.

The reference cannot be imported as-is here because
  * `torch_geometric==1.7.0`, `torch_scatter==2.0.7` (pinned in reference README.md:33-35) are
    not installed and there is no network, and
  * `modeling/modeling_encoder.py:5-6` imports `*_PRETRAINED_CONFIG_ARCHIVE_MAP` symbols that
    transformers >= 4 removed.
This shim registers stand-ins for exactly the third-party entry points the hot path calls
(`modeling/modeling_qagnn.py:371-376`):
  * `torch_geometric.nn.MessagePassing.propagate`  (source_to_target flow, aggr="add")
  * `torch_geometric.utils.softmax`                 (max-subtracted, denominator + 1e-16)
  * `torch_scatter.scatter`                          (reduce in {sum, add, max, mean})
restated from their published semantics (SURVEY.md §8 rows a6-a8).  Everything under
/root/reference then runs verbatim.

Only `oracle/make_goldens.py` calls into this file; the tests read what it recorded under
tests/golden/ and never need the reference tree.
"""
import inspect
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("QAGNN_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "modeling", "modeling_qagnn.py"))


# ----------------------------------------------------------------------------------------------
# torch_scatter.scatter  (2.0.7 semantics: out has size dim_size along `dim`, zeros where empty)
# ----------------------------------------------------------------------------------------------
def _scatter(src, index, dim=-1, out=None, dim_size=None, reduce="sum"):
    if dim < 0:
        dim += src.dim()
    if dim_size is None:
        dim_size = int(index.max()) + 1 if index.numel() > 0 else 0
    shape = list(src.shape)
    shape[dim] = dim_size
    # broadcast index to src's shape along `dim`
    view = [1] * src.dim()
    view[dim] = -1
    idx = index.view(view).expand_as(src)
    if reduce in ("sum", "add"):
        res = torch.zeros(shape, dtype=src.dtype, device=src.device)
        return res.scatter_add_(dim, idx, src)
    if reduce == "mean":
        res = torch.zeros(shape, dtype=src.dtype, device=src.device).scatter_add_(dim, idx, src)
        cnt = torch.zeros(shape, dtype=src.dtype, device=src.device).scatter_add_(dim, idx, torch.ones_like(src))
        return res / cnt.clamp_(min=1)
    if reduce == "max":
        res = torch.full(shape, float("-inf"), dtype=src.dtype, device=src.device)
        res = res.scatter_reduce(dim, idx, src, reduce="amax", include_self=True)
        return torch.where(torch.isinf(res), torch.zeros_like(res), res)
    raise ValueError(reduce)


def _scatter_add(src, index, dim=-1, out=None, dim_size=None):
    return _scatter(src, index, dim, out, dim_size, "sum")


# ----------------------------------------------------------------------------------------------
# torch_geometric.utils.softmax  (1.7.0)
# ----------------------------------------------------------------------------------------------
def _pyg_softmax(src, index, ptr=None, num_nodes=None, dim=0):
    n = int(index.max()) + 1 if num_nodes is None else num_nodes
    smax = _scatter(src, index, dim, dim_size=n, reduce="max")
    out = (src - smax.index_select(dim, index)).exp()
    ssum = _scatter(out, index, dim, dim_size=n, reduce="sum")
    return out / (ssum.index_select(dim, index) + 1e-16)


def _add_self_loops(edge_index, edge_weight=None, fill_value=1.0, num_nodes=None):
    n = int(edge_index.max()) + 1 if num_nodes is None else num_nodes
    loop = torch.arange(n, dtype=torch.long, device=edge_index.device).unsqueeze(0).repeat(2, 1)
    return torch.cat([edge_index, loop], dim=1), edge_weight


def _degree(index, num_nodes=None, dtype=None):
    n = int(index.max()) + 1 if num_nodes is None else num_nodes
    out = torch.zeros(n, dtype=dtype or torch.float, device=index.device)
    return out.scatter_add_(0, index, torch.ones(index.numel(), dtype=out.dtype, device=index.device))


# ----------------------------------------------------------------------------------------------
# torch_geometric.nn.MessagePassing  (1.7.0, only what GATConvE uses: Tensor edge_index,
# tuple x, flow="source_to_target", aggr="add", identity update)
# ----------------------------------------------------------------------------------------------
class _MessagePassing(torch.nn.Module):
    def __init__(self, aggr="add", flow="source_to_target", node_dim=0):
        super().__init__()
        assert aggr in ("add", "mean", "max") and flow == "source_to_target"
        self.aggr, self.flow, self.node_dim = aggr, flow, node_dim

    def propagate(self, edge_index, size=None, **kwargs):
        j, i = edge_index[0], edge_index[1]  # _j <- edge_index[0] (source), _i <- edge_index[1] (target)
        msg_kwargs = {}
        dim_size = None
        for name in inspect.signature(self.message).parameters:
            if name.endswith("_i") or name.endswith("_j"):
                data = kwargs[name[:-2]]
                if isinstance(data, (tuple, list)):
                    data = data[1] if name.endswith("_i") else data[0]
                if name.endswith("_i"):
                    dim_size = kwargs[name[:-2]][1].size(0) if isinstance(kwargs[name[:-2]], (tuple, list)) else data.size(0)
                msg_kwargs[name] = data.index_select(self.node_dim, i if name.endswith("_i") else j)
            elif name == "edge_index":
                msg_kwargs[name] = edge_index
            else:
                msg_kwargs[name] = kwargs[name]
        if dim_size is None:
            first = next(iter(kwargs.values()))
            dim_size = (first[1] if isinstance(first, (tuple, list)) else first).size(0)
        out = self.message(**msg_kwargs)
        reduce = {"add": "sum", "mean": "mean", "max": "max"}[self.aggr]
        return _scatter(out, i, dim=self.node_dim, dim_size=dim_size, reduce=reduce)

    def message(self, x_j):  # pragma: no cover - always overridden
        return x_j


def _install_stubs():
    if "torch_scatter" not in sys.modules:
        m = types.ModuleType("torch_scatter")
        m.scatter, m.scatter_add = _scatter, _scatter_add
        sys.modules["torch_scatter"] = m
    if "torch_geometric" not in sys.modules:
        tg = types.ModuleType("torch_geometric")
        nn_ = types.ModuleType("torch_geometric.nn")
        nn_.MessagePassing = _MessagePassing
        for unused in ("global_add_pool", "global_mean_pool", "global_max_pool", "GlobalAttention", "Set2Set"):
            setattr(nn_, unused, None)
        ut = types.ModuleType("torch_geometric.utils")
        ut.softmax, ut.add_self_loops, ut.degree = _pyg_softmax, _add_self_loops, _degree
        inits = types.ModuleType("torch_geometric.nn.inits")
        inits.glorot = lambda t: None
        inits.zeros = lambda t: None
        tg.nn, tg.utils, nn_.inits = nn_, ut, inits
        sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": nn_,
                            "torch_geometric.utils": ut, "torch_geometric.nn.inits": inits})
    import transformers  # noqa: F401  (lazy module swaps itself into sys.modules on first import)
    from transformers import AutoModel  # noqa: F401
    tr = sys.modules["transformers"]
    for name in ("OPENAI_GPT", "BERT", "XLNET", "ROBERTA", "ALBERT"):
        key = f"{name}_PRETRAINED_CONFIG_ARCHIVE_MAP"
        if key not in tr.__dict__:
            tr.__dict__[key] = {"roberta-large": ""} if name == "ROBERTA" else {}
        try:
            object.__setattr__(tr, key, tr.__dict__[key])
        except Exception:
            pass


_REF = None


def load_reference():
    """Returns the reference's `modeling.modeling_qagnn` module (imported verbatim)."""
    global _REF
    if _REF is not None:
        return _REF
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    _REF = importlib.import_module("modeling.modeling_qagnn")
    return _REF


def load_reference_data_utils():
    """Returns the reference's `utils.data_utils` module (adjacency loader and batch generator, imported verbatim)."""
    if not os.path.isfile(os.path.join(REFERENCE_ROOT, "utils", "data_utils.py")):
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    return importlib.import_module("utils.data_utils")
