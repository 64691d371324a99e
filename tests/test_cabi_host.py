"""CPU: the C-ABI library loads, exports every symbol include/pgnn_b200.h declares, validates arguments
without touching a device, and the host-side modules keep the reference's state_dict contract."""
import importlib
import os

import pytest
import torch

from oracle import gnn_oracle as O
from oracle import reference_runner as R

cabi = importlib.import_module("pretrain-gnns_b200._cabi")


def test_library_built_and_exports_header_symbols():
    assert os.path.exists(cabi.LIB_PATH), "run `python pretrain-gnns_b200/build.py`"
    protos = cabi.parse_header()
    assert len(protos) >= 38
    dll = cabi.lib.load()
    for name in protos:
        assert hasattr(dll, name), name
    assert dll.pgnn_version() >= 100
    assert dll.pgnn_error_string(-3) == b"workspace too small"


def test_argument_validation_without_gpu():
    dll = cabi.lib.load()
    assert dll.pgnn_bucket_workspace_bytes(-1, 3) == -1
    assert dll.pgnn_bucket_workspace_bytes(100, 10) > 0
    assert dll.pgnn_linear_fwd(None, 0, None, None, 4, 0, 3, 0, None, 0, 0, None) == -1   # N == 0
    assert dll.pgnn_linear_fwd(None, 0, None, None, 0, 4, 3, 0, None, 0, 0, None) == 0    # M == 0: nothing to do
    assert dll.pgnn_aggregate_fwd(None, 0, None, None, 0, 0, 300, None, None, 0, None, None, 0, None, 0, None, 0, None) == 0
    assert dll.pgnn_aggregate_fwd(None, 0, None, None, 0, 5, 300, None, None, 7, None, None, 0, None, 0, None, 0, None) == -1
    with pytest.raises(cabi.PgnnError):
        cabi.check(-4, "x")


@pytest.mark.parametrize("domain", ["chem", "bio"])
@pytest.mark.parametrize("t", ["gin", "gcn", "graphsage", "gat"])
def test_state_dict_contract(domain, t):
    mod = importlib.import_module(f"pretrain-gnns_b200.{domain}.model")
    model = mod.GNN(5, 300, gnn_type=t)
    P = O.make_params(domain, t, 5, 300, seed=1)
    assert set(model.state_dict().keys()) == set(P.keys())
    for k, v in model.state_dict().items():
        assert tuple(v.shape) == tuple(P[k].shape), k
    assert sum(p.numel() for p in model.parameters()) == {
        ("chem", "gin"): 1857900, ("chem", "gcn"): 504900, ("chem", "graphsage"): 504900, ("chem", "gat"): 977400,
        ("bio", "gin"): 2726100, ("bio", "gcn"): 467100, ("bio", "graphsage"): 467100, ("bio", "gat"): 941100}[(domain, t)]


@pytest.mark.skipif(not os.path.exists(os.path.join(R.REF_SRC, "chem", "model_gin", "masking.pth")),
                    reason="the reference's shipped checkpoints are not available (2-11 MB each: not part of the repository)")
def test_shipped_checkpoints_load():
    import glob
    chem = importlib.import_module("pretrain-gnns_b200.chem.model")
    bio = importlib.import_module("pretrain-gnns_b200.bio.model")
    n = 0
    for mod, dom in ((chem, "chem"), (bio, "bio")):
        for f in sorted(glob.glob(os.path.join(R.REF_SRC, dom, "model_gin", "*.pth"))):
            sd = torch.load(f, map_location="cpu", weights_only=True)
            assert str(mod.GNN(5, 300).load_state_dict(sd)) == "<All keys matched successfully>"
            n += 1
        for f in sorted(glob.glob(os.path.join(R.REF_SRC, dom, "model_architecture", "*.pth"))):
            t = "gcn" if "gcn" in f else "gat" if "gat" in f else "graphsage" if "graphsage" in f else None
            if t is None:
                continue
            sd = torch.load(f, map_location="cpu", weights_only=True)
            assert str(mod.GNN(5, 300, gnn_type=t).load_state_dict(sd)) == "<All keys matched successfully>", f
            n += 1
    assert n >= 18


def test_cpu_forward_fails_loudly():
    chem = importlib.import_module("pretrain-gnns_b200.chem.model")
    g = chem.GNN(5, 300)
    with pytest.raises(cabi.PgnnError):
        g(torch.zeros(3, 2, dtype=torch.long), torch.zeros(2, 0, dtype=torch.long), torch.zeros(0, 2, dtype=torch.long))


def test_constructor_errors():
    chem = importlib.import_module("pretrain-gnns_b200.chem.model")
    bio = importlib.import_module("pretrain-gnns_b200.bio.model")
    for mod in (chem, bio):
        with pytest.raises(ValueError):
            mod.GNN(1, 300)
        with pytest.raises(ValueError):
            mod.GNN_graphpred(1, 300, 3)
        with pytest.raises(ValueError):
            mod.GNN_graphpred(5, 300, 3, graph_pooling="nope")
