"""CPU: the oracle restatement must reproduce the golden vectors frozen from the reference's model.py."""
import pytest
import torch

from oracle import gnn_oracle as O
from golden_util import TYPES, check_against_golden, golden_batch, golden_params, input_checksum, load, probe


@pytest.mark.parametrize("domain", ["chem", "bio"])
@pytest.mark.parametrize("t", TYPES)
def test_oracle_matches_reference_golden(domain, t):
    torch.set_num_threads(1)
    G = load(domain, t)
    b = golden_batch(domain)
    assert input_checksum(b) == G["input_checksum"], "synthetic generator drifted from the golden inputs"
    P = golden_params(domain, t)
    fwd = O.chem_gnn if domain == "chem" else O.bio_gnn
    with torch.no_grad():
        out_eval = fwd(P, b["x"], b["edge_index"], b["edge_attr"], 5, t, False)
    L = O.leaf_params(P)
    stats = {}
    out_train = fwd(L, b["x"], b["edge_index"], b["edge_attr"], 5, t, True, stats)
    loss = (out_train * probe(out_train.shape, 99)).sum()
    loss.backward()
    grads = {k: v.grad for k, v in L.items() if v.requires_grad}
    bad = check_against_golden(G, out_eval, out_train.detach(), grads, stats)
    assert not bad, bad


def test_oracle_fp64_agrees_with_fp32():
    b = golden_batch("chem")
    P = golden_params("chem", "gin")
    P64 = {k: (v.double() if v.is_floating_point() else v) for k, v in P.items()}
    a = O.chem_gnn(P, b["x"], b["edge_index"], b["edge_attr"], 5, "gin", True)
    c = O.chem_gnn(P64, b["x"], b["edge_index"], b["edge_attr"], 5, "gin", True)
    assert (a.double() - c).abs().max() < 1e-4


def test_segment_mean_golden():
    import numpy as np, os
    G = np.load(os.path.join(os.path.dirname(__file__), "golden", "heads.npz"))
    b = golden_batch("chem")
    rep = probe((b["x"].shape[0], 300), 5)
    assert torch.allclose(O.segment_mean(rep, b["batch"], 4), torch.from_numpy(G["pooled"]), atol=1e-6)


def test_cycle_rows_matches_reference_definition():
    # chem/pretrain_contextpred.py:36-39: arr = arange(num)+shift; arr[-shift:] = arange(shift)
    for num, shift in [(5, 1), (7, 3), (128, 1)]:
        arr = torch.arange(num) + shift
        arr[-shift:] = torch.arange(shift)
        assert torch.equal(arr, O.cycle_rows(num, shift))


@pytest.mark.parametrize("name", sorted(__import__("golden_util").PRETRAINED))
def test_oracle_matches_reference_with_shipped_checkpoint(name):
    """SURVEY.md 8(d) config 1: eval-mode forward with the reference's shipped weights (chem GIN masking.pth at B = 32; the GCN
    checkpoint reaches |x| ~ 190; GAT / GraphSAGE / bio GIN).  Golden = the reference's own model.py on the same checkpoint."""
    import hashlib
    import numpy as np
    import os
    from golden_util import HERE, PRETRAINED, pretrained_batch, pretrained_state_dict
    torch.set_num_threads(1)
    c = PRETRAINED[name]
    G = np.load(os.path.join(HERE, "golden", "pretrained.npz"))
    sd, path = pretrained_state_dict(name)
    if sd is None:
        pytest.skip("the reference's shipped checkpoints are not available (2-11 MB each: not part of the repository)")
    assert bytes(G[name + ":sha256"]) == hashlib.sha256(open(path, "rb").read()).digest(), "staged checkpoint differs"
    b = pretrained_batch(name)
    assert input_checksum(b) == G[name + ":input_checksum"], "synthetic generator drifted from the golden inputs"
    fwd = O.chem_gnn if c["domain"] == "chem" else O.bio_gnn
    with torch.no_grad():
        out = fwd(sd, b["x"], b["edge_index"], b["edge_attr"], 5, c["type"], False)
    ref = torch.from_numpy(G[name + ":out_eval"])
    assert bool(((out - ref).abs() <= 1e-4 + 1e-4 * ref.abs()).all()), float((out - ref).abs().max())
