"""CPU: the oracle restatement against the reference's OWN model.py / batch.py / util.py.  What the reference's files compute
on the inputs built here is stored in tests/golden/reference_checks.npz (tests/golden/make_golden_reference.py runs them
over the PyG stand-in on exactly these inputs): exact results as digests; float results as golden_util.summary records
(a few elements, the max-norm and a seeded projection), on which the element-wise bound each test states is checked.  Symmetric AND one-direction-only graphs (the direction convention),
every conv type, both domains, heads, the batch collators, the masking transforms and the substructure/context extraction."""
import functools
import importlib

import numpy as np
import pytest
import torch

from golden_util import digest, reference_checks, summary_close
from oracle import gnn_oracle as O
from oracle import step_io_oracle as SO

syn = importlib.import_module("pretrain-gnns_b200.synthetic")
TYPES = ("gin", "gcn", "graphsage", "gat")
NO_CONTEXT = -1   # stands for every digest of an extraction that yields no context graph


@functools.lru_cache(maxsize=1)
def ref():
    return reference_checks()


def ref_prefixed(prefix):
    return {k[len(prefix):]: v for k, v in ref().items() if k.startswith(prefix)}


def assert_digests(prefix, mine):
    for k, v in mine.items():
        assert digest(v) == ref()[prefix + k], k


# ---------------------------------------------------------------------------------------------------------------------
# inputs (make_golden_reference.py builds the reference's side from these same functions)
# ---------------------------------------------------------------------------------------------------------------------
def _batch(domain, directed, seed):
    b = syn.zinc_batch(6, seed) if domain == "chem" else syn.ppi_batch(2, seed, n_lo=30, n_hi=50, num_tasks=8)
    return syn.one_direction_only(b, seed) if directed else b


def fwd_bwd_key(domain, t, directed):
    return "fwd_bwd:%s_%s_%s:" % (domain, t, "directed" if directed else "symmetric")


def graphpred_inputs():
    g = torch.Generator().manual_seed(5)
    out = {}
    for domain, T in (("chem", 12), ("bio", 40)):
        b = _batch(domain, False, 17)
        P = O.make_params(domain, "gin", 5, 300, seed=2)
        full = {"gnn." + k: v for k, v in P.items()}
        width = 300 if domain == "chem" else 600
        full["graph_pred_linear.weight"] = torch.randn(T, width, generator=g) * 0.05
        full["graph_pred_linear.bias"] = torch.randn(T, generator=g) * 0.05
        out[domain] = (T, b, full)
    return out


def collate_masking_inputs():
    graphs = syn.split_graphs(syn.zinc_batch(9, 23))
    return graphs, [3, 0, 8, 8, 5]


def train_body_inputs(config, T=24):
    from oracle import steps_oracle as S
    ts = importlib.import_module("pretrain-gnns_b200.train_steps")
    if config == "bio_supervised":
        b = {k: v for k, v in syn.ppi_batch(3, 5, n_lo=30, n_hi=50, num_tasks=T).items() if k in ts.BioSupervisedStep.KEYS}
    elif config == "contextpred":
        b = {k: v for k, v in syn.substruct_context_batch(8, 5).items() if k in ts.ContextPredStep.KEYS}
    else:
        mb = syn.mask_atoms(syn.zinc_batch(8, 5), 5)
        b = {k: mb[k] for k in ("x", "edge_index", "edge_attr", "masked_atom_indices")} | {"labels": mb["mask_node_label"][:, 0].contiguous()}
    return b, S.make_params(config, 3, num_tasks=T)


def mask_atoms_inputs():
    b = syn.zinc_batch(7, 41)
    node_off = b["ptr"].numpy()
    return b, syn.split_graphs(b), node_off, SO.mask_atom_choice(node_off, 0.15, seed=12345)


def substruct_context_inputs():
    G = 6
    sub, ctx = syn.zinc_batch(G, 51, n_lo=12, n_hi=22), syn.zinc_batch(G, 52, n_lo=4, n_hi=14, tree_only=True)
    sg, cg = syn.split_graphs(sub), syn.split_graphs(ctx)
    rng = np.random.default_rng(3)
    center = [int(rng.integers(0, len(g[0]))) for g in sg]
    overlap = [sorted(rng.choice(len(g[0]), size=int(rng.integers(1, min(4, len(g[0])) + 1)), replace=False).tolist()) for g in cg]
    return G, sg, cg, center, overlap, [4, 1, 1, 5]


def bio_graphs(pb, count):
    """Per-graph (num_nodes, edge_index, edge_attr) of a ppi_batch, edges local to the graph."""
    ptr = pb["ptr"].numpy()
    ei, ea = pb["edge_index"].numpy(), pb["edge_attr"].numpy()
    owner = np.searchsorted(ptr, ei[0], side="right") - 1
    eptr = np.searchsorted(owner, np.arange(len(ptr)))
    return [(int(ptr[g + 1] - ptr[g]), ei[:, eptr[g]:eptr[g + 1]] - ptr[g], ea[eptr[g]:eptr[g + 1]]) for g in range(count)], eptr


def bio_collate_inputs():
    graphs, _ = bio_graphs(syn.ppi_batch(5, 9, n_lo=20, n_hi=35, num_tasks=4), 5)
    return graphs, [0, 3, 1, 0, 2], [2, 0, 4]


EXTRACT_CHEM_PARAMS = [(5, 4, 7), (2, 1, 3), (1, 0, 2), (0, 0, 1), (3, 3, 3), (2, 5, 3)]


def extract_chem_inputs():
    """(x, edge_index, edge_attr, root) for every extraction of the chem test."""
    rng = np.random.default_rng(7)
    cases = []
    for x, ei, ea in syn.split_graphs(syn.zinc_batch(10, 61)):
        for root in {0, len(x) - 1, int(rng.integers(0, len(x)))}:
            cases.append((x, ei, ea, root))
    return cases


def extract_pairs_batch_inputs():
    graphs = syn.split_graphs(syn.zinc_batch(8, 71))
    ids = [3, 0, 7, 7, 2, 5]
    roots = SO.draw_roots([len(graphs[g][0]) for g in ids], seed=99)
    tiny = (graphs[1][0][:1], np.zeros((2, 0), np.int64), np.zeros((0, 2), np.int64))   # a one-atom molecule: no context -> dropped
    graphs = graphs + [tiny]
    ids, roots = ids[:3] + [8] + ids[3:], np.concatenate([roots[:3], [0], roots[3:]])
    return graphs, ids, roots


def extract_bio_inputs():
    """(num_nodes, edge_index, edge_attr, l1) for every extraction of the bio test: graphs without isolated nodes
    (bio/loader.py:119-142 builds the networkx graph from the edges only: an isolated node would not exist in it and the
    reference raises a KeyError on the overlap map)."""
    graphs, _ = bio_graphs(syn.ppi_batch(3, 19, n_lo=30, n_hi=45, pairs_per_node=2, num_tasks=4), 3)
    cases = []
    for n, e, a in graphs:
        a = a.copy()
        a[0:2, 8] = 1   # a masked pair (bio/util.py:100-102): the round trip through networkx drops the bit
        if len(np.unique(e)) != n:
            continue
        for l1 in (1, 2):
            cases.append((n, e, a, l1))
    return cases


def mask_edges_chem_inputs():
    b = syn.zinc_batch(9, 43)
    node_off = b["ptr"].numpy()
    return b, syn.split_graphs(b), node_off, SO.mask_atom_choice(node_off, 0.15, seed=777)


def mask_edges_bio_inputs():
    pb = syn.ppi_batch(4, 23, n_lo=20, n_hi=35, pairs_per_node=3, num_tasks=4)
    graphs, eptr = bio_graphs(pb, 4)
    return graphs, pb["edge_attr"].numpy(), eptr, SO.mask_edge_choice_bio(eptr, 0.15, seed=31)


def _canon_edges(ei, ea, nodes):
    """Edge multiset in ORIGINAL node ids: sorted rows (u, v, attr...)."""
    rows = [(int(nodes[int(ei[0, j])]), int(nodes[int(ei[1, j])])) + tuple(float(a) for a in np.asarray(ea[j]).ravel()) for j in range(ei.shape[1])]
    return sorted(rows)


# ---------------------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("directed", [False, True])
@pytest.mark.parametrize("domain", ["chem", "bio"])
@pytest.mark.parametrize("t", TYPES)
def test_oracle_equals_reference_fwd_bwd(domain, t, directed):
    torch.set_num_threads(1)
    key = fwd_bwd_key(domain, t, directed)
    b = _batch(domain, directed, 31)
    P = O.make_params(domain, t, 5, 300, seed=8)
    fwd = O.chem_gnn if domain == "chem" else O.bio_gnn
    with torch.no_grad():
        mine_eval = fwd(P, b["x"], b["edge_index"], b["edge_attr"], 5, t, False)
    assert summary_close(mine_eval, ref()[key + "eval"], 2e-6, 2e-6)
    # train-mode forward + backward, float64 on both sides: the two formulations must agree to rounding
    Rm = torch.randn(mine_eval.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    L = O.leaf_params(P, torch.float64)
    x = b["x"].double() if b["x"].is_floating_point() else b["x"]
    ea = b["edge_attr"].double() if b["edge_attr"].is_floating_point() else b["edge_attr"]
    stats = {}
    y2 = fwd(L, x, b["edge_index"], ea, 5, t, True, stats)
    (y2 * Rm).sum().backward()
    assert summary_close(y2, ref()[key + "train"], 1e-10, 1e-9)
    # per-tensor scale; a conv bias in front of BatchNorm has an exactly-zero gradient (pure rounding noise on both sides),
    # so the scale is floored at 1e-4 of the model's largest gradient
    grads = ref_prefixed(key + "grad:")
    assert set(grads) == {k for k, v in L.items() if v.requires_grad}
    gmax = max(float(S[1]) for S in grads.values())
    for k, S in grads.items():
        scale = max(float(S[1]), 1e-4 * gmax)
        assert summary_close(L[k].grad, S, 1e-9 * scale, 0.0), k
    for k, v in stats.items():
        assert summary_close(v, ref()[key + "stat:" + k], 1e-12, 1e-10), k


def test_direction_convention_is_visible_on_one_direction_graphs():
    """On the reference's symmetric inputs a swapped target/source is invisible for GIN (SURVEY.md 8(c)); on the
    one-direction-only graphs used by the parity tests it is not — so those tests do pin the convention."""
    P = O.make_params("chem", "gin", 5, 300, seed=8)
    for directed, differs in ((False, False), (True, True)):
        b = _batch("chem", directed, 31)
        with torch.no_grad():
            flipped = O.chem_gnn(P, b["x"], b["edge_index"].flip(0), b["edge_attr"], 5, "gin", False)
        assert (not summary_close(flipped, ref()[fwd_bwd_key("chem", "gin", directed) + "eval"], 1e-3, 1e-5)) == differs


def test_graphpred_heads_equal_reference():
    """chem/model.py:358-369 and bio/model.py:338-347 (mean pooling, centre-node concat, Linear)."""
    for domain, (T, b, full) in graphpred_inputs().items():
        with torch.no_grad():
            if domain == "chem":
                mine = O.chem_graphpred(full, b["x"], b["edge_index"], b["edge_attr"], b["batch"], b["num_graphs"], 5, "gin", False)
            else:
                mine = O.bio_graphpred(full, b["x"], b["edge_index"], b["edge_attr"], b["batch"], b["center_node_idx"], b["num_graphs"], 5, "gin", False)
        assert torch.allclose(mine, torch.from_numpy(ref()["graphpred:" + domain]), atol=2e-6, rtol=2e-6)


def test_collate_oracle_equals_reference_batch_masking():
    """oracle/step_io_oracle.collate_chem against BatchMasking.from_data_list itself (chem/batch.py:17-52), fed
    per-molecule Data objects that carry MaskAtom's extra keys (masked atoms: each molecule's first and last)."""
    graphs, ids = collate_masking_inputs()
    mine = SO.collate_chem(graphs, ids)
    exp_masked = np.concatenate([np.array([0, graphs[g][0].shape[0] - 1]) + mine["node_off"][i] for i, g in enumerate(ids)])
    assert_digests("collate_masking:", {k: mine[k] for k in ("x", "edge_index", "edge_attr", "batch")} | {"masked_atom_indices": exp_masked})


@pytest.mark.parametrize("config", ["masking", "contextpred", "bio_supervised", "gcn", "gat", "graphsage"])
def test_train_bodies_port_equals_reference(config):
    """oracle/steps_oracle.py: the restated train() bodies (loss + every gradient) against the same bodies on the
    reference's own modules, at a small batch."""
    from oracle import steps_oracle as S
    torch.set_num_threads(1)
    key = "train_body:%s:" % config
    b, P = train_body_inputs(config)
    L = O.leaf_params(P)
    loss, _ = S.LOSSES[config](L, b)
    loss.backward()
    loss_ref = float(ref()[key + "loss"])
    assert abs(float(loss) - loss_ref) <= 1e-6 * max(1.0, abs(loss_ref))
    grads = ref_prefixed(key + "grad:")
    assert set(grads) == {k for k, v in L.items() if v.requires_grad}
    gmax = max(float(Sg[1]) for Sg in grads.values())
    L64 = O.leaf_params(P, torch.float64)
    S.LOSSES[config](L64, b)[0].backward()
    for k, Sg in grads.items():
        # a bias in front of train-mode BatchNorm has a structurally zero gradient (fp64: ~1e-17): rounding noise on both sides
        zero = float(L64[k].grad.abs().max()) < 1e-9 * gmax
        scale = gmax if zero else max(float(Sg[1]), 1e-3 * gmax)
        # same arithmetic in a different order (fp32): agreement to a few ulps of the accumulated magnitude
        assert summary_close(L[k].grad, Sg, 2e-4 * scale, 0.0), k


def test_mask_atoms_oracle_equals_reference_maskatom():
    """oracle/step_io_oracle.mask_atoms against the reference's own MaskAtom.__call__ fed the same atom choice (its
    `masked_atom_indices` debugging argument, chem/util.py:206,225-241) followed by BatchMasking.from_data_list."""
    b, graphs, node_off, choice = mask_atoms_inputs()
    assert [len(c) for c in choice] == [int(len(g[0]) * 0.15 + 1) for g in graphs]
    x2, idx, labels, off = SO.mask_atoms(b["x"].numpy(), node_off, 0.15, seed=12345)
    assert_digests("mask_atoms:", {"x": x2, "masked_atom_indices": idx, "mask_node_label": labels})
    assert off[-1] == len(idx)
    # the draw is a uniform k-subset: over many seeds every node of a graph is chosen about equally often
    n0 = int(node_off[1])
    hits = np.zeros(n0)
    for s in range(400):
        hits[SO.mask_atom_choice(node_off[:2], 0.15, seed=s)[0]] += 1
    k = int(n0 * 0.15 + 1)
    assert abs(hits.mean() - 400 * k / n0) < 1e-9 and hits.min() > 0.5 * 400 * k / n0 and hits.max() < 1.6 * 400 * k / n0


def test_substruct_context_collate_oracle_equals_reference():
    """chem/batch.py:141-210: BatchSubstructContext.from_data_list on per-pair Data objects vs collate_chem x 2 + collate_lists."""
    G, sg, cg, center, overlap, ids = substruct_context_inputs()
    s, c = SO.collate_chem(sg, ids), SO.collate_chem(cg, ids)
    cptr, optr = np.arange(G + 1), np.cumsum([0] + [len(o) for o in overlap])
    cen, _, _, _ = SO.collate_lists(cptr, np.array(center), ids, add=s["node_off"])
    ov, seg, sizes, _ = SO.collate_lists(optr, np.concatenate(overlap), ids, add=c["node_off"])
    assert_digests("substruct_context_collate:", {
        "x_substruct": s["x"], "edge_index_substruct": s["edge_index"], "edge_attr_substruct": s["edge_attr"], "center_substruct_idx": cen,
        "x_context": c["x"], "edge_index_context": c["edge_index"], "edge_attr_context": c["edge_attr"],
        "overlap_context_substruct_idx": ov, "batch_overlapped_context": seg, "overlapped_context_size": sizes})


def test_bio_collate_oracle_equals_reference():
    """bio/batch.py:17-50 (BatchFinetune.from_data_list, the collator of bio/dataloader.py's DataLoaderFinetune: edge_index
    and center_node_idx offset by the running node count) vs collate_bio + collate_lists."""
    graphs, centers, ids = bio_collate_inputs()
    mine = SO.collate_bio(graphs, ids)
    cen, _, _, _ = SO.collate_lists(np.arange(6), np.array(centers), ids, add=mine["node_off"])
    assert_digests("bio_collate:", {k: mine[k] for k in ("x", "edge_index", "edge_attr", "batch")} | {"center_node_idx": cen})


def pair_digests(nodes_s, nodes_c, canon_s, canon_c, center, overlap):
    return [digest(v) for v in (nodes_s, nodes_c, canon_s, canon_c, [center], overlap)]


@pytest.mark.parametrize("k,l1,l2", EXTRACT_CHEM_PARAMS)
def test_extract_substruct_context_oracle_equals_reference_chem(k, l1, l2):
    """oracle/step_io_oracle.extract_pair against the reference's own ExtractSubstructureContextPair.__call__(data, root_idx)
    (chem/util.py:55-151) on molecules with duplicate bonds (the synthetic generator's extra pairs can repeat one), for the
    script's default (k, l1, l2) = (5, 4, 7) (chem/pretrain_contextpred.py:145-150), small radii, the 0 -> -1 quirk, an
    empty context (l1 == l2) and l1 > l2.  Compared in original node ids (the reference's own numbering undone through the
    maps it built): node sets, edge multisets, centre and overlap nodes."""
    rows = []
    for x, ei, ea, root in extract_chem_inputs():
        mine = SO.extract_pair(x, ei, ea, root, k, l1, l2)
        if mine is None:
            rows.append([NO_CONTEXT] * 6)
            continue
        ns, nc = mine["nodes_substruct"], mine["nodes_context"]
        assert np.array_equal(mine["x_substruct"], x[ns]) and np.array_equal(mine["x_context"], x[nc])
        assert ns[mine["center_substruct_idx"]] == root
        rows.append(pair_digests(ns.tolist(), nc.tolist(), _canon_edges(mine["edge_index_substruct"], mine["edge_attr_substruct"], ns),
                                 _canon_edges(mine["edge_index_context"], mine["edge_attr_context"], nc), root,
                                 nc[mine["overlap_context_substruct_idx"]].tolist()))
    want = ref()["extract_chem:%d_%d_%d" % (k, l1, l2)]
    assert want.shape == (len(rows), 6)
    for i, r in enumerate(rows):
        assert np.array_equal(np.array(r, np.int64), want[i]), (i, ["nodes_s", "nodes_c", "edges_s", "edges_c", "center", "overlap"])


def test_extract_pairs_batch_oracle_equals_reference_collation():
    """extract_pairs_batch = the per-graph extraction followed by BatchSubstructContext.from_data_list (chem/batch.py:141-210),
    including the reference's silent drop of pairs without a context.  The per-graph Data objects handed to the reference's
    collator carry THIS oracle's (canonically ordered) fields, so the comparison is exact."""
    graphs, ids, roots = extract_pairs_batch_inputs()
    mine = SO.extract_pairs_batch(graphs, ids, roots, 2, 1, 3)
    assert mine["kept"].tolist() == [0, 1, 2, 4, 5, 6]
    assert_digests("extract_pairs_batch:", {k_: mine[k_] for k_ in (
        "x_substruct", "edge_index_substruct", "edge_attr_substruct", "center_substruct_idx", "x_context", "edge_index_context",
        "edge_attr_context", "overlap_context_substruct_idx", "batch_overlapped_context", "overlapped_context_size")})


def test_extract_context_oracle_equals_reference_bio():
    """bio/util.py:123-205 (substructure = the whole ego graph, context = everything further than l1 hops from the centre,
    every context node an overlap node); nx_to_graph_data_obj (bio/loader.py:76-116) re-emits w1..w7 and zeros for the
    self-loop / mask columns of the context edges."""
    rows = []
    for n, e, a, l1 in extract_bio_inputs():
        mine = SO.extract_pair(np.ones((n, 1), np.float32), e, a, 0, 0, l1, 0, whole_graph=True)
        if mine is None:
            rows.append([NO_CONTEXT] * 4)
            continue
        nc = mine["nodes_context"]
        rows.append([digest(v) for v in (nc.tolist(), list(mine["x_context"].shape), _canon_edges(mine["edge_index_context"], mine["edge_attr_context"], nc),
                                          nc[mine["overlap_context_substruct_idx"]].tolist())])
    want = ref()["extract_bio"]
    assert len(rows) > 0 and want.shape == (len(rows), 4)
    for i, r in enumerate(rows):
        assert np.array_equal(np.array(r, np.int64), want[i]), (i, ["nodes_c", "x_context_shape", "edges_c", "overlap"])


def test_mask_edges_chem_oracle_equals_reference_maskatom_mask_edge():
    """oracle mask_edges_chem against the reference's MaskAtom(mask_edge=True).__call__(data, masked_atom_indices=choice)
    (chem/util.py:243-272) followed by BatchMasking.from_data_list (chem/batch.py:17-52: connected_edge_indices + cumsum_edge)."""
    b, graphs, node_off, _ = mask_edges_chem_inputs()
    _, idx, _, _ = SO.mask_atoms(b["x"].numpy(), node_off, 0.15, seed=777)
    edge_off = np.concatenate([[0], np.cumsum([g[1].shape[1] for g in graphs])])
    ea2, conn, lab, off = SO.mask_edges_chem(b["edge_index"].numpy(), b["edge_attr"].numpy(), edge_off, idx)
    assert_digests("mask_edges_chem:", {"edge_attr": ea2, "connected_edge_indices": conn, "mask_edge_label": lab})
    assert off[-1] == len(conn) and len(conn) > 0


def test_mask_edges_bio_oracle_equals_reference_maskedge():
    """oracle mask_edges_bio against the reference's MaskEdge.__call__(data, masked_edge_indices=[2 i ...]) (bio/util.py:46-104)
    followed by bio BatchMasking.from_data_list (bio/batch.py:71-105: masked_edge_idx + cumsum_edge)."""
    _, ea, eptr, choice = mask_edges_bio_inputs()
    assert [len(c) for c in choice] == [int((eptr[g + 1] - eptr[g]) // 2 * 0.15 + 1) for g in range(4)]
    ea2, idx, lab, off = SO.mask_edges_bio(ea, eptr, 0.15, seed=31)
    assert_digests("mask_edges_bio:", {"edge_attr": ea2, "masked_edge_idx": idx, "mask_edge_label": lab})
    assert off[-1] == len(idx)
