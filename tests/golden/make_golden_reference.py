"""Store what the REFERENCE's own, unmodified model.py / batch.py / util.py compute on the inputs of
tests/test_oracle_vs_reference.py, so that the oracle is checked against them wherever the tests run.

Needs the reference's sources (oracle/reference_runner.py finds them):

    python tests/golden/make_golden_reference.py

Inputs are not stored: the test module's own input functions build them from seeds here and in the tests.  Stored in
tests/golden/reference_checks.npz:

    fwd_bwd:<domain>_<type>_<symmetric|directed>:eval|train|grad:<param>|stat:<key>   golden_util.summary records
    train_body:<config>:loss / :grad:<param>                                          fp64 loss, summary records
    graphpred:<domain>                                                                full head outputs (fp32)
    collate_masking:, mask_atoms:, substruct_context_collate:, bio_collate:,
    extract_pairs_batch:, mask_edges_chem:, mask_edges_bio: <field>                   golden_util.digest of the field
    extract_chem:<k>_<l1>_<l2>, extract_bio                                          digests, one row per extraction

The gradient / statistics summaries and the single digests are written as two tables (golden_util.reference_checks).
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import test_oracle_vs_reference as T  # noqa: E402
from golden_util import REFERENCE_CHECKS, SUMMARY_K, digest, summary  # noqa: E402
from oracle import gnn_oracle as O  # noqa: E402
from oracle import reference_runner as R  # noqa: E402
from oracle import step_io_oracle as SO  # noqa: E402
from oracle import steps_oracle as S  # noqa: E402


def data(**kw):
    from torch_geometric.data import Data  # the stand-in (oracle/pyg103_standin), on sys.path once R.load has run
    return Data(**{k: torch.from_numpy(np.ascontiguousarray(v)) if isinstance(v, np.ndarray) else v for k, v in kw.items()})


def ref_step(mod, P, b, t, training, dtype=torch.float32):
    model = mod.GNN(5, 300, JK="last", drop_ratio=0, gnn_type=t)
    assert str(model.load_state_dict(P)) == "<All keys matched successfully>"
    model.to(dtype).train(training)
    x = b["x"].to(dtype) if b["x"].is_floating_point() else b["x"]
    ea = b["edge_attr"].to(dtype) if b["edge_attr"].is_floating_point() else b["edge_attr"]
    return model, model(x, b["edge_index"], ea)


def fwd_bwd(out):
    for domain in ("chem", "bio"):
        mod = R.load(domain)
        for t in T.TYPES:
            for directed in (False, True):
                key = T.fwd_bwd_key(domain, t, directed)
                b = T._batch(domain, directed, 31)
                P = O.make_params(domain, t, 5, 300, seed=8)
                with torch.no_grad():
                    _, y_eval = ref_step(mod, P, b, t, False)
                out[key + "eval"] = summary(y_eval, 64)
                Rm = torch.randn(y_eval.shape, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
                model, y = ref_step(mod, P, b, t, True, torch.float64)
                (y * Rm).sum().backward()
                out[key + "train"] = summary(y, 64)
                for k, p in model.named_parameters():
                    out[key + "grad:" + k] = summary(p.grad)
                for k, v in model.state_dict().items():
                    if k.endswith(("running_mean", "running_var", "num_batches_tracked")):
                        out[key + "stat:" + k] = summary(v)


def graphpred(out):
    for domain, (n_tasks, b, full) in T.graphpred_inputs().items():
        mod = R.load(domain)
        model = mod.GNN_graphpred(5, 300, n_tasks, JK="last", drop_ratio=0, graph_pooling="mean", gnn_type="gin")
        assert str(model.load_state_dict(full)) == "<All keys matched successfully>"
        model.eval()
        with torch.no_grad():
            if domain == "chem":
                y = model(b["x"], b["edge_index"], b["edge_attr"], b["batch"])
            else:
                y = model(types.SimpleNamespace(**{k: b[k] for k in ("x", "edge_index", "edge_attr", "batch", "center_node_idx")}))
        out["graphpred:" + domain] = y.numpy()


def train_bodies(out):
    torch.set_num_threads(1)
    for config in ("masking", "contextpred", "bio_supervised", "gcn", "gat", "graphsage"):
        b, P = T.train_body_inputs(config)
        step = S.REFERENCE_STEPS[config]() if config != "bio_supervised" else S.ReferenceBioSupervisedStep(24)
        step.load(P)
        out["train_body:%s:loss" % config] = np.float64(float(step(b)))
        for name, m in step.named.items():
            for k, p in m.named_parameters():
                out["train_body:%s:grad:%s.%s" % (config, name, k)] = summary(p.grad)


def put_digests(out, prefix, ref, keys):
    for k in keys:
        out[prefix + k] = digest(ref[k].numpy())


def collators(out):
    chem_batch, bio_batch = R.load("chem", "batch"), R.load("bio", "batch")
    graphs, ids = T.collate_masking_inputs()
    ref = chem_batch.BatchMasking.from_data_list([data(x=graphs[g][0], edge_index=graphs[g][1], edge_attr=graphs[g][2],
                                                       masked_atom_indices=torch.tensor([0, graphs[g][0].shape[0] - 1])) for g in ids])
    put_digests(out, "collate_masking:", ref, ("x", "edge_index", "edge_attr", "batch", "masked_atom_indices"))

    G, sg, cg, center, overlap, ids = T.substruct_context_inputs()
    datas = [data(x=sg[g][0], edge_index=sg[g][1], edge_attr=sg[g][2],   # the main graph (unused by the collator but num_nodes reads x)
                  x_substruct=sg[g][0], edge_index_substruct=sg[g][1], edge_attr_substruct=sg[g][2], center_substruct_idx=torch.tensor([center[g]]),
                  x_context=cg[g][0], edge_index_context=cg[g][1], edge_attr_context=cg[g][2],
                  overlap_context_substruct_idx=torch.tensor(overlap[g])) for g in ids]
    ref = chem_batch.BatchSubstructContext.from_data_list(datas)
    put_digests(out, "substruct_context_collate:", ref, (
        "x_substruct", "edge_index_substruct", "edge_attr_substruct", "center_substruct_idx", "x_context", "edge_index_context",
        "edge_attr_context", "overlap_context_substruct_idx", "batch_overlapped_context", "overlapped_context_size"))

    graphs, centers, ids = T.bio_collate_inputs()
    ref = bio_batch.BatchFinetune.from_data_list([data(x=torch.ones(graphs[g][0], 1), edge_index=graphs[g][1], edge_attr=graphs[g][2],
                                                       center_node_idx=torch.tensor([centers[g]])) for g in ids])
    put_digests(out, "bio_collate:", ref, ("x", "edge_index", "edge_attr", "batch", "center_node_idx"))


def masking_transforms(out):
    util, chem_batch = R.load("chem", "util"), R.load("chem", "batch")
    _, graphs, _, choice = T.mask_atoms_inputs()
    t = util.MaskAtom(num_atom_type=119, num_edge_type=5, mask_rate=0.15, mask_edge=False)
    ref = chem_batch.BatchMasking.from_data_list([t(data(x=x, edge_index=ei, edge_attr=ea), masked_atom_indices=list(c))
                                                  for (x, ei, ea), c in zip(graphs, choice)])
    put_digests(out, "mask_atoms:", ref, ("x", "masked_atom_indices", "mask_node_label"))

    _, graphs, _, choice = T.mask_edges_chem_inputs()
    t = util.MaskAtom(num_atom_type=119, num_edge_type=5, mask_rate=0.15, mask_edge=True)
    ref = chem_batch.BatchMasking.from_data_list([t(data(x=x, edge_index=ei, edge_attr=ea), masked_atom_indices=list(c))
                                                  for (x, ei, ea), c in zip(graphs, choice)])
    put_digests(out, "mask_edges_chem:", ref, ("edge_attr", "connected_edge_indices", "mask_edge_label"))

    util, bio_batch = R.load("bio", "util"), R.load("bio", "batch")
    graphs, _, _, choice = T.mask_edges_bio_inputs()
    t = util.MaskEdge(mask_rate=0.15)
    ref = bio_batch.BatchMasking.from_data_list([t(data(x=torch.ones(n, 1), edge_index=e, edge_attr=a.copy()), masked_edge_indices=[2 * i for i in c])
                                                 for (n, e, a), c in zip(graphs, choice)])
    put_digests(out, "mask_edges_bio:", ref, ("edge_attr", "masked_edge_idx", "mask_edge_label"))


def ref_extract(util, transform, d, root):
    """Run the reference's ExtractSubstructureContextPair and return its output together with the old->new node maps it
    built (util.reset_idxes is a module-level function looked up at call time: wrap it to record the maps)."""
    maps = []
    orig = util.reset_idxes

    def recording(G):
        new_G, mapping = orig(G)
        maps.append(dict(mapping))
        return new_G, mapping

    util.reset_idxes = recording
    try:
        res = transform(d, root_idx=root)
    finally:
        util.reset_idxes = orig
    return res, maps


def has_context(ref):
    return hasattr(ref, "x_context") and ref.x_context is not None


def extraction(out):
    util = R.load("chem", "util")
    for k, l1, l2 in T.EXTRACT_CHEM_PARAMS:
        t = util.ExtractSubstructureContextPair(k, l1, l2)
        rows = []
        for x, ei, ea, root in T.extract_chem_inputs():
            ref, maps = ref_extract(util, t, data(x=x, edge_index=ei, edge_attr=ea), root)
            if not has_context(ref):
                rows.append([T.NO_CONTEXT] * 6)
                continue
            inv_s = {new: old for old, new in maps[0].items()}
            inv_c = {new: old for old, new in maps[1].items()}
            for new, old in inv_s.items():
                assert np.array_equal(ref.x_substruct[new].numpy(), x[old])
            for new, old in inv_c.items():
                assert np.array_equal(ref.x_context[new].numpy(), x[old])
            center = inv_s[int(ref.center_substruct_idx)]
            assert center == root
            ov = sorted(inv_c[int(i)] for i in ref.overlap_context_substruct_idx) \
                if getattr(ref, "overlap_context_substruct_idx", None) is not None else []
            rows.append(T.pair_digests(sorted(maps[0]), sorted(maps[1]),
                                       T._canon_edges(ref.edge_index_substruct.numpy(), ref.edge_attr_substruct.numpy(), inv_s),
                                       T._canon_edges(ref.edge_index_context.numpy(), ref.edge_attr_context.numpy(), inv_c), center, ov))
        out["extract_chem:%d_%d_%d" % (k, l1, l2)] = np.array(rows, np.int64)

    chem_batch = R.load("chem", "batch")
    graphs, ids, roots = T.extract_pairs_batch_inputs()
    datas = []
    for g, r in zip(ids, roots):
        x, ei, ea = graphs[g]
        p = SO.extract_pair(x, ei, ea, int(r), 2, 1, 3)   # the collator is fed this oracle's per-graph fields
        d = data(x=x, edge_index=ei, edge_attr=ea)
        if p is not None:
            for k_ in ("x_substruct", "edge_index_substruct", "edge_attr_substruct", "x_context", "edge_index_context", "edge_attr_context",
                       "overlap_context_substruct_idx"):
                setattr(d, k_, torch.from_numpy(np.ascontiguousarray(p[k_])))
            d.center_substruct_idx = torch.tensor([p["center_substruct_idx"]])
        datas.append(d)
    ref = chem_batch.BatchSubstructContext.from_data_list(datas)
    put_digests(out, "extract_pairs_batch:", ref, (
        "x_substruct", "edge_index_substruct", "edge_attr_substruct", "center_substruct_idx", "x_context", "edge_index_context",
        "edge_attr_context", "overlap_context_substruct_idx", "batch_overlapped_context", "overlapped_context_size"))

    util = R.load("bio", "util")
    rows = []
    for n, e, a, l1 in T.extract_bio_inputs():
        t = util.ExtractSubstructureContextPair(l1, center=True)
        ref, maps = ref_extract(util, t, data(x=torch.ones(n, 1), edge_index=e, edge_attr=a, center_node_idx=torch.tensor([0])), None)
        if not has_context(ref):
            rows.append([T.NO_CONTEXT] * 4)
            continue
        assert np.array_equal(ref.edge_index_substruct.numpy(), e) and int(ref.center_substruct_idx) == 0
        inv_c = {new: old for old, new in maps[0].items()}
        rows.append([digest(v) for v in (sorted(maps[0]), list(ref.x_context.shape),
                                          T._canon_edges(ref.edge_index_context.numpy(), ref.edge_attr_context.numpy(), inv_c),
                                          sorted(inv_c[int(i)] for i in ref.overlap_context_substruct_idx))])
    out["extract_bio"] = np.array(rows, np.int64)


def main():
    assert R.available(), "the reference's sources are not available"
    torch.manual_seed(0)
    torch.set_num_threads(1)
    out = {}
    for part in (fwd_bwd, graphpred, train_bodies, collators, masking_transforms, extraction):
        part(out)
    summaries = {k: out.pop(k) for k in [k for k in out if ":grad:" in k or ":stat:" in k]}
    digests = {k: out.pop(k) for k in [k for k in out if isinstance(out[k], np.int64)]}
    rows = np.zeros((len(summaries), 3 + SUMMARY_K))
    for i, v in enumerate(summaries.values()):
        rows[i, :len(v)] = v
    out.update({"summaries|names": np.array(list(summaries)), "summaries|rows": rows,
                "digests|names": np.array(list(digests)), "digests|values": np.array(list(digests.values()), np.int64)})
    np.savez_compressed(REFERENCE_CHECKS, **out)
    print(REFERENCE_CHECKS, os.path.getsize(REFERENCE_CHECKS) // 1024, "KiB,", len(out), "arrays")


if __name__ == "__main__":
    main()
