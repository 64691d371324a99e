"""Shared helpers: regenerate the golden inputs from seeds and compare against the stored vectors."""
import importlib
import os

import numpy as np
import torch

from oracle import gnn_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
syn = importlib.import_module("pretrain-gnns_b200.synthetic")
CASES = {"chem": dict(graphs=4, data_seed=11, param_seed=5), "bio": dict(graphs=2, data_seed=12, param_seed=6)}
TYPES = ("gin", "gcn", "graphsage", "gat")


def golden_batch(domain):
    c = CASES[domain]
    if domain == "chem":
        return syn.zinc_batch(c["graphs"], c["data_seed"])
    return syn.ppi_batch(c["graphs"], c["data_seed"], n_lo=40, n_hi=60, num_tasks=16)


# Shipped checkpoints of the reference (SURVEY.md section 8(d) config 1 and section 8(c) "what does pin behaviour" (i)): goldens in
# tests/golden/pretrained.npz (make_golden_pretrained.py); the files travel to the GPU box as git-ignored
# oracle/_ref/weights/<domain>/<dir>/<file> (oracle/reference_runner.stage).
PRETRAINED = {
    "chem_gin": dict(domain="chem", type="gin", file="chem/model_gin/masking.pth", graphs=32, seed=1001),
    "chem_gcn": dict(domain="chem", type="gcn", file="chem/model_architecture/gcn_contextpred.pth", graphs=32, seed=1002),
    "chem_gat": dict(domain="chem", type="gat", file="chem/model_architecture/gat_contextpred.pth", graphs=8, seed=1003),
    "chem_graphsage": dict(domain="chem", type="graphsage", file="chem/model_architecture/graphsage_contextpred.pth", graphs=8,
                           seed=1004),
    "bio_gin": dict(domain="bio", type="gin", file="bio/model_gin/masking.pth", graphs=2, seed=1005),
}


def pretrained_batch(name):
    c = PRETRAINED[name]
    if c["domain"] == "chem":
        return syn.zinc_batch(c["graphs"], c["seed"])
    return syn.ppi_batch(c["graphs"], c["seed"], n_lo=80, n_hi=120, num_tasks=16)


def pretrained_state_dict(name):
    """The checkpoint of PRETRAINED[name]: from the reference's tree, or from the copy build() staged from it under oracle/_ref."""
    from oracle import reference_runner as R
    c = PRETRAINED[name]
    for root in (R.REF_SRC, os.path.join(R.REF_STAGED, "weights")):
        path = os.path.join(root, c["file"])
        if os.path.isfile(path):
            return torch.load(path, map_location="cpu", weights_only=True), path
    return None, None


def golden_params(domain, t):
    return O.make_params(domain, t, 5, 300, seed=CASES[domain]["param_seed"])


# ---------------------------------------------------------------------------------------------------------------------
# Stored results of the reference's own code on the inputs of tests/test_oracle_vs_reference.py
# (tests/golden/make_golden_reference.py).  Full tensors would take megabytes, so exact results are kept as digests and
# float results as summaries that still carry the element-wise bound the tests state.
# ---------------------------------------------------------------------------------------------------------------------
REFERENCE_CHECKS = os.path.join(HERE, "golden", "reference_checks.npz")
SUMMARY_PROBE_SEED = 12345


SUMMARY_K = 20      # elements kept by summary() for gradients and BatchNorm statistics


def reference_checks():
    """name -> stored array.  Gradient and statistics summaries and the digests are stored as two tables (names + rows):
    every npz member costs a few hundred bytes of headers."""
    G = dict(np.load(REFERENCE_CHECKS))
    for name, row in zip(G.pop("summaries|names"), G.pop("summaries|rows")):
        G[str(name)] = row[:3 + min(int(row[0]), SUMMARY_K)]
    for name, value in zip(G.pop("digests|names"), G.pop("digests|values")):
        G[str(name)] = value
    return G


def digest(a):
    """64-bit digest of an array's values and shape, for exact comparisons (as np.array_equal: the dtype does not count)."""
    import hashlib
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64) + 0.0)   # + 0.0: -0.0 and 0.0 compare equal
    h = hashlib.sha256(repr(a.shape).encode() + a.tobytes()).digest()
    return np.frombuffer(h[:8], np.int64)[0]


def _flat(t):
    t = t.detach().cpu() if torch.is_tensor(t) else torch.from_numpy(np.asarray(t))
    return t.reshape(-1).double()


def _positions(n, k):
    return torch.tensor([(j * 2654435761 + 97) % n for j in range(k)] if n > k else list(range(n)), dtype=torch.long)


def _unit_probe(n):
    p = probe((n,), SUMMARY_PROBE_SEED).double()
    return p / p.norm()


def summary(t, k=SUMMARY_K):
    """float64 [numel, max|t|, <t, p>, t at k fixed positions], p a seeded unit vector over all elements."""
    t = _flat(t)
    n = t.numel()
    if n == 0:
        return np.zeros(3)
    head = [float(n), float(t.abs().max()), float(t @ _unit_probe(n))]
    return np.concatenate([head, t[_positions(n, k)].numpy()])


def summary_close(mine, S, atol, rtol):
    """Does `mine` meet |mine - ref| <= atol + rtol |ref| on what summary(ref) kept?  The kept elements carry that bound
    itself; the max-norm and the projection carry what it implies for all elements together:
    |max|mine| - max|ref|| <= max|mine - ref| and |<mine - ref, p>| <= ||mine - ref||_2 <= sqrt(n) max_i (atol + rtol |ref_i|)."""
    m = _flat(mine)
    n = int(S[0])
    if m.numel() != n:
        return False
    if n == 0:
        return True
    amax, proj, vals = float(S[1]), float(S[2]), torch.from_numpy(np.asarray(S[3:]))
    bound = atol + rtol * amax
    if not bool(((m[_positions(n, len(vals))] - vals).abs() <= atol + rtol * vals.abs()).all()):
        return False
    if abs(float(m.abs().max()) - amax) > bound:
        return False
    mp = float(m @ _unit_probe(n))
    return abs(mp - proj) <= n ** 0.5 * bound + 1e-13 * (abs(proj) + float(m.norm()))


def load(domain, t):
    return dict(np.load(os.path.join(HERE, "golden", f"{domain}_{t}.npz")))


def probe(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=g)


def input_checksum(b):
    h = 0
    for k in ("x", "edge_index", "edge_attr"):
        h = (h * 1000003 + int(b[k].to(torch.float64).sum().item() * 8 + b[k].numel())) % (2 ** 61 - 1)
    return np.int64(h)


def close(a, b, atol=1e-4, rtol=1e-4):
    """north_star tolerance: 1e-4 fp32, stated abs + rel (SURVEY.md §7.2)."""
    a = torch.as_tensor(np.asarray(a), dtype=torch.float64)
    b = torch.as_tensor(np.asarray(b), dtype=torch.float64)
    err = (a - b).abs()
    bound = atol + rtol * b.abs()
    worst = (err - bound).max().item() if err.numel() else -1.0
    return worst <= 0, float(err.max().item() if err.numel() else 0.0)


def close_scaled(a, b, tol=1e-4, floor=1.0):
    """Gradient check: max error relative to the reference tensor's largest magnitude (sums over
    hundreds of rows cancel, so an element-wise relative bound is meaningless for them).

    ReLU-boundary allowance: a hidden pre-activation within rounding distance of 0 lands on the other side
    of the ReLU under a different (equally valid) fp32 summation order; its gradient mask flips and the
    change propagates to every upstream gradient.  With ~10^5-10^6 hidden units per step a handful of such
    flips is the expected case, not an accident (P ~ units * rounding_error / activation_scale).  A flip
    moves a few rows of some gradients by a finite amount but leaves the tensor as a whole where it was, so a
    tensor that misses the max-norm bound is still accepted when its relative L2 (Frobenius) error is below
    0.5% -- a wrong formula or a wrong index shows up as O(10%-100%) there."""
    a = torch.as_tensor(np.asarray(a), dtype=torch.float64)
    b = torch.as_tensor(np.asarray(b), dtype=torch.float64)
    if not b.numel():
        return True, 0.0
    scale = max(float(b.abs().max().item()), floor)
    err = (a - b).abs() / scale
    e = float(err.max().item())
    if e <= tol:
        return True, e
    if b.numel() >= 64:
        fro = float((a - b).norm().item() / max(b.norm().item(), 1e-30))
        if fro <= 5e-3:
            return True, e
    return False, e


def check_against_golden(G, out_eval, out_train, grads, stats, atol=1e-4, rtol=1e-4, gtol=2e-4, slack=4.0):
    """Compare a full set of results with one golden file. `grads`: name -> tensor; `stats`: name -> tensor.

    Outputs: |mine - reference_fp32| <= atol + rtol*|ref| (the north_star bound).
    Gradients: train-mode BatchNorm makes them ill-conditioned in fp32 (the reference's own fp32 and fp64
    runs differ by up to ~1e-2 of the tensor scale), so the bound is relative to that yardstick:
        err(mine, ref_fp64) <= max(gtol, slack * err(ref_fp32, ref_fp64)),
    errors measured against the tensor's largest magnitude (floored at the model's typical gradient scale)."""
    bad = []
    gmax = sorted(float(np.abs(v).max()) for k, v in G.items() if k.startswith("g:") and v.size)
    floor = max(gmax[len(gmax) // 2], 1.0) if gmax else 1.0
    for name, mine in (("out_eval", out_eval), ("out_train", out_train)):
        if mine is None:
            continue
        ok, e = close(mine, G[name], atol, rtol)
        if not ok:
            bad.append((name, e))

    def summarise(kind, t):
        t = torch.as_tensor(np.asarray(t), dtype=torch.float64)
        if kind == "g":
            return t
        t2 = t.reshape(t.shape[0], -1)
        if kind == "gs0":
            return t2.sum(0)
        if kind == "gs1":
            return t2.sum(1)
        return (t * probe(t.shape, 77).double()).sum()

    for k, ref32 in G.items():
        kind, _, name = k.partition(":")
        if kind in ("g", "gs0", "gs1", "gp") and grads is not None:
            ref64 = G.get(kind + "64:" + name)
            mine = summarise(kind, grads[name])
            if ref64 is None:
                ok, e = close_scaled(mine, ref32, gtol, floor)
            else:
                _, e_ref = close_scaled(ref32, ref64, 0.0, floor)
                tol = max(gtol, slack * e_ref)
                ok, e = close_scaled(mine, ref64, tol, floor)
                if not ok:  # also acceptable: as close to the fp32 reference as that is to fp64
                    ok, e = close_scaled(mine, ref32, tol, floor)
        elif kind == "rs" and stats is not None:
            ok, e = close(stats[name], ref32, atol, rtol)
        else:
            continue
        if not ok:
            bad.append((k, e))
    return bad


def grad_close(mine, ref32, ref64, floor=1.0, gtol=2e-4, slack=4.0):
    """Same yardstick for oracle-based (non-golden) tests: returns (ok, err, tol)."""
    _, e_ref = close_scaled(ref32, ref64, 0.0, floor)
    tol = max(gtol, slack * e_ref)
    ok, e = close_scaled(mine, ref64, tol, floor)
    return ok, e, tol


# ---------------------------------------------------------------------------------------------------------------------
# Full-size oracle parity (tests/test_gpu_parity_full.py): per-tensor bounds stated against what is measured.
#
# Forward outputs: the north_star bound |mine - ref32| <= 1e-4 + 1e-4 |ref32|, AND max|mine - ref64| <= OUT_REL x the
# tensor's largest magnitude (measured on B200: 1-4e-6 for the 3xTF32 path; OUT_REL is ~10x that).
# Gradients, per tensor: err = max|mine - ref64| / scale with scale = the tensor's own largest |ref64| (floored at 1e-3 of the
# model's largest gradient; a structurally zero gradient -- a bias in front of train-mode BatchNorm -- is compared on the
# model's scale).  Train-mode BatchNorm makes fp32 gradients ill-conditioned: the oracle's OWN fp32 run misses its fp64 run
# by e_ref (up to ~1e-3 of scale at B=256), so the bound is  err <= max(GRAD_REL, SLACK x e_ref)  (measured: err <= ~1.5 e_ref).
# ReLU-boundary allowance (relative Frobenius error <= 5e-3) ONLY when the fp64 oracle run actually has a ReLU
# pre-activation within rounding distance of zero (oracle.gnn_oracle.near_zero_preactivations), and it is reported.
# ---------------------------------------------------------------------------------------------------------------------
OUT_REL = 4e-5
GRAD_REL = 5e-5
SLACK = 3.0


def output_check(name, mine, ref32, ref64, rows):
    mine, ref32, ref64 = (torch.as_tensor(t).detach().cpu().double() for t in (mine, ref32, ref64))
    scale = max(float(ref64.abs().max()), 1e-30)
    e64 = float((mine - ref64).abs().max()) / scale
    eref = float((ref32 - ref64).abs().max()) / scale
    north = bool(((mine - ref32).abs() <= 1e-4 + 1e-4 * ref32.abs()).all())
    ok = north and e64 <= max(OUT_REL, SLACK * eref)
    rows.append(dict(kind="out", name=name, err=e64, err_ref32=eref, north_star=north, ok=ok))
    return ok


def gradient_check(named_mine, g32, g64, near_zero, rows):
    gmax = max(float(v.abs().max()) for v in g64.values())
    ok_all = True
    for k, mine in named_mine:
        mine = mine.detach().cpu().double()
        r64, r32 = g64[k].double(), g32[k].double()
        tmax = float(r64.abs().max())
        zero = tmax < 1e-9 * gmax
        scale = gmax if zero else max(tmax, 1e-3 * gmax)
        e = float((mine - r64).abs().max()) / scale
        eref = float((r32 - r64).abs().max()) / scale
        tol = max(GRAD_REL, SLACK * eref)
        ok, via = e <= tol, "max"
        if not ok and near_zero > 0 and r64.numel() >= 64:
            fro = float((mine - r64).norm() / max(float(r64.norm()), 1e-30))
            if fro <= 5e-3:
                ok, via = True, "relu-boundary allowance (fro %.2e, %d near-zero pre-activations)" % (fro, near_zero)
        rows.append(dict(kind="grad", name=k, err=e, err_ref32=eref, tol=tol, ok=ok, via=via, structurally_zero=zero))
        ok_all &= ok
    return ok_all


def write_report(test_name, rows, extra=None):
    """Measured errors of a parity test -> gpurun_out/parity/<test>.json (travels back from the GPU box)."""
    import json
    d = os.path.join(os.path.dirname(HERE), "gpurun_out", "parity")
    try:
        os.makedirs(d, exist_ok=True)
        worst = {}
        for r in rows:
            w = worst.setdefault(r["kind"], dict(err=0.0, err_ref32=0.0))
            w["err"], w["err_ref32"] = max(w["err"], r["err"]), max(w["err_ref32"], r["err_ref32"])
        with open(os.path.join(d, test_name + ".json"), "w") as fh:
            json.dump(dict(test=test_name, worst=worst, extra=extra or {}, rows=rows), fh, indent=1)
    except OSError:
        pass
