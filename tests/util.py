"""Shared helpers for the tests: fixture loading and engine construction."""
import os
import types

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WKEYS = ["W1", "b1", "W2", "b2", "W3", "b3", "Wp", "bp"]


def load_fixture(name):
    """-> namespace(N, edges, feat, label, pred, weights, rowptr, col, pred_label, gold)"""
    import gnnx_oracle as O
    g = np.load(os.path.join(GOLDEN, name + "_graph.npz"))
    gold = np.load(os.path.join(GOLDEN, name + "_golden.npz"))
    N = int(g["N"])
    rowptr, col = O.csr_from_edges(N, g["edges"])
    return types.SimpleNamespace(
        name=name, N=N, edges=g["edges"], feat=g["feat"], label=g["label"], pred=g["pred"],
        weights={k: g[k] for k in WKEYS}, rowptr=rowptr, col=col,
        pred_label=np.argmax(g["pred"], axis=1).astype(np.int32), gold=gold,
        nodes=[int(x) for x in gold["nodes"]])


def make_engine(fx, device=0):
    import gnnx
    eng = gnnx.Engine(device)
    eng.set_model(fx.weights)
    eng.set_graph_csr(fx.rowptr, fx.col, fx.feat, fx.label, fx.pred_label)
    return eng


def golden_m0(fx, plan):
    """Concatenate the golden M0 edge entries in plan order (checks the edge counts on the way)."""
    m0 = np.empty(plan.total_edges, np.float32)
    for t, node in enumerate(plan.nodes):
        g = fx.gold["n%d_m0" % node]
        assert len(g) == plan.edge_off[t + 1] - plan.edge_off[t], "directed edge count differs from the reference"
        m0[plan.edge_off[t]:plan.edge_off[t + 1]] = g
    return m0


def node_tolerances(name, epochs):
    """Per-node parity tolerance at a horizon: 1e-4 wherever the REFERENCE's own result is reproducible, i.e. max(1e-4, 3 x spread)
    with spread = how far the bit-exact port of the reference moves when every M0 entry (and the weights) is nudged by +-1 ulp
    (oracle/gen_sensitivity.py -> golden/*_sens.npz) and, at 100 epochs, how far its fp64 / fp32 closed-form restatements land
    (oracle/gen_conditioning.py -> golden/*_cond.npz).  Nine updates (10 epochs) leave no room for amplification: 1e-4 flat."""
    sens = np.load(os.path.join(GOLDEN, name + "_sens.npz"))
    nodes = [int(n) for n in sens["nodes"]]
    if epochs <= 10:
        return {n: 1e-4 for n in nodes}
    spread = np.array(sens["spread_e30"] if epochs <= 30 else sens["spread_e100"], np.float64)
    if epochs > 30:
        cond = np.load(os.path.join(GOLDEN, name + "_cond.npz"))
        assert [int(n) for n in cond["nodes"]] == nodes
        spread = np.maximum(spread, np.maximum(cond["err_closed64"], cond["err_closed32"]))
    return {n: max(1e-4, 3.0 * float(s)) for n, s in zip(nodes, spread)}


def assert_per_node(errs, name, epochs):
    """errs: {node: rel-L2 vs the reference golden}.  Every node within its tolerance; every reproducible node within 1e-4."""
    tol = node_tolerances(name, epochs)
    bad = {n: (e, tol[n]) for n, e in errs.items() if not e <= tol[n]}
    assert not bad, bad
    return tol


def write_tu_toy(tmp, name, rng):
    """Five small graphs in the TU graph-kernel text format under tmp/name/ (one of 12 nodes); returns their sizes."""
    os.makedirs(os.path.join(tmp, name), exist_ok=True)
    pre = os.path.join(tmp, name, name)
    sizes = [5, 9, 3, 12, 7]
    gi, nl, A = [], [], []
    base = 1
    for g, n in enumerate(sizes, 1):
        gi += [g] * n
        nl += list(rng.integers(3, 8, n))
        perm = rng.permutation(n)
        es = [(base + int(perm[i]), base + int(perm[i + 1])) for i in range(n - 1)] + [(base + int(rng.integers(0, n)), base + int(rng.integers(0, n))) for _ in range(2)]
        for a, b in es:
            if a != b:
                A += [(a, b), (b, a)]
        base += n
    open(pre + "_graph_indicator.txt", "w").write("\n".join(map(str, gi)) + "\n")
    open(pre + "_node_labels.txt", "w").write("\n".join(map(str, nl)) + "\n")
    open(pre + "_graph_labels.txt", "w").write("\n".join(map(str, [1, -1, -1, 1, 1])) + "\n")
    open(pre + "_A.txt", "w").write("\n".join("%d, %d" % e for e in A) + "\n")
    return sizes


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    den = np.linalg.norm(b)
    return float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b))
