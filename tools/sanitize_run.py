#!/usr/bin/env python
"""Small invocation of every kernel for compute-sanitizer (racecheck / memcheck / synccheck are ~100x slower than a plain run):
    compute-sanitizer --tool racecheck python tools/sanitize_run.py
k-hop extraction + shared-memory kernel on a mix of task sizes (syn1: hub node 0 and tiny tasks), the streaming kernel (forced),
the gradient baseline, graph mode (tuned kernel and graph-variant kernel), densify, neighbourhood rows.  A few epochs each."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("gnn-model-explainer_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))
import util  # noqa: E402
import gnnx  # noqa: E402
from gnnx import _abi  # noqa: E402

EPOCHS = int(os.environ.get("SAN_EPOCHS", "4"))


def main():
    which = sys.argv[1:] or ["node", "stream", "graph", "graphvar", "misc", "var", "cluster"]
    fx = util.load_fixture("syn1")
    if "node" in which:
        eng = util.make_engine(fx)
        nodes = [0, 3, 300, 301, 683, 699, 13, 550]
        plan = eng.plan_nodes(nodes, 3)
        out = np.zeros(plan.total_edges, np.float32)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS), util.golden_m0(fx, plan), out)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS, init=_abi.GX_INIT_PHILOX, seed=3), None, out)
        eng.grad_nodes_host(out)
        print("node ok", float(out.sum()))
        eng.close()
    if "stream" in which:
        fr = util.load_fixture("rand")
        for gang in (0, 3, -1):          # explain_gang.cu (automatic gang size, 3 CTAs per task) and explain_stream.cu
            eng = util.make_engine(fr)
            eng.debug_force_stream(True)
            eng.debug_gang(gang)
            plan = eng.plan_nodes(fr.nodes[:4], 3)
            out = np.zeros(plan.total_edges, np.float32)
            eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS), util.golden_m0(fr, plan), out)
            eng.grad_nodes_host(out)
            print("stream ok (gang %d)" % gang, float(out.sum()))
            eng.close()
    if "var" in which:
        g = np.load(util.GOLDEN + "/variants_golden.npz")
        import gnnx_oracle as O
        N = int(g["N"])
        rowptr, col = O.csr_from_edges(N, g["edges"])
        for tag, L, bn in (("bn", 3, True), ("L4", 4, False)):
            w = {k[len(tag) + 1:]: g[k] for k in g.files if k.startswith(tag + "_W") or k.startswith(tag + "_b")}
            eng = gnnx.Engine(0)
            eng.set_model(w, num_layers=L, bn=bn)
            eng.set_graph_csr(rowptr, col, g["feat"].astype(np.float32), g["label"].astype(np.int32), np.argmax(g[tag + "_pred"], 1).astype(np.int32))
            plan = eng.plan_nodes([0, 17], L)
            out = np.zeros(plan.total_edges, np.float32)
            eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS, init=_abi.GX_INIT_PHILOX, seed=2), None, out)
            print("var ok", tag, float(out.sum()))
            eng.close()
        rng = np.random.default_rng(5)   # a wide model (hidden 64 / output 48): two lane chunks per row
        sc = lambda *s_: (rng.normal(size=s_) * 0.4).astype(np.float32)
        d0 = g["feat"].shape[1]
        ww = dict(W1=sc(d0, 64), b1=sc(64), W2=sc(64, 64), b2=sc(64), W3=sc(64, 48), b3=sc(48), Wp=sc(3, 176), bp=sc(3))
        eng = gnnx.Engine(0)
        eng.set_model(ww, num_layers=3, bn=False)
        eng.set_graph_csr(rowptr, col, g["feat"].astype(np.float32), g["label"].astype(np.int32), np.zeros(N, np.int32))
        plan = eng.plan_nodes([0, 17], 3)
        out = np.zeros(plan.total_edges, np.float32)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS, init=_abi.GX_INIT_PHILOX, seed=2), None, out)
        print("var ok wide", float(out.sum()))
        eng.close()
        eng = util.make_engine(fx)     # default model, optimiser other than Adam -> the variant kernel
        plan = eng.plan_nodes([300, 5], 3)
        out = np.zeros(plan.total_edges, np.float32)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS, opt=1), util.golden_m0(fx, plan), out)
        print("var ok sgd", float(out.sum()))
        eng.close()
    if "cluster" in which:
        eng = util.make_engine(fx)
        eng.debug_cluster(4, 1)
        plan = eng.plan_nodes([0, 300, 13], 3)
        out = np.zeros(plan.total_edges, np.float32)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=EPOCHS), util.golden_m0(fx, plan), out)
        print("cluster ok", float(out.sum()))
        eng.close()
    if "graph" in which:
        g = np.load(util.GOLDEN + "/graphs_golden.npz")
        eng = gnnx.Engine(0)
        eng.set_model({k: g[k] for k in util.WKEYS})
        eng.set_graph_batch(g["adj"], g["feat"], g["label"])
        gids = [0, 3, 5, 11]
        eoff = eng.plan_graphs(gids)
        m0 = np.concatenate([g["g%d_m0" % i] for i in gids]).astype(np.float32)
        out = np.zeros(int(eoff[-1]), np.float32)
        eng.explain_graphs_host(eng.make_hparams(num_epochs=EPOCHS), m0, out)
        print("graph ok", float(out.sum()))
        eng.close()
    if "graphvar" in which:
        # explain_graph_var.cu: 4 layers + bn (small-slab class), a 128-wide model, the default model with sgd, and the default model
        # on a batch padded to 600 nodes whose largest graph exceeds the shared-memory kernel (large-slab class next to the tuned kernel)
        g = np.load(util.GOLDEN + "/graphs_golden.npz")
        gv = np.load(util.GOLDEN + "/graph_variants_golden.npz")
        gids = [0, 3, 5, 11]
        m0 = np.concatenate([g["g%d_m0" % i] for i in gids]).astype(np.float32)
        for tag, L, bn in (("L4bn", 4, True), ("w128", 2, False)):
            w = {k[len(tag) + 1:]: gv[k] for k in gv.files if k.startswith(tag + "_W") or (k.startswith(tag + "_b") and k != tag + "_bn")}
            eng = gnnx.Engine(0)
            eng.set_model(w, num_layers=L, bn=bn)
            eng.set_graph_batch(g["adj"], g["feat"], g["label"])
            eoff = eng.plan_graphs(gids)
            out = np.zeros(int(eoff[-1]), np.float32)
            eng.explain_graphs_host(eng.make_hparams(num_epochs=EPOCHS), m0, out)
            eng.explain_graphs_host(eng.make_hparams(num_epochs=EPOCHS, init=_abi.GX_INIT_PHILOX, seed=4), None, out)
            print("graphvar ok", tag, float(out.sum()))
            eng.close()
        eng = gnnx.Engine(0)
        eng.set_model({k: g[k] for k in util.WKEYS})
        eng.set_graph_batch(g["adj"], g["feat"], g["label"])
        eoff = eng.plan_graphs(gids)
        out = np.zeros(int(eoff[-1]), np.float32)
        eng.explain_graphs_host(eng.make_hparams(num_epochs=EPOCHS, opt=1), m0, out)
        print("graphvar ok sgd", float(out.sum()))
        eng.close()
        n, d = 600, g["feat"].shape[2]
        rng = np.random.default_rng(8)
        adj = np.zeros((3, n, n), np.uint8); feat = np.zeros((3, n, d), np.float32)
        for gi, k in enumerate((550, 30, 300)):
            par = np.array([rng.integers(0, i) for i in range(1, k)])
            adj[gi, np.arange(1, k), par] = 1; adj[gi, par, np.arange(1, k)] = 1
            feat[gi, np.arange(k), rng.integers(0, d, k)] = 1.0
        eng = gnnx.Engine(0)
        eng.set_model({k: g[k] for k in util.WKEYS})
        eng.set_graph_batch(adj, feat, np.array([0, 1, 0], np.int32))
        eoff = eng.plan_graphs([0, 1, 2])
        out = np.zeros(int(eoff[-1]), np.float32)
        eng.explain_graphs_host(eng.make_hparams(num_epochs=EPOCHS, init=_abi.GX_INIT_PHILOX, seed=1), None, out)
        print("graphvar ok large", float(out.sum()))
        eng.close()
    if "misc" in which:
        eng = util.make_engine(fx)
        rows = eng.neighborhood_rows(np.arange(0, 700, 50), 3)
        plan = eng.plan_nodes([300, 5], 3)
        out = np.zeros(plan.total_edges, np.float32)
        eng.explain_nodes_host(eng.make_hparams(num_epochs=2), util.golden_m0(fx, plan), out)
        dense = eng.densify_host(out, int(sum(plan.n(t) ** 2 for t in range(plan.count))))
        print("misc ok", int(rows.sum()), float(dense.sum()))
        eng.close()


if __name__ == "__main__":
    main()
