"""gen_graph_variants_golden.py -- graph-classification mode with model and optimiser variants, pinned by EXECUTING THE
UNMODIFIED REFERENCE (needs the reference tree, see oracle/ref_harness.py):

    python tools/gen_graph_variants_golden.py        -> tests/golden/graph_variants_golden.npz

Graphs: the 12 padded molecule-like graphs of tests/golden/graphs_golden.npz (max_nodes 40, d = 14, C = 2).
Model cases: GcnEncoderGraph with random weights and non-zero biases -- 2 layers, 4 layers, --bn, 4 layers + --bn, widths
64/48, widths 128/96 with 2 layers.  Optimiser cases: the 3-layer 20/20 model of graphs_golden.npz with --opt sgd / rmsprop /
adagrad, Adam + step scheduler, sgd + cos scheduler.  30 epochs; per graph the mask initialisation M0 (torch.manual_seed(7000 + g),
drawn at the padded size like construct_edge_mask, explain.py:645-652) and the returned mask, both at the adjacency entries in
row-major order.  The torch port (oracle/gnnx_oracle.explain_dense_torch) is checked against every returned mask here.
"""
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import gen_golden  # noqa: E402
import gnnx_oracle as O  # noqa: E402
import ref_harness  # noqa: E402

MODEL_CASES = (("L2", 2, False, 20, 20), ("L4", 4, False, 20, 20), ("bn", 3, True, 20, 20), ("L4bn", 4, True, 20, 20),
               ("w64", 3, False, 64, 48), ("w128", 2, False, 128, 96))
OPT_CASES = (("sgd", dict(opt="sgd")), ("rmsprop", dict(opt="rmsprop")), ("adagrad", dict(opt="adagrad")),
             ("adamstep", dict(opt="adam", opt_scheduler="step", opt_decay_step=8, opt_decay_rate=0.5)),
             ("sgdcos", dict(opt="sgd", opt_scheduler="cos", opt_restart=12)))


def model_weights_np(model, L):
    sd = model.state_dict()
    keys = ["conv_first"] + ["conv_block.%d" % i for i in range(L - 2)] + ["conv_last"]
    w = {}
    for l, k in enumerate(keys, 1):
        w["W%d" % l] = sd[k + ".weight"].numpy().astype(np.float32)
        w["b%d" % l] = sd[k + ".bias"].numpy().astype(np.float32)
    w["Wp"] = sd["pred_model.weight"].numpy().astype(np.float32)
    w["bp"] = sd["pred_model.bias"].numpy().astype(np.float32)
    return w


def main(epochs=30):
    R = ref_harness.load()
    gg = np.load(os.path.join(gen_golden.OUT, "graphs_golden.npz"))
    G_n, n, d, C = int(gg["num_graphs"]), int(gg["max_nodes"]), gg["feat"].shape[2], 2
    adj, feat, label = gg["adj"].astype(np.float64), gg["feat"].astype(np.float32), gg["label"].astype(np.int64)
    out = dict(num_epochs=np.int64(epochs), num_graphs=np.int64(G_n), max_nodes=np.int64(n))
    for g in range(G_n):
        torch.manual_seed(7000 + g)
        std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (n + n))
        M0 = torch.FloatTensor(n, n).normal_(1.0, std).numpy()
        ei, ej = np.nonzero(adj[g])
        out["g%d_m0" % g] = M0[ei, ej].astype(np.float32)
        out["g%d_seed" % g] = np.int64(7000 + g)

    def run(tag, model, L, bn, w, **eover):
        eargs = ref_harness.explainer_args(dataset="gvar" + tag, num_gc_layers=L, bn=bn, num_epochs=epochs, **eover)
        with ref_harness.quiet():
            ex = R.explain.Explainer(model=model, adj=torch.tensor(adj, dtype=torch.float), feat=torch.tensor(feat, dtype=torch.float),
                                     label=torch.tensor(label), pred=np.zeros((1, G_n, C), np.float32), train_idx=list(range(G_n)), args=eargs,
                                     writer=None, print_training=False, graph_mode=True, graph_idx=0)
        worst = 0.0
        for g in range(G_n):
            torch.manual_seed(7000 + g)
            with ref_harness.quiet():
                masked = np.asarray(ex.explain(node_idx=0, graph_idx=g, graph_mode=True))
            ei, ej = np.nonzero(adj[g])
            off = masked.copy(); off[ei, ej] = 0
            assert np.all(off == 0), "reference mask non-zero off the edges"
            out["%s_g%d_mask" % (tag, g)] = masked[ei, ej].astype(np.float32)
            torch.manual_seed(7000 + g)
            std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (n + n))
            M0 = torch.FloatTensor(n, n).normal_(1.0, std).numpy()
            mine = O.explain_dense_torch(adj[g], feat[g], int(label[g]), None, 0, w, M0,
                                         hp=O.default_hparams(num_epochs=epochs, **eover), graph_mode=True, bn=bn)
            worst = max(worst, O.rel_l2(mine[ei, ej], masked[ei, ej]))
        assert worst < 1e-6, (tag, worst)
        print("  %s: %d graphs, torch port rel-L2 %.1e" % (tag, G_n, worst))

    for k, (tag, L, bn, hid, emb) in enumerate(MODEL_CASES):
        torch.manual_seed(300 + k)
        model = R.models.GcnEncoderGraph(d, hid, emb, C, L, bn=bn, args=gen_golden.train_args(input_dim=d, num_gc_layers=L, bn=bn))
        with torch.no_grad():
            for name, p_ in model.named_parameters():
                if name.endswith("bias"):
                    p_.normal_(0.0, 0.3)
        model.eval()
        w = model_weights_np(model, L)
        for key, v in w.items():
            out["%s_%s" % (tag, key)] = v
        out[tag + "_L"] = np.int64(L); out[tag + "_bn"] = np.int64(bn)
        run(tag, model, L, bn, w)
    # optimiser cases: the 3-layer 20/20 model of graphs_golden.npz
    model = R.models.GcnEncoderGraph(d, 20, 20, C, 3, bn=False, args=gen_golden.train_args(input_dim=d))
    keys = {"conv_first.weight": "W1", "conv_first.bias": "b1", "conv_block.0.weight": "W2", "conv_block.0.bias": "b2",
            "conv_last.weight": "W3", "conv_last.bias": "b3", "pred_model.weight": "Wp", "pred_model.bias": "bp"}
    model.load_state_dict({k: torch.tensor(gg[v]) for k, v in keys.items()})
    model.eval()
    w = {v: gg[v] for v in keys.values()}
    for tag, over in OPT_CASES:
        run(tag, model, 3, False, w, **over)
    dst = os.path.join(gen_golden.OUT, "graph_variants_golden.npz")
    np.savez_compressed(dst, **out)
    print("  written %s" % dst)


if __name__ == "__main__":
    main()
