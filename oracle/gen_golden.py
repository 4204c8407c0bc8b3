"""gen_golden.py -- generates tests/golden/*.npz by EXECUTING THE UNMODIFIED REFERENCE.

Run in the authoring container only (needs /root/reference):
    python oracle/gen_golden.py [--only syn1|syn4|rand|graph|auc|grad|denoise|teacher|trace|opts|variants|options|tu]

What is pinned (SURVEY.md section 8c: the reference has no tests of its own, so the
only possible pin is the reference's own output under a fixed seed):
  * graph + trained model weights + cg 'pred' (gengraph.gen_syn1/gen_syn4 with
    np.random.seed(0); train.train_node_classifier, reference defaults)
  * per explained node: neighbors / node_idx_new from Explainer.extract_neighborhood
    (explain.py:492-501), the mask initialisation M0 drawn exactly as
    ExplainModule.construct_edge_mask does (explain.py:645-652) under
    torch.manual_seed(seed), and the mask returned by Explainer.explain
    (explain.py:74-221), both stored at the directed-edge entries of the
    sub-adjacency in row-major (canonical CSR) order.  Off-edge entries of the
    returned mask are asserted to be exactly 0 here.
"""
import argparse
import math
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def state_to_np(model):
    sd = model.state_dict()
    return {
        "W1": sd["conv_first.weight"].numpy().astype(np.float32),
        "b1": sd["conv_first.bias"].numpy().astype(np.float32),
        "W2": sd["conv_block.0.weight"].numpy().astype(np.float32),
        "b2": sd["conv_block.0.bias"].numpy().astype(np.float32),
        "W3": sd["conv_last.weight"].numpy().astype(np.float32),
        "b3": sd["conv_last.bias"].numpy().astype(np.float32),
        "Wp": sd["pred_model.weight"].numpy().astype(np.float32),
        "bp": sd["pred_model.bias"].numpy().astype(np.float32),
    }


def edges_of(adj):
    iu, ju = np.nonzero(np.triu(adj, 1))
    return np.stack([iu, ju], 1).astype(np.int32)


def explain_nodes_ref(R, model, cg, args, nodes, seed_base):
    """Run the reference explainer; return dict of per-node golden arrays."""
    with ref_harness.quiet():
        ex = R.explain.Explainer(model=model, adj=cg["adj"], feat=cg["feat"], label=cg["label"],
                                 pred=cg["pred"], train_idx=cg["train_idx"], args=args,
                                 writer=None, print_training=False, graph_idx=-1)
    out = {}
    t0 = time.time()
    for node in nodes:
        seed = seed_base + int(node)
        with ref_harness.quiet():
            node_idx_new, sub_adj, sub_feat, sub_label, nbrs = ex.extract_neighborhood(node, 0)
        n = len(nbrs)
        # M0 exactly as construct_edge_mask draws it (explain.py:645-652)
        torch.manual_seed(seed)
        std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (n + n))
        M0 = torch.FloatTensor(n, n).normal_(1.0, std).numpy()
        torch.manual_seed(seed)
        with ref_harness.quiet():
            masked = ex.explain(node, graph_idx=0)
        masked = np.asarray(masked)
        ei, ej = np.nonzero(sub_adj)          # row-major == canonical CSR order
        off = masked.copy()
        off[ei, ej] = 0
        assert np.all(off == 0), "reference mask non-zero off the edges"
        out["n%d_nbrs" % node] = nbrs.astype(np.int32)
        out["n%d_idx_new" % node] = np.int64(node_idx_new)
        out["n%d_seed" % node] = np.int64(seed)
        out["n%d_m0" % node] = M0[ei, ej].astype(np.float32)
        out["n%d_mask" % node] = masked[ei, ej].astype(np.float32)
    print("  explained %d nodes in %.1fs" % (len(nodes), time.time() - t0))
    # sanity of the M0 capture: a 1-epoch run returns A * sym(sigmoid(M0)) (SURVEY 'north_star' table)
    node = int(nodes[0])
    args1 = ref_harness.explainer_args(**{**vars(args), "num_epochs": 1})
    with ref_harness.quiet():
        ex1 = R.explain.Explainer(model=model, adj=cg["adj"], feat=cg["feat"], label=cg["label"],
                                  pred=cg["pred"], train_idx=cg["train_idx"], args=args1,
                                  writer=None, print_training=False, graph_idx=-1)
        torch.manual_seed(seed_base + node)
        m1 = np.asarray(ex1.explain(node, graph_idx=0))
        _, sub_adj, _, _, nbrs = ex1.extract_neighborhood(node, 0)
    n = len(nbrs)
    torch.manual_seed(seed_base + node)
    std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (n + n))
    M0 = torch.FloatTensor(n, n).normal_(1.0, std)
    S = torch.sigmoid(M0)
    exp1 = ((S + S.t()) / 2).numpy() * sub_adj
    assert np.abs(exp1 - m1).max() < 1e-7, "M0 capture does not reproduce the reference's draw"
    return out


def train_args(**over):
    import types
    d = dict(datadir="data", logdir="/tmp/gnnx_ref_log", ckptdir="/tmp/gnnx_ref_ckpt", dataset="syn1",
             bmname=None, opt="adam", opt_scheduler="none", max_nodes=100, cuda="1",
             feature_type="default", lr=0.001, clip=2.0, batch_size=20, num_epochs=1000,
             train_ratio=0.8, test_ratio=0.1, num_workers=1, input_dim=10, hidden_dim=20,
             output_dim=20, num_classes=2, num_gc_layers=3, dropout=0.0, weight_decay=0.005,
             method="base", name_suffix="", assign_ratio=0.1, gpu=False, bias=True, bn=False)
    d.update(over)
    os.makedirs(d["ckptdir"], exist_ok=True)
    os.makedirs(d["logdir"], exist_ok=True)
    return types.SimpleNamespace(**d)


def gen_syn(R, which, nodes, train_epochs):
    np.random.seed(0)
    torch.manual_seed(0)
    fg = R.featgen.ConstFeatureGen(np.ones(10, dtype=float))
    with ref_harness.quiet():
        if which == "syn1":
            G, labels, _ = R.gengraph.gen_syn1(feature_generator=fg)
        else:
            G, labels, _ = R.gengraph.gen_syn4(feature_generator=fg)
    C = max(labels) + 1
    targs = train_args(dataset=which, num_epochs=train_epochs)
    model = R.models.GcnEncoderNode(10, 20, 20, C, 3, bn=False, args=targs)
    t0 = time.time()
    with ref_harness.quiet():
        R.train.train_node_classifier(G, labels, model, targs, writer=None)
    print("  trained %s (%d nodes) in %.1fs" % (which, G.number_of_nodes(), time.time() - t0))
    ck = torch.load(
        R.io_utils.create_filename(targs.ckptdir, targs), weights_only=False)
    cg = ck["cg"]
    model.eval()
    acc = (np.argmax(cg["pred"][0], 1) == cg["label"][0]).mean()
    print("  %s: N=%d edges=%d C=%d acc=%.3f" % (which, cg["adj"].shape[1], int(cg["adj"].sum() / 2), C, acc))
    eargs = ref_harness.explainer_args(dataset=which)
    gold = explain_nodes_ref(R, model, cg, eargs, nodes, seed_base=1000)
    graph = dict(N=np.int64(cg["adj"].shape[1]), edges=edges_of(cg["adj"][0]),
                 feat=cg["feat"][0].astype(np.float32), label=cg["label"][0].astype(np.int64),
                 pred=cg["pred"][0].astype(np.float32), **state_to_np(model))
    np.savez_compressed(os.path.join(OUT, which + "_graph.npz"), **graph)
    np.savez_compressed(os.path.join(OUT, which + "_golden.npz"), nodes=np.asarray(nodes, np.int64), **gold)
    # the dense hop matrix rows for a few nodes pin graph_utils.neighborhoods itself
    with ref_harness.quiet():
        hop = R.graph_utils.neighborhoods(cg["adj"], 3, False)
    np.savez_compressed(os.path.join(OUT, which + "_hops.npz"),
                        hop_rowsum=hop[0].sum(1).astype(np.int32),
                        hop_bits=np.packbits(hop[0].astype(np.uint8), axis=1))


def gen_rand(R):
    """BA graph, Gaussian features, random (untrained) weights AND non-zero biases: exercises
    feature masking and the bias/normalise path harder than the all-ones syn features."""
    import networkx as nx
    rng = np.random.default_rng(7)
    G = nx.barabasi_albert_graph(150, 2, seed=3)
    N, d, C = G.number_of_nodes(), 16, 3
    adj = nx.to_numpy_array(G)[None]
    feat = rng.normal(size=(1, N, d))
    label = rng.integers(0, C, size=(1, N))
    torch.manual_seed(11)
    targs = train_args(input_dim=d)
    model = R.models.GcnEncoderNode(d, 20, 20, C, 3, bn=False, args=targs)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("bias"):
                p.normal_(0.0, 0.3)
    model.eval()
    with torch.no_grad():
        pred, _ = model(torch.tensor(feat, dtype=torch.float), torch.tensor(adj, dtype=torch.float))
    cg = dict(adj=adj, feat=feat, label=label, pred=pred.numpy(), train_idx=list(range(N)))
    eargs = ref_harness.explainer_args(dataset="rand")
    nodes = [0, 1, 7, 33, 77, 100, 149]
    gold = explain_nodes_ref(R, model, cg, eargs, nodes, seed_base=5000)
    graph = dict(N=np.int64(N), edges=edges_of(adj[0]), feat=feat[0].astype(np.float32),
                 label=label[0].astype(np.int64), pred=cg["pred"][0].astype(np.float32),
                 **state_to_np(model))
    np.savez_compressed(os.path.join(OUT, "rand_graph.npz"), **graph)
    np.savez_compressed(os.path.join(OUT, "rand_golden.npz"), nodes=np.asarray(nodes, np.int64), **gold)


def gen_short_horizon(R, which, epochs):
    """Same graph / weights / seeds as <which>_golden.npz, but the reference runs only `epochs` mask-
    optimisation epochs.  Some 100-epoch trajectories are chaotic (DESIGN.md 'Parity'): a short horizon
    pins the arithmetic of EVERY node before rounding differences are amplified."""
    g = np.load(os.path.join(OUT, which + "_graph.npz"))
    gold = np.load(os.path.join(OUT, which + "_golden.npz"))
    N = int(g["N"])
    adj = np.zeros((1, N, N))
    adj[0, g["edges"][:, 0], g["edges"][:, 1]] = 1
    adj[0, g["edges"][:, 1], g["edges"][:, 0]] = 1
    C = g["Wp"].shape[0]
    targs = train_args(dataset=which)
    model = R.models.GcnEncoderNode(g["feat"].shape[1], 20, 20, C, 3, bn=False, args=targs)
    sd = {"conv_first.weight": g["W1"], "conv_first.bias": g["b1"], "conv_block.0.weight": g["W2"],
          "conv_block.0.bias": g["b2"], "conv_last.weight": g["W3"], "conv_last.bias": g["b3"],
          "pred_model.weight": g["Wp"], "pred_model.bias": g["bp"]}
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    model.eval()
    eargs = ref_harness.explainer_args(dataset=which, num_epochs=epochs)
    with ref_harness.quiet():
        ex = R.explain.Explainer(model=model, adj=adj, feat=g["feat"][None].astype(np.float64), label=g["label"][None],
                                 pred=g["pred"][None], train_idx=list(range(N)), args=eargs,
                                 writer=None, print_training=False, graph_idx=-1)
    out = {}
    for node in gold["nodes"]:
        node = int(node)
        torch.manual_seed(int(gold["n%d_seed" % node]))
        with ref_harness.quiet():
            masked = np.asarray(ex.explain(node, graph_idx=0))
            _, sub_adj, _, _, nbrs = ex.extract_neighborhood(node, 0)
        assert np.array_equal(nbrs, gold["n%d_nbrs" % node])
        ei, ej = np.nonzero(sub_adj)
        out["n%d_mask" % node] = masked[ei, ej].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "%s_golden_e%d.npz" % (which, epochs)), nodes=gold["nodes"],
                        num_epochs=np.int64(epochs), **out)
    print("  %s: %d nodes at %d epochs" % (which, len(gold["nodes"]), epochs))


def gen_graph_mode(R, epochs_list=(10, 100)):
    """Graph-classification mode (explain.py:80-85,356-363; models.py:269-316): synthetic stand-in for
    Mutagenicity (dataset absent, no network): padded molecule-like graphs, one-hot 14-d node features,
    GcnEncoderGraph(14,20,20,2,3) with random weights and non-zero biases."""
    import networkx as nx
    rng = np.random.default_rng(21)
    G_n, max_nodes, d, C = 12, 40, 14, 2
    adj = np.zeros((G_n, max_nodes, max_nodes)); feat = np.zeros((G_n, max_nodes, d)); label = rng.integers(0, C, G_n)
    num_nodes = []
    for g in range(G_n):
        n = int(rng.integers(6, 36))
        T = nx.random_labeled_tree(n, seed=int(rng.integers(1 << 30))) if hasattr(nx, "random_labeled_tree") else nx.random_tree(n, seed=int(rng.integers(1 << 30)))
        for _ in range(max(1, n // 6)):
            u, v = rng.integers(0, n, 2)
            if u != v:
                T.add_edge(int(u), int(v))
        if g == 3:                       # one graph with an isolated real node
            T.remove_edges_from(list(T.edges(0)))
        A = nx.to_numpy_array(T, nodelist=range(n))
        adj[g, :n, :n] = A
        feat[g, np.arange(n), rng.integers(0, d, n)] = 1.0
        num_nodes.append(n)
    torch.manual_seed(3)
    targs = train_args(input_dim=d)
    model = R.models.GcnEncoderGraph(d, 20, 20, C, 3, bn=False, args=targs)
    with torch.no_grad():
        for name, p_ in model.named_parameters():
            if name.endswith("bias"):
                p_.normal_(0.0, 0.3)
    model.eval()
    with torch.no_grad():
        pred = np.stack([model(torch.tensor(feat[g:g + 1], dtype=torch.float), torch.tensor(adj[g:g + 1], dtype=torch.float))[0][0].numpy()
                         for g in range(G_n)])[None]
    out = dict(num_graphs=np.int64(G_n), max_nodes=np.int64(max_nodes), adj=adj.astype(np.uint8), feat=feat.astype(np.float32),
               label=label.astype(np.int64), pred=pred.astype(np.float32), num_nodes=np.asarray(num_nodes, np.int64), **state_to_np(model))
    for epochs in epochs_list:
        eargs = ref_harness.explainer_args(dataset="graphs", num_epochs=epochs)
        with ref_harness.quiet():
            ex = R.explain.Explainer(model=model, adj=torch.tensor(adj, dtype=torch.float), feat=torch.tensor(feat, dtype=torch.float),
                                     label=torch.tensor(label), pred=pred, train_idx=list(range(G_n)), args=eargs,
                                     writer=None, print_training=False, graph_mode=True, graph_idx=0)
        for g in range(G_n):
            seed = 7000 + g
            if epochs == epochs_list[0]:
                torch.manual_seed(seed)
                std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (max_nodes + max_nodes))
                M0 = torch.FloatTensor(max_nodes, max_nodes).normal_(1.0, std).numpy()
                ei, ej = np.nonzero(adj[g])
                out["g%d_m0" % g] = M0[ei, ej].astype(np.float32)
                out["g%d_seed" % g] = np.int64(seed)
            torch.manual_seed(seed)
            with ref_harness.quiet():
                masked = np.asarray(ex.explain(node_idx=0, graph_idx=g, graph_mode=True))
            ei, ej = np.nonzero(adj[g])
            off = masked.copy(); off[ei, ej] = 0
            assert np.all(off == 0)
            out["g%d_mask_e%d" % (g, epochs)] = masked[ei, ej].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "graphs_golden.npz"), **out)
    print("  graph mode: %d graphs, max_nodes %d, epochs %s" % (G_n, max_nodes, list(epochs_list)))


def gen_auc(R):
    """Known-answer check downstream of the masks: Explainer.make_pred_real (explain.py:535-579) + roc_auc_score
    (explain.py:328) evaluated BY THE REFERENCE on its own golden masks (motif-start nodes only)."""
    from sklearn.metrics import roc_auc_score
    import types
    out = {}
    for which, nodes in (("syn1", [300, 350, 400, 450, 550, 620]), ("syn4", [511])):
        gold = np.load(os.path.join(OUT, which + "_golden.npz"))
        g = np.load(os.path.join(OUT, which + "_graph.npz"))
        N = int(g["N"])
        A = np.zeros((N, N)); A[g["edges"][:, 0], g["edges"][:, 1]] = 1; A[g["edges"][:, 1], g["edges"][:, 0]] = 1
        fake = types.SimpleNamespace(args=types.SimpleNamespace(dataset=which))
        preds, reals = [], []
        nodes = [n for n in nodes if ("n%d_mask" % n) in gold]
        for node in nodes:
            nbrs = gold["n%d_nbrs" % node]
            sub = A[nbrs][:, nbrs]
            ei, ej = np.nonzero(sub)
            M = np.zeros_like(sub); M[ei, ej] = gold["n%d_mask" % node]
            pred, real = R.explain.Explainer.make_pred_real(fake, M, int(gold["n%d_idx_new" % node]))
            out["%s_n%d_real" % (which, node)] = real.astype(np.uint8)
            out["%s_n%d_pred" % (which, node)] = pred.astype(np.float32)
            preds.append(pred); reals.append(real)
        out[which + "_nodes"] = np.asarray(nodes, np.int64)
        out[which + "_auc"] = np.float64(roc_auc_score(np.concatenate(reals), np.concatenate(preds)))
        print("  %s: AUC of the reference on %d golden nodes = %.4f" % (which, len(nodes), out[which + "_auc"]))
    np.savez_compressed(os.path.join(OUT, "auc_golden.npz"), **out)


def gen_grad(R):
    """Gradient baseline (explain(model="grad"), explain.py:125-133,717-738) of the unmodified reference on the syn1
    and rand fixtures' graphs/weights -> tests/golden/grad_golden.npz (per node: mask entries at the nonzeros of sub_adj)."""
    import gnnx_oracle as O
    out = {}
    for which, nodes in (("syn1", [300, 450, 683, 13, 0, 699]), ("rand", [0, 7, 33, 100, 149])):
        g = np.load(os.path.join(OUT, which + "_graph.npz"))
        N = int(g["N"]); d = g["feat"].shape[1]; C = g["Wp"].shape[0]
        adj = np.zeros((1, N, N)); e = g["edges"]; adj[0, e[:, 0], e[:, 1]] = 1; adj[0, e[:, 1], e[:, 0]] = 1
        model = R.models.GcnEncoderNode(d, 20, 20, C, 3, bn=False, args=train_args(input_dim=d))
        sd = {"conv_first.weight": g["W1"], "conv_first.bias": g["b1"], "conv_block.0.weight": g["W2"], "conv_block.0.bias": g["b2"],
              "conv_last.weight": g["W3"], "conv_last.bias": g["b3"], "pred_model.weight": g["Wp"], "pred_model.bias": g["bp"]}
        model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
        model.eval()
        cg = dict(adj=adj, feat=g["feat"][None].astype(np.float64), label=g["label"][None], pred=g["pred"][None], train_idx=list(range(N)))
        args = ref_harness.explainer_args(dataset=which)
        with ref_harness.quiet():
            ex = R.explain.Explainer(model=model, adj=cg["adj"], feat=cg["feat"], label=cg["label"], pred=cg["pred"],
                                     train_idx=cg["train_idx"], args=args, writer=None, print_training=False, graph_idx=-1)
        W = {k: g[k] for k in ["W1", "b1", "W2", "b2", "W3", "b3", "Wp", "bp"]}
        for node in nodes:
            with ref_harness.quiet():
                torch.manual_seed(1)
                masked = np.asarray(ex.explain(node, graph_idx=0, model="grad"))
                idx_new, sub_adj, sub_feat, sub_label, nbrs = ex.extract_neighborhood(node, 0)
            ei, ej = np.nonzero(sub_adj)
            off = masked.copy(); off[ei, ej] = 0
            assert np.all(off == 0)
            out["%s_n%d_mask" % (which, node)] = masked[ei, ej].astype(np.float32)
            # the oracle restatement must agree with the reference
            pl = int(np.argmax(g["pred"][nbrs], 1)[idx_new])
            mine = O.grad_baseline_dense_torch(sub_adj, sub_feat, pl, idx_new, W)
            err = O.rel_l2(mine[ei, ej], masked[ei, ej])
            assert err < 1e-6, (which, node, err)
        out[which + "_nodes"] = np.asarray(nodes, np.int64)
    np.savez_compressed(os.path.join(OUT, "grad_golden.npz"), **out)
    print("  grad baseline golden written")


def gen_variants(R, epochs=30):
    """Model variants the kernels do not build yet (SURVEY 8 f3: --bn, num_gc_layers != 3), pinned for the oracle now:
    the unmodified reference on the rand graph with random weights, 2 / 4 layers and 3 layers + --bn ->
    tests/golden/variants_golden.npz (weights, per node M0 at the edges and the returned mask at the edges)."""
    import networkx as nx
    rng = np.random.default_rng(21)
    G = nx.barabasi_albert_graph(60, 2, seed=4)
    N, d, C = G.number_of_nodes(), 12, 3
    adj = nx.to_numpy_array(G)[None]
    feat = rng.normal(size=(1, N, d))
    label = rng.integers(0, C, size=(1, N))
    out = dict(N=np.int64(N), edges=edges_of(adj[0]), feat=feat[0].astype(np.float32), label=label[0].astype(np.int64), num_epochs=np.int64(epochs))
    for tag, L, bn in (("L2", 2, False), ("L4", 4, False), ("bn", 3, True)):
        torch.manual_seed(100 + L + int(bn))
        targs = train_args(input_dim=d, num_gc_layers=L, bn=bn)
        model = R.models.GcnEncoderNode(d, 20, 20, C, L, bn=bn, args=targs)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith("bias"):
                    p.normal_(0.0, 0.3)
        model.eval()
        with torch.no_grad():
            pred, _ = model(torch.tensor(feat, dtype=torch.float), torch.tensor(adj, dtype=torch.float))
        cg = dict(adj=adj, feat=feat, label=label, pred=pred.numpy(), train_idx=list(range(N)))
        eargs = ref_harness.explainer_args(dataset="var" + tag, num_gc_layers=L, bn=bn, num_epochs=epochs)
        nodes = [0, 5, 17, 40]
        gold = explain_nodes_ref(R, model, cg, eargs, nodes, seed_base=7000 + 10 * L)
        sd = model.state_dict()
        keys = ["conv_first"] + ["conv_block.%d" % i for i in range(L - 2)] + ["conv_last"]
        for l, k in enumerate(keys, 1):
            out["%s_W%d" % (tag, l)] = sd[k + ".weight"].numpy().astype(np.float32)
            out["%s_b%d" % (tag, l)] = sd[k + ".bias"].numpy().astype(np.float32)
        out[tag + "_Wp"] = sd["pred_model.weight"].numpy().astype(np.float32)
        out[tag + "_bp"] = sd["pred_model.bias"].numpy().astype(np.float32)
        out[tag + "_pred"] = cg["pred"][0].astype(np.float32)
        out[tag + "_nodes"] = np.asarray(nodes, np.int64)
        for k, v in gold.items():
            out[tag + "_" + k] = v
    np.savez_compressed(os.path.join(OUT, "variants_golden.npz"), **out)
    print("  variants golden written")


def gen_options(R, node=5, seed=77, epochs=12):
    """--mask-bias and --mask-act ReLU (SURVEY 8 f3; explain.py:657-660,673-676,755-770): the unmodified reference on a BA(40, 2)
    graph with a randomly initialised model, run with the default options, with --mask-bias and with --mask-act ReLU under the same
    seed -> tests/golden/options_golden.npz (graph, weights, M0 at the edges and the three returned (n, n) masks)."""
    import networkx as nx
    rng = np.random.default_rng(3)
    G = nx.barabasi_albert_graph(40, 2, seed=5)
    N, d, C = 40, 8, 3
    adj = nx.to_numpy_array(G)[None]
    feat = rng.normal(size=(1, N, d))
    label = rng.integers(0, C, size=(1, N))
    torch.manual_seed(2)
    model = R.models.GcnEncoderNode(d, 20, 20, C, 3, bn=False, args=train_args(input_dim=d))
    model.eval()
    with torch.no_grad():
        pred, _ = model(torch.tensor(feat, dtype=torch.float), torch.tensor(adj, dtype=torch.float))
    cg = dict(adj=adj, feat=feat, label=label, pred=pred.numpy(), train_idx=list(range(N)))
    gold = explain_nodes_ref(R, model, cg, ref_harness.explainer_args(dataset="opt", num_epochs=epochs), [node], seed_base=seed - node)
    out = dict(N=np.int64(N), edges=edges_of(adj[0]), feat=feat[0], label=label[0].astype(np.int64), pred=cg["pred"][0].astype(np.float32),
               node=np.int64(node), num_epochs=np.int64(epochs), **state_to_np(model), **gold)
    for tag, over in (("default", {}), ("mask_bias", dict(mask_bias=True)), ("relu", dict(mask_act="ReLU"))):
        args = ref_harness.explainer_args(dataset="opt", num_epochs=epochs, **over)
        with ref_harness.quiet():
            ex = R.explain.Explainer(model=model, adj=cg["adj"], feat=cg["feat"], label=cg["label"], pred=cg["pred"],
                                     train_idx=cg["train_idx"], args=args, writer=None, print_training=False, graph_idx=-1)
            torch.manual_seed(seed)
            out[tag + "_mask"] = np.asarray(ex.explain(node, graph_idx=0), np.float32)
    np.savez_compressed(os.path.join(OUT, "options_golden.npz"), **out)
    print("  option-variant golden written")


def gen_tu(R, max_nodes=10):
    """utils/io_utils.read_graphfile (io_utils.py:426-562) of the unmodified reference on the toy TU-format dataset that
    tests/util.write_tu_toy writes with seed 4 -> tests/golden/tu_golden.npz: per graph kept, the adjacency padded to max_nodes
    (diagonal zeroed), the graph label and the node features."""
    import tempfile
    import networkx as nx
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
    import util
    with tempfile.TemporaryDirectory() as tmp:
        util.write_tu_toy(tmp, "TOY", np.random.default_rng(4))
        ver, nx.__version__ = nx.__version__, "2.5"      # the reference parses the version as a float (io_utils.py:551)
        try:
            graphs = R.io_utils.read_graphfile(tmp, "TOY", max_nodes=max_nodes)
        finally:
            nx.__version__ = ver
    out = dict(count=np.int64(len(graphs)))
    for g, Gx in enumerate(graphs):
        n = Gx.number_of_nodes()
        A = np.zeros((max_nodes, max_nodes)); A[:n, :n] = nx.to_numpy_array(Gx)
        np.fill_diagonal(A, 0)
        out["g%d_adj" % g] = A
        out["g%d_label" % g] = np.int64(Gx.graph["label"])
        out["g%d_feat" % g] = np.array([np.asarray(Gx.nodes[u]["label"], np.float32) for u in Gx.nodes()])
    np.savez_compressed(os.path.join(OUT, "tu_golden.npz"), **out)
    print("  TU-reader golden written: %d graphs" % len(graphs))


OPT_VARIANTS = (("sgd", dict(opt="sgd")), ("rmsprop", dict(opt="rmsprop")), ("adagrad", dict(opt="adagrad")),
                ("adamstep", dict(opt="adam", opt_scheduler="step", opt_decay_step=8, opt_decay_rate=0.5)),
                ("adamcos", dict(opt="adam", opt_scheduler="cos", opt_restart=12)),
                ("sgdstep", dict(opt="sgd", opt_scheduler="step", opt_decay_step=10, opt_decay_rate=0.3)))


def gen_opts(R, epochs=30):
    """Optimiser / scheduler variants (SURVEY 8 f3; utils/train_utils.py:7-23, explain.py:145-146,622): the unmodified reference
    on the rand fixture (its graph, trained weights, nodes and seeds) with --opt sgd / rmsprop / adagrad and the step / cos
    schedulers -> tests/golden/opts_golden.npz (per variant and node: the returned mask at the edges; M0 = rand_golden's)."""
    import gnnx_oracle as O
    out = dict(num_epochs=np.int64(epochs))
    for tag, over in OPT_VARIANTS:
        make, g, gold = _load_fixture_model(R, "rand", num_epochs=epochs, **over)
        ex = make()
        nodes = [int(x) for x in gold["nodes"]]
        for node in nodes:
            torch.manual_seed(int(gold["n%d_seed" % node]))
            with ref_harness.quiet():
                node_idx_new, sub_adj, sub_feat, sub_label, nbrs = ex.extract_neighborhood(node, 0)
                masked = np.asarray(ex.explain(node, graph_idx=0))
            ei, ej = np.nonzero(sub_adj)
            out["%s_n%d_mask" % (tag, node)] = masked[ei, ej].astype(np.float32)
            # the oracle restatement must agree with the reference bit for bit
            M0 = np.ones(sub_adj.shape, np.float32); M0[ei, ej] = gold["n%d_m0" % node]
            W = {k: g[k] for k in ["W1", "b1", "W2", "b2", "W3", "b3", "Wp", "bp"]}
            pl = np.argmax(g["pred"][nbrs], 1)
            mine = O.explain_dense_torch(sub_adj, sub_feat, int(g["label"][node]), pl, node_idx_new, W, M0, hp=O.default_hparams(num_epochs=epochs, **over))
            err = O.rel_l2(mine[ei, ej], masked[ei, ej])
            assert err < 1e-6, (tag, node, err)
        out[tag + "_nodes"] = np.asarray(nodes, np.int64)
        print("  %s: %d nodes" % (tag, len(nodes)))
    np.savez_compressed(os.path.join(OUT, "opts_golden.npz"), **out)
    print("  optimiser-variant golden written")


def _load_fixture_model(R, which, **eargs_over):
    """(explainer, graph npz, golden npz) of a committed fixture: the reference Explainer on the fixture's graph and weights."""
    g = np.load(os.path.join(OUT, which + "_graph.npz"))
    gold = np.load(os.path.join(OUT, which + "_golden.npz"))
    N = int(g["N"]); d = g["feat"].shape[1]; C = g["Wp"].shape[0]
    adj = np.zeros((1, N, N)); e = g["edges"]; adj[0, e[:, 0], e[:, 1]] = 1; adj[0, e[:, 1], e[:, 0]] = 1
    model = R.models.GcnEncoderNode(d, 20, 20, C, 3, bn=False, args=train_args(input_dim=d))
    sd = {"conv_first.weight": g["W1"], "conv_first.bias": g["b1"], "conv_block.0.weight": g["W2"], "conv_block.0.bias": g["b2"],
          "conv_last.weight": g["W3"], "conv_last.bias": g["b3"], "pred_model.weight": g["Wp"], "pred_model.bias": g["bp"]}
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    model.eval()

    def make(print_training=False, **over):
        args = ref_harness.explainer_args(dataset=which, **{**eargs_over, **over})
        with ref_harness.quiet():
            return R.explain.Explainer(model=model, adj=adj, feat=g["feat"][None].astype(np.float64), label=g["label"][None], pred=g["pred"][None],
                                       train_idx=list(range(N)), args=args, writer=None, print_training=print_training, graph_idx=-1)
    return make, g, gold


def gen_teacher(R, steps=(25, 50, 75)):
    """Teacher-forcing fixtures (immune to chaotic trajectories): the optimiser state of the UNMODIFIED reference after t0 Adam steps
    and after t0+1, captured by wrapping torch.optim.Adam.step while Explainer.explain runs (nothing in the reference is modified).
    A kernel that is handed the state at t0 must reproduce the state at t0+1 to rounding, on the chaotic syn1 nodes too.
    -> tests/golden/teacher_golden.npz: per (fixture, node, t0): M / exp_avg / exp_avg_sq at the edge slots, feat_mask state (3,d),
    and after one more step: M at the edges, sigmoid-symmetrised mask at the edges (what forward() builds), sigmoid(feat_mask)."""
    out = {"steps": np.asarray(steps, np.int64)}
    orig = torch.optim.Adam.step
    for which, nodes in (("syn1", [0, 3, 33, 163, 293, 300, 683]), ("rand", [0, 33, 149])):
        make, g, gold = _load_fixture_model(R, which)
        ex = make()
        out[which + "_nodes"] = np.asarray(nodes, np.int64)
        for node in nodes:
            cap = {}

            def hooked(self, *a, **k):
                r = orig(self, *a, **k)
                ps = self.param_groups[0]["params"]
                t = int(self.state[ps[0]]["step"])
                if t in steps or (t - 1) in steps:
                    cap[t] = [(p.detach().clone().numpy(), self.state[p]["exp_avg"].clone().numpy(), self.state[p]["exp_avg_sq"].clone().numpy()) for p in ps]
                return r
            torch.optim.Adam.step = hooked
            try:
                torch.manual_seed(int(gold["n%d_seed" % node]))
                with ref_harness.quiet():
                    masked = np.asarray(ex.explain(node, graph_idx=0))
                    _, sub_adj, _, _, nbrs = ex.extract_neighborhood(node, 0)
            finally:
                torch.optim.Adam.step = orig
            ei, ej = np.nonzero(sub_adj)
            assert np.abs(masked[ei, ej] - gold["n%d_mask" % node]).max() == 0, "instrumented run differs from the golden run"
            for t0 in steps:
                (M, m, v), (F, mF, vF) = cap[t0]
                (M1, _, _), (F1, _, _) = cap[t0 + 1]
                key = "%s_n%d_t%d_" % (which, node, t0)
                out[key + "M"] = M[ei, ej].astype(np.float32); out[key + "m"] = m[ei, ej].astype(np.float32); out[key + "v"] = v[ei, ej].astype(np.float32)
                out[key + "feat"] = np.stack([F, mF, vF]).astype(np.float32)
                out[key + "M_next"] = M1[ei, ej].astype(np.float32)
                S = torch.sigmoid(torch.tensor(M1))
                out[key + "mask_next"] = ((S + S.t()) / 2).numpy()[ei, ej].astype(np.float32)      # explain.py:665-678
                out[key + "sF_next"] = torch.sigmoid(torch.tensor(F1)).numpy().astype(np.float32)
        print("  teacher: %s %d nodes x %d steps" % (which, len(nodes), len(steps)))
    np.savez_compressed(os.path.join(OUT, "teacher_golden.npz"), **out)


def gen_trace(R, epochs=12):
    """SURVEY 8 row a12: what print_training=True prints every epoch (explain.py:148-159) -- loss, mask density, softmax row --
    parsed from the stdout of the UNMODIFIED reference.  M0 is not stored: the test regenerates the (n,n) draw from the seed.
    -> tests/golden/trace_golden.npz"""
    import contextlib, io, re
    out = {"num_epochs": np.int64(epochs)}
    for which, nodes in (("syn1", [300, 683, 13]), ("rand", [0, 33])):
        make, g, gold = _load_fixture_model(R, which, num_epochs=epochs)
        ex = make(print_training=True)
        out[which + "_nodes"] = np.asarray(nodes, np.int64)
        for node in nodes:
            buf = io.StringIO()
            torch.manual_seed(int(gold["n%d_seed" % node]))
            torch.set_printoptions(precision=8, sci_mode=False)
            with contextlib.redirect_stdout(buf):
                ex.explain(node, graph_idx=0)
            rows = []
            for mt in re.finditer(r"epoch:\s+(\d+)\s+; loss:\s+(\S+)\s+; mask density:\s+(\S+)\s+; pred:\s+tensor\(\[([^\]]*)\]", buf.getvalue()):
                rows.append([float(mt.group(2)), float(mt.group(3))] + [float(x) for x in mt.group(4).replace("\n", " ").split(",")])
            assert len(rows) == epochs, (which, node, len(rows), buf.getvalue()[:300])
            out["%s_n%d_trace" % (which, node)] = np.asarray(rows, np.float64)      # [epoch] = (loss, density, softmax row)
        print("  trace: %s %d nodes x %d epochs" % (which, len(nodes), epochs))
    torch.set_printoptions(profile="default")
    np.savez_compressed(os.path.join(OUT, "trace_golden.npz"), **out)


def gen_denoise(R, k=20):
    """io_utils.denoise_graph(masked_adj, node_idx_new, threshold_num=20) of the UNMODIFIED reference (utils/io_utils.py:193-245) on
    its own golden masks -> tests/golden/denoise_golden.npz: per node the thresholded edge list (max_component=False) and the node
    set of the largest component (max_component=True), plus precision_recall_curve of the six motif-start nodes (explain.py:329)."""
    from sklearn.metrics import precision_recall_curve
    out = {"threshold_num": np.int64(k)}
    for which, nodes in (("syn1", [300, 350, 400, 450, 550, 620, 0, 13]), ("syn4", [511, 512])):
        gold = np.load(os.path.join(OUT, which + "_golden.npz"))
        g = np.load(os.path.join(OUT, which + "_graph.npz"))
        N = int(g["N"])
        A = np.zeros((N, N)); A[g["edges"][:, 0], g["edges"][:, 1]] = 1; A[g["edges"][:, 1], g["edges"][:, 0]] = 1
        nodes = [n for n in nodes if ("n%d_mask" % n) in gold]
        out[which + "_nodes"] = np.asarray(nodes, np.int64)
        for node in nodes:
            nbrs = gold["n%d_nbrs" % node]
            sub = A[nbrs][:, nbrs]
            ei, ej = np.nonzero(sub)
            M = np.zeros_like(sub); M[ei, ej] = gold["n%d_mask" % node]
            idx = int(gold["n%d_idx_new" % node])
            G0 = R.io_utils.denoise_graph(M.copy(), idx, threshold_num=k, max_component=False)
            G1 = R.io_utils.denoise_graph(M.copy(), idx, threshold_num=k, max_component=True)
            e = np.array(sorted((min(u, v), max(u, v)) for u, v in G0.edges()), np.int32).reshape(-1, 2)
            out["%s_n%d_edges" % (which, node)] = e
            out["%s_n%d_weights" % (which, node)] = np.array([G0[u][v]["weight"] for u, v in e], np.float32)
            out["%s_n%d_cc" % (which, node)] = np.array(sorted(G1.nodes()), np.int32)
    au = np.load(os.path.join(OUT, "auc_golden.npz"))
    real = np.concatenate([au["syn1_n%d_real" % n] for n in au["syn1_nodes"]]); pred = np.concatenate([au["syn1_n%d_pred" % n] for n in au["syn1_nodes"]])
    pr, rc, th = precision_recall_curve(real, pred)
    out["syn1_pr_precision"] = pr; out["syn1_pr_recall"] = rc; out["syn1_pr_thresholds"] = th
    np.savez_compressed(os.path.join(OUT, "denoise_golden.npz"), **out)
    print("  denoise golden written")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    ap.add_argument("--short", type=int, default=0, help="also/only generate the short-horizon golden (epochs)")
    a = ap.parse_args()
    if a.only == "auc":
        gen_auc(ref_harness.load())
        return
    if a.only == "grad":
        gen_grad(ref_harness.load())
        return
    if a.only == "denoise":
        gen_denoise(ref_harness.load())
        return
    if a.only == "teacher":
        torch.set_num_threads(8)
        gen_teacher(ref_harness.load())
        return
    if a.only == "trace":
        torch.set_num_threads(8)
        gen_trace(ref_harness.load())
        return
    if a.only == "opts":
        torch.set_num_threads(8)
        gen_opts(ref_harness.load())
        return
    if a.only == "variants":
        torch.set_num_threads(8)
        gen_variants(ref_harness.load())
        return
    if a.only == "graph":
        torch.set_num_threads(8)
        gen_graph_mode(ref_harness.load())
        return
    if a.only == "options":
        gen_options(ref_harness.load())
        return
    if a.only == "tu":
        gen_tu(ref_harness.load())
        return
    if a.short:
        torch.set_num_threads(8)
        R = ref_harness.load()
        for which in (["syn1", "syn4", "rand"] if a.only is None else [a.only]):
            gen_short_horizon(R, which, a.short)
        return
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    R = ref_harness.load()
    if a.only in (None, "syn1"):
        nodes = sorted(set([300, 301, 400, 550, 699, 10, 0, 5, 350, 450, 620, 683] + list(range(3, 700, 10))))
        gen_syn(R, "syn1", nodes, 1000)
    if a.only in (None, "syn4"):
        nodes = sorted(set([512, 0, 1, 8, 100, 511, 870] + list(range(4, 871, 20))))
        gen_syn(R, "syn4", nodes, 1000)
    if a.only in (None, "rand"):
        gen_rand(R)


if __name__ == "__main__":
    main()
