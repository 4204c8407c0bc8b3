"""Drop-in for the reference's explainer/explain.py:Explainer (node-classification path).

Same constructor, same method names/arguments, same return values (dense (n,n) float64 numpy
arrays, one per node, in input order) and the same .npy side effect
(explain.py:216-220).  The per-node optimisation is NOT executed in Python: the whole batch of
nodes goes through libgnnx (k-hop extraction kernel + one persistent CTA per node).

Differences that are deliberate and documented:
  * explain_nodes() batches all nodes into one launch; it returns the list of masks like the
    reference (explain.py:234-236,290-292) but does not run the reference's matplotlib/tensorboard
    post-processing (denoise_graph/align/log_graph, explain.py:238-288: viz, out of scope).
  * M0 policy (args.gnnx_init, default "torch"): "torch" draws FloatTensor(n,n).normal_(1, std)
    from torch's global CPU generator per node in call order, exactly the RNG consumption of
    ExplainModule.construct_edge_mask (explain.py:645-652) -> bit-identical M0 under the same
    torch.manual_seed; "device" draws N(1, 2/n) with Philox on the GPU (no n^2 host work).
  * args.gnnx_latency (default False): True lets small batches (one explain() call, a shard of a multi-GPU run) split their most
    expensive tasks over thread-block clusters (one syn1 hub node 2.85 -> 1.56 ms); masks then agree with the default mode to
    round-off instead of bit for bit (gx_debug_set_cluster in include/gnnx.h).
  * a node outside its own k-hop set (isolated) raises instead of explaining a wrong row.
"""
import math
import os

import numpy as np
import torch

from . import _abi
from .engine import Engine
from . import graph_utils as _gu


def gen_prefix(args):
    """utils/io_utils.py:37-51 (file-name compatibility of the .npy side effect)."""
    name = args.bmname if getattr(args, "bmname", None) is not None else args.dataset
    name += "_" + args.method
    name += "_h" + str(args.hidden_dim) + "_o" + str(args.output_dim)
    if not args.bias:
        name += "_nobias"
    if len(args.name_suffix) > 0:
        name += "_" + args.name_suffix
    return name


def gen_explainer_prefix(args):
    """utils/io_utils.py:54-60."""
    name = gen_prefix(args) + "_explain"
    if len(args.explainer_suffix) > 0:
        name += "_" + args.explainer_suffix
    return name


def model_weights(model):
    """state_dict of a reference (or gnnx) GcnEncoderNode/GcnEncoderGraph -> weight dict.
    Keys as in the reference checkpoints (SURVEY 8a8): conv_first / conv_block.i / conv_last /
    pred_model."""
    sd = {k: v.detach().cpu().float().numpy() for k, v in model.state_dict().items()}
    if "pred_model.weight" not in sd:
        raise NotImplementedError("pred_hidden_dims != [] (MLP prediction head) is not built")
    n_block = 0
    while ("conv_block.%d.weight" % n_block) in sd:
        n_block += 1
    names = ["conv_first"] + ["conv_block.%d" % i for i in range(n_block)] + ["conv_last"]
    w = {}
    for l, nm in enumerate(names, 1):
        w["W%d" % l] = sd[nm + ".weight"]
        w["b%d" % l] = sd.get(nm + ".bias")
        if (nm + ".self_weight") in sd or (nm + ".att_weight") in sd:
            raise NotImplementedError("add_self / att GraphConv variants are out of scope")
    w["Wp"], w["bp"] = sd["pred_model.weight"], sd["pred_model.bias"]
    return w, len(names)


class Explainer:
    def __init__(self, model, adj, feat, label, pred, train_idx, args, writer=None,
                 print_training=True, graph_mode=False, graph_idx=False, device=None):
        self.model = model
        if hasattr(self.model, "eval"):
            self.model.eval()
        self.adj = adj
        self.feat = feat
        self.label = label
        self.pred = pred
        self.train_idx = train_idx
        self.n_hops = args.num_gc_layers
        self.graph_mode = graph_mode
        self.graph_idx = graph_idx
        self.args = args
        self.writer = writer
        self.print_training = print_training
        self._neighborhoods = None
        if getattr(args, "mask_act", "sigmoid") != "sigmoid":
            raise NotImplementedError("mask_act=%r is not built (default: sigmoid; the reference's ReLU variant returns NaN masks, "
                                      "tests/test_oracle.py)" % args.mask_act)
        # args.mask_bias: accepted.  The reference's bias matrix starts at 0 where ReLU6 has zero gradient, Adam never moves it and the
        # masks equal the default run bit for bit (explain.py:657-660,673-676; pinned by tests/test_oracle.py) -- no extra state needed.
        # utils/train_utils.py:7-23: adam / sgd / rmsprop / adagrad, schedulers none / step / cos
        if getattr(args, "opt", "adam") not in _abi.GX_OPT or getattr(args, "opt_scheduler", "none") not in _abi.GX_SCHED:
            raise ValueError("unknown optimiser / scheduler: %r / %r" % (getattr(args, "opt", None), getattr(args, "opt_scheduler", None)))
        # graph mode takes every model variant (layers, --bn, widths) and optimiser too: the graphs that explain_graph.cu does not
        # build run in explain_graph_var.cu
        bn = bool(getattr(model, "bn", False))
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if torch.cuda.is_available() else 0
        self.engine = Engine(device)
        weights, num_layers = model_weights(model)
        self.engine.set_model(weights, num_layers=num_layers, bn=bn)
        if getattr(args, "gnnx_latency", False):
            self.engine.debug_cluster(0, 0)   # latency mode: thread-block clusters for the expensive tasks of batches that leave SMs idle
        # model / optimiser variants run in the variant kernel, which does not log the per-epoch trace print_training replays
        self._no_trace = bn or num_layers != 3 or getattr(args, "opt", "adam") != "adam"
        adj_np = np.asarray(adj)
        if graph_mode:
            # graph classification: the whole padded batch goes to the device once (explain.py:80-85)
            if adj_np.ndim != 3:
                raise ValueError("graph mode expects adj of shape (G,n,n)")
            self.engine.set_graph_batch(adj_np, np.asarray(feat), np.asarray(label))
            return
        if adj_np.ndim != 3:
            raise ValueError("node mode expects adj of shape (B,N,N)")
        # node tasks on a batch of graphs (explain.py:80-95 index adj / feat / label / pred with graph_idx): the engine holds one graph
        # at a time, graph 0 is uploaded now, another one when a call names it
        self._csr_cache = {}
        self._own_pred = {}
        self._current_graph = None
        self._select_graph(0)

    def _select_graph(self, graph_idx):
        g = 0 if graph_idx in (-1, None, False) else int(graph_idx)
        if g == self._current_graph:
            return g
        adj_np = np.asarray(self.adj)
        if not 0 <= g < adj_np.shape[0]:
            raise IndexError("graph_idx %d out of range for adj of shape %s" % (g, adj_np.shape))
        if g not in self._csr_cache:
            self._csr_cache[g] = _gu.csr_from_dense(adj_np[g])
        self._rowptr, self._col = self._csr_cache[g]
        feat_np = np.asarray(self.feat, dtype=np.float32)[g]
        label_np = np.asarray(self.label)[g].astype(np.int32)
        if self.pred is None or g in self._own_pred:
            # no stored predictions (the reference reads cg["pred"] from the checkpoint, explainer_main.py:186-193): run the model's
            # forward on the device (gx_model_forward = GcnEncoderNode.forward on the whole graph) and keep the logits
            if g not in self._own_pred:
                self.engine.set_graph_csr(self._rowptr, self._col, feat_np, label_np, np.zeros(len(label_np), np.int32))
                self._own_pred[g] = self.engine.model_forward()
            pred_g = self._own_pred[g]
        else:
            pred_g = np.asarray(self.pred)[g]
        self._pred_label = np.argmax(pred_g, axis=1).astype(np.int32)          # explain.py:105
        self.engine.set_graph_csr(self._rowptr, self._col, feat_np, label_np, self._pred_label)
        self._current_graph = g
        return g

    # the reference computes this dense (B,N,N) matrix eagerly in __init__ (explain.py:67); here
    # it is materialised on demand only (the engine never needs it).
    @property
    def neighborhoods(self):
        if self._neighborhoods is None:
            keep = self._current_graph
            mats = []
            for g in range(np.asarray(self.adj).shape[0]):
                self._select_graph(g)
                N = self.engine.num_nodes
                mats.append(self.engine.neighborhood_rows(np.arange(N, dtype=np.int32), self.n_hops).astype(int))
            self._select_graph(keep)
            self._neighborhoods = np.stack(mats)
        return self._neighborhoods

    def extract_neighborhood(self, node_idx, graph_idx=0):
        """explain.py:492-501: (node_idx_new, sub_adj, sub_feat, sub_label, neighbors)."""
        graph_idx = self._select_graph(graph_idx)
        plan = self.engine.plan_nodes([int(node_idx)], self.n_hops)
        nbrs = plan.neighbors_of(0).astype(np.int64)
        # the caller's own adjacency rows / columns, exactly like the reference (adj[g][nbrs][:, nbrs]): self loops, if any, stay in
        # sub_adj (the plan's edge list drops them, as the explainer's diag_mask does for the optimisation)
        sub_adj = np.asarray(self.adj)[graph_idx][nbrs][:, nbrs]
        sub_feat = np.asarray(self.feat)[graph_idx, nbrs]
        sub_label = np.asarray(self.label)[graph_idx][nbrs]
        return int(plan.node_idx_new[0]), sub_adj, sub_feat, sub_label, nbrs

    # ---------------------------------------------------------------- internals
    def _hparams(self):
        a = self.args
        init = getattr(a, "gnnx_init", "torch")
        if init not in ("torch", "device"):
            raise ValueError("args.gnnx_init must be 'torch' or 'device'")
        hp = self.engine.make_hparams(
            num_epochs=a.num_epochs, lr=a.lr,
            init=_abi.GX_INIT_M0 if init == "torch" else _abi.GX_INIT_PHILOX,
            seed=int(getattr(a, "gnnx_seed", 0)))
        hp.opt = _abi.GX_OPT[getattr(a, "opt", "adam")]
        hp.opt_scheduler = _abi.GX_SCHED[getattr(a, "opt_scheduler", "none")]
        if hp.opt_scheduler == _abi.GX_SCHED["step"]:
            hp.opt_decay_step = int(a.opt_decay_step); hp.opt_decay_rate = float(a.opt_decay_rate)
        elif hp.opt_scheduler == _abi.GX_SCHED["cos"]:
            hp.opt_restart = int(a.opt_restart)
        return hp, init

    def _draw_m0(self, plan, keep_dense=False):
        """Per node, in call order: FloatTensor(n,n).normal_(1, std) (explain.py:645-652), gathered at the
        directed-edge slots.  Consumes torch's global CPU RNG exactly like the reference (the n^2 draw per node IS the
        cost of this policy: ~3 ns per normal on one core; args.gnnx_init="device" has no host work).
        keep_dense: also return the dense draws (the off-edge entries only matter for the printed loss)."""
        m0 = np.empty(plan.total_edges, dtype=np.float32)
        gain = torch.nn.init.calculate_gain("relu")
        flat = plan.flat_index()            # row * n + col of every edge slot, whole batch at once
        dense = [] if keep_dense else None
        for t in range(plan.count):
            n = plan.n(t)
            std = gain * math.sqrt(2.0 / (n + n))
            M = torch.FloatTensor(n, n).normal_(1.0, std).numpy()
            np.take(M.reshape(-1), flat[plan.edge_off[t]:plan.edge_off[t + 1]], out=m0[plan.edge_off[t]:plan.edge_off[t + 1]])
            if keep_dense:
                dense.append(M)
        return (m0, dense) if keep_dense else m0

    def _draw_m0_subset(self, plan, n_all, positions):
        """Sharded runs with the torch-compatible init: walk the WHOLE node list in order (n_all[p] = sub-graph size of list entry
        p, from gx_count_nodes) drawing every node's n^2 normals like one process would, and keep the edge entries of the entries
        this rank owns (`positions`, ascending; `plan` is the plan of exactly those nodes)."""
        m0 = np.empty(plan.total_edges, dtype=np.float32)
        gain = torch.nn.init.calculate_gain("relu")
        flat = plan.flat_index()
        mine = {int(p): t for t, p in enumerate(positions)}
        for p, n in enumerate(n_all):
            n = int(n)
            M = torch.FloatTensor(n, n).normal_(1.0, gain * math.sqrt(2.0 / (n + n)))
            t = mine.get(p)
            if t is not None:
                np.take(M.numpy().reshape(-1), flat[plan.edge_off[t]:plan.edge_off[t + 1]], out=m0[plan.edge_off[t]:plan.edge_off[t + 1]])
        return m0

    def _explain_batch(self, node_indices, graph_idx=0, model="exp", unconstrained=False):
        if model not in ("exp", "grad"):
            raise NotImplementedError("model=%r (att) is not built" % model)
        if unconstrained:
            raise NotImplementedError("unconstrained=True is not built")
        self._select_graph(graph_idx)
        nodes = [int(i) for i in node_indices]
        plan = self.engine.plan_nodes(nodes, self.n_hops)
        edge_mask = np.empty(plan.total_edges, dtype=np.float32)
        if model == "grad":        # explain.py:125-133: one backward to the adjacency, no mask parameters (the reference still
            if self._hparams()[1] == "torch":      # constructs an ExplainModule per node, i.e. consumes n^2 normals: keep the RNG in step)
                self._draw_m0(plan)
            self.engine.grad_nodes_host(edge_mask)
            return plan, edge_mask
        hp, init = self._hparams()
        if not self.print_training or self._no_trace:
            if self.print_training:
                print("(per-epoch trace is not built for --bn / num_gc_layers != 3 / optimisers other than Adam)")
            m0 = self._draw_m0(plan) if init == "torch" else None
            self.engine.explain_nodes_host(hp, m0, edge_mask)
            return plan, edge_mask
        # print_training (explain.py:148-159): the kernels log every epoch's loss terms / density / softmax row (gx_explain_io.trace)
        m0, dense = self._draw_m0(plan, keep_dense=True) if init == "torch" else (None, None)
        trace = np.zeros((plan.count, hp.num_epochs, _abi.GX_TRACE_COLS), np.float32)
        pred = np.zeros((plan.count, hp.num_epochs, self.engine.num_classes), np.float32)
        self.engine.explain_nodes_ex(hp, m0, edge_mask, trace=trace, trace_pred=pred)
        off = self.engine.offedge_regularisers(hp, np.concatenate([D.reshape(-1) for D in dense])) if dense is not None else None
        self.last_trace = self._print_trace(plan, hp, trace, pred, off)
        return plan, edge_mask

    def _print_trace(self, plan, hp, trace, pred, off):
        """Replays the reference's per-epoch print (explain.py:148-159).  With the torch-compatible init the loss is the
        reference's own number (edge part from the kernels + the regulariser sums over the n^2 - E_d mask entries that never reach
        the result, gx_offedge_regularisers); with the device init those entries are never materialised and the printed loss
        covers the edge entries only."""
        loss = trace[:, :, _abi.TR_LOSS_EDGES].astype(np.float64)
        if off is not None:
            nn = np.diff(plan.node_off).astype(np.float64)[:, None] ** 2
            loss = loss + hp.coef_size * off[:, :, 0] + hp.coef_ent * off[:, :, 1] / nn
        for t in range(plan.count):
            for epoch in range(hp.num_epochs):
                print("epoch: ", epoch, "; loss: ", float(loss[t, epoch]), "; mask density: ", float(trace[t, epoch, _abi.TR_DENSITY]),
                      "; pred: ", torch.from_numpy(pred[t, epoch]))
            print("finished training in ", 0.0)
        return dict(loss=loss, density=trace[:, :, _abi.TR_DENSITY].copy(), pred=pred, terms=trace)

    def _save(self, masked_adj, node_idx):
        fname = "masked_adj_" + gen_explainer_prefix(self.args) + (
            "node_idx_" + str(node_idx) + "graph_idx_" + str(self.graph_idx) + ".npy")
        os.makedirs(self.args.logdir, exist_ok=True)
        with open(os.path.join(self.args.logdir, fname), "wb") as outfile:
            np.save(outfile, np.asarray(masked_adj.copy()))
        return fname

    # ---------------------------------------------------------------- public API
    def _explain_graph_batch(self, graph_indices):
        gids = [int(g) for g in graph_indices]
        edge_off = self.engine.plan_graphs(gids)
        hp, init = self._hparams()
        n = self.engine.batch_n
        m0 = None
        rc = [self.engine.graph_rows_cols(g) for g in gids]
        if init == "torch":
            m0 = np.empty(int(edge_off[-1]), dtype=np.float32)
            std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (n + n))
            for t, (rows, cols) in enumerate(rc):
                M = torch.FloatTensor(n, n).normal_(1.0, std).numpy()      # explain.py:645-652, n = padded size
                m0[edge_off[t]:edge_off[t + 1]] = M[rows, cols]
        edge_mask = np.empty(int(edge_off[-1]), dtype=np.float32)
        self.engine.explain_graphs_host(hp, m0, edge_mask)
        out = []
        for t, (rows, cols) in enumerate(rc):
            D = np.zeros((n, n), dtype=np.float64)
            D[rows, cols] = edge_mask[edge_off[t]:edge_off[t + 1]]
            out.append(D)
        return out

    def explain_graphs(self, graph_indices, save=True):
        """explain.py:356-402 -> list of (n,n) masked adjacencies (one batched launch; the reference's
        denoise_graph/log_graph drawing is out of scope)."""
        if not self.graph_mode:
            raise ValueError("Explainer was not constructed with graph_mode=True")
        out = self._explain_graph_batch(graph_indices)
        if save:
            for m in out:
                self._save(m, 0)      # the reference overwrites one file: node_idx_0 graph_idx_<self.graph_idx>
        return out

    def explain(self, node_idx, graph_idx=0, graph_mode=False, unconstrained=False, model="exp"):
        """explain.py:74-221 -> (n,n) float64 masked adjacency of the node's k-hop subgraph (node mode)
        or of the whole padded graph `graph_idx` (graph_mode=True)."""
        if graph_mode or self.graph_mode:
            if not self.graph_mode:
                raise ValueError("Explainer was not constructed with graph_mode=True")
            if model != "exp" or unconstrained:
                raise NotImplementedError("only model='exp', unconstrained=False are built")
            masked_adj = self._explain_graph_batch([graph_idx])[0]
            fname = self._save(masked_adj, node_idx)
            if self.print_training:
                print("Saved adjacency matrix to ", fname)
            return masked_adj
        plan, edge_mask = self._explain_batch([node_idx], graph_idx, model, unconstrained)
        masked_adj = plan.dense_of(0, edge_mask, dtype=np.float64)
        fname = self._save(masked_adj, node_idx)
        if self.print_training:
            print("Saved adjacency matrix to ", fname)
        return masked_adj

    def explain_nodes(self, node_indices, args=None, graph_idx=0, save=True, copy=True):
        """explain.py:225-292 -> list of (n,n) float64 masked adjacencies in input order.  One batched launch; the dense arrays are
        built ON DEVICE (gx_densify) and come back in one transfer -- the list entries are views of that one buffer:
          copy=True  (default) independent results like the reference's: views of a pinned buffer that is not reused while any of them is alive;
          copy=False ONE pinned buffer owned by the Explainer, overwritten by the next call.
        save=True writes the reference's per-node .npy files (explain.py:216-220), which at ~0.4 MB per node dominates the call;
        args.gnnx_init="device" removes the n^2 host normals per node of the torch-compatible init."""
        self._select_graph(graph_idx)
        if self.print_training:
            plan, edge_mask = self._explain_batch(node_indices, graph_idx)
            out = [plan.dense_of(t, edge_mask, dtype=np.float64) for t in range(plan.count)]
        else:
            nodes = [int(i) for i in node_indices]
            eng = self.engine
            plan = eng.plan_nodes(nodes, self.n_hops)
            hp, init = self._hparams()
            dev = torch.device("cuda", eng.device)
            m0_dev = None
            if init == "torch":
                m0_dev = torch.from_numpy(self._draw_m0(plan)).to(dev, non_blocking=False)
            mask_dev = eng.explain_nodes_device(hp, m0_dev)
            dense_dev = eng.densify_device(mask_dev)
            if copy:
                host = self._result_buffer(dense_dev.numel())       # pinned, never handed out twice while a result still refers to it
                torch.from_numpy(host)[:dense_dev.numel()].copy_(dense_dev)
            else:
                if getattr(self, "_pinned", None) is None or self._pinned.numel() < dense_dev.numel():
                    self._pinned = torch.empty(max(dense_dev.numel(), 1), dtype=torch.float64).pin_memory()
                self._pinned[:dense_dev.numel()].copy_(dense_dev)
                host = self._pinned.numpy()
            n_t = np.diff(plan.node_off).astype(np.int64)
            offs = np.concatenate([[0], np.cumsum(n_t * n_t)])
            out = [host[offs[t]:offs[t + 1]].reshape(n_t[t], n_t[t]) for t in range(plan.count)]
        if save:
            for t, node in enumerate(node_indices):
                self._save(out[t], int(node))
        return out

    def _result_buffer(self, numel):
        """Host memory for one call's dense results: a pinned buffer from a small pool.  The returned arrays are views of it
        (numpy keeps the buffer alive through .base), and a buffer is reused only when no earlier result refers to it any more
        (sys.getrefcount), so results stay independent like the reference's -- without a 0.3 GB pageable allocation + copy per call."""
        import sys
        pool = self.__dict__.setdefault("_pool", [])
        for i, (t, a) in enumerate(pool):
            if t.numel() >= numel and sys.getrefcount(a) <= 3:      # pool tuple + loop variable + getrefcount's argument
                return a
        pool[:] = [(t, a) for (t, a) in pool if sys.getrefcount(a) > 3][-2:]     # drop idle buffers that are too small
        t = torch.empty(max(int(numel), 1), dtype=torch.float64).pin_memory()
        a = t.numpy()
        pool.append((t, a))
        return a

    # ---------------------------------------------------------------- evaluation step right after the masks
    # planted-motif edges relative to the first motif node, in the sorted local numbering (explain.py:537-577)
    _MOTIF_EDGES = {
        "syn1": [(0, 1), (1, 2), (2, 3), (0, 3), (0, 4), (1, 4)],          # house
        "syn2": [(0, 1), (1, 2), (2, 3), (0, 3), (0, 4), (1, 4)],
        "syn4": [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5), (0, 5)],          # 6-cycle
    }

    def make_pred_real(self, adj, start):
        """explain.py:535-579: (pred, real) over the upper-triangular positive entries of a masked adjacency;
        real = 1 on the planted motif's edges (fixed offsets from `start`)."""
        if self.args.dataset not in self._MOTIF_EDGES:
            raise NotImplementedError("make_pred_real knows syn1/syn2/syn4 only (like the reference)")
        adj = np.asarray(adj)
        upper = np.triu(adj) > 0
        pred = adj[upper]
        truth = np.zeros(adj.shape, dtype=bool)
        for (p_, q_) in self._MOTIF_EDGES[self.args.dataset]:
            if adj[start + p_][start + q_] > 0:        # IndexError past the subgraph, like the reference
                truth[start + p_, start + q_] = True
        real = truth[upper].astype(adj.dtype)
        return pred, real

    def explain_nodes_gnn_stats(self, node_indices, args=None, graph_idx=0, model="exp"):
        """explain.py:295-353: explain the nodes (one batched launch), score the edge masks against the planted
        motifs with ROC-AUC and write log/pr/auc_<dataset>_<model>.txt; returns the masks.  The PR-curve PNG
        and the tensorboard drawings of the reference are not produced (viz, out of scope)."""
        from sklearn.metrics import roc_auc_score
        plan, edge_mask = self._explain_batch(node_indices, graph_idx, model)
        masked_adjs = [plan.dense_of(t, edge_mask, dtype=np.float64) for t in range(plan.count)]
        pred_all, real_all = [], []
        for t in range(plan.count):
            pred, real = self.make_pred_real(masked_adjs[t], int(plan.node_idx_new[t]))
            pred_all.append(pred); real_all.append(real)
        real_cat, pred_cat = np.concatenate(real_all), np.concatenate(pred_all)
        self.auc = float(roc_auc_score(real_cat, pred_cat))
        os.makedirs(os.path.join("log", "pr"), exist_ok=True)
        # explain.py:308,329-335: the denoised graphs (threshold_num=20) and the precision/recall curve.  The reference draws both
        # (tensorboard / matplotlib); here the graphs are kept on the object and the curve is written as arrays (+ PNG if matplotlib exists)
        self.denoised, _ = self.denoise_nodes(plan, edge_mask, threshold_num=20, with_feat=True)
        from sklearn.metrics import precision_recall_curve
        precision, recall, thresholds = precision_recall_curve(real_cat, pred_cat)
        self.pr_curve = (precision, recall, thresholds)
        np.savez(os.path.join("log", "pr", "pr_" + self.args.dataset + "_" + model + ".npz"), precision=precision, recall=recall, thresholds=thresholds)
        try:
            import matplotlib
            matplotlib.use("agg")
            import matplotlib.pyplot as plt
            plt.plot(recall, precision)
            plt.savefig(os.path.join("log", "pr", "pr_" + self.args.dataset + "_" + model + ".png"))
            plt.close()
        except ImportError:
            pass
        with open(os.path.join("log", "pr", "auc_" + self.args.dataset + "_" + model + ".txt"), "w") as f:
            f.write("dataset: {}, model: {}, auc: {}\n".format(self.args.dataset, "exp", str(self.auc)))
        return masked_adjs

    def denoise_nodes(self, plan, edge_mask, threshold_num=20, max_component=True, with_feat=False):
        """io_utils.denoise_graph(masked_adj, node_idx_new, feat, threshold_num=20) (explain.py:308, utils/io_utils.py:193-245) for
        every node of a packed result: the 2*threshold_num-largest threshold and the surviving edges are computed on device
        (gx_denoise_topk); only those <= ~40 edges per node come back, the networkx object is assembled from them."""
        from . import io_utils
        thr, cnt, slots, vals = self.engine.denoise_topk(edge_mask, threshold_num)
        cap = slots.shape[1]
        if int(cnt.max(initial=0)) > cap:          # many values tie at the threshold: fetch again with room for all of them
            thr, cnt, slots, vals = self.engine.denoise_topk(edge_mask, threshold_num, cap=int(cnt.max()))
        flat = plan.flat_index()
        out = []
        for t in range(plan.count):
            n = plan.n(t)
            k = int(cnt[t])
            f = flat[plan.edge_off[t] + slots[t, :k]]
            feat = np.asarray(self.feat)[0, plan.neighbors_of(t)] if with_feat else None
            out.append(io_utils.graph_from_edges(n, int(plan.node_idx_new[t]), f // n, f % n, vals[t, :k], feat, None, max_component))
        return out, thr

    def explain_nodes_packed(self, node_indices, graph_idx=0):
        """Same computation, returning (plan, edge_mask) without densifying: edge_mask[edge_off[t]:
        edge_off[t+1]] are the masked_adj entries of node t at plan.csr_of(t) (row-major order)."""
        return self._explain_batch(node_indices, graph_idx)

    def iter_explain_nodes_packed(self, node_indices, chunk_size, graph_idx=0, model="exp"):
        """Large graphs (BASELINE configs[4]: a k-hop neighbourhood is most of a 10^5-node graph, ~0.4 GB of plan and optimiser
        state per explained node): explain the list `chunk_size` nodes at a time and yield (nodes_of_chunk, plan, edge_mask)
        per chunk, so that neither the device workspace nor the host ever holds more than one chunk (one CTA per SM => 148 is a
        natural chunk on a B200).  The dense (n,n) arrays of explain_nodes would need 80 GB per node there."""
        nodes = [int(i) for i in node_indices]
        if chunk_size < 1:
            raise ValueError("chunk_size must be >= 1")
        for s0 in range(0, len(nodes), int(chunk_size)):
            part = nodes[s0:s0 + int(chunk_size)]
            plan, edge_mask = self._explain_batch(part, graph_idx, model)
            yield part, plan, edge_mask
