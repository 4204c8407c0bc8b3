"""GPU (-m gpu): graph-classification mode through the graph-variant kernel (explain_graph_var.cu) -- model variants (2 / 4 layers,
--bn, widths up to 128), optimisers other than Adam and graphs beyond the shared-memory layout -- against the masks the UNMODIFIED
reference returned (tests/golden/graph_variants_golden.npz), the line-by-line torch port, and the drop-in Explainer."""
import types

import numpy as np
import pytest
import torch

import gnnx
from gnnx import _abi
import gnnx_oracle as O
import util
from test_oracle_graph_variants import MODEL_CASES, OPT_CASES, case_weights, dense_m0, load

pytestmark = pytest.mark.gpu


def engine_hparams(eng, tag, epochs):
    hp = eng.make_hparams(num_epochs=epochs)
    over = dict(OPT_CASES).get(tag, {})
    hp.opt = _abi.GX_OPT[over.get("opt", "adam")]
    hp.opt_scheduler = _abi.GX_SCHED[over.get("opt_scheduler", "none")]
    if "opt_decay_step" in over:
        hp.opt_decay_step = over["opt_decay_step"]; hp.opt_decay_rate = over["opt_decay_rate"]
    if "opt_restart" in over:
        hp.opt_restart = over["opt_restart"]
    return hp


def run(eng, gids, m0_of, hp):
    edge_off = eng.plan_graphs(gids)
    m0 = np.concatenate([m0_of(g) for g in gids]).astype(np.float32)
    out = np.zeros(int(edge_off[-1]), np.float32)
    eng.explain_graphs_host(hp, m0, out)
    return edge_off, out


@pytest.mark.parametrize("tag", [c[0] for c in MODEL_CASES] + [c[0] for c in OPT_CASES])
def test_golden_case_matches_reference(tag):
    gv, gg = load()
    w, L, bn = case_weights(gv, gg, tag)
    E = int(gv["num_epochs"])
    eng = gnnx.Engine(0)
    eng.set_model(w, num_layers=L, bn=bn)
    eng.set_graph_batch(gg["adj"], gg["feat"], gg["label"])
    gids = list(range(int(gv["num_graphs"])))
    m0_of = lambda g: gv["g%d_m0" % g]
    edge_off, out = run(eng, gids, m0_of, engine_hparams(eng, tag, E))
    errs = {g: util.rel_l2(out[edge_off[t]:edge_off[t + 1]], gv["%s_g%d_mask" % (tag, g)]) for t, g in enumerate(gids)}
    assert max(errs.values()) <= 1e-4, errs
    # deterministic, and independent of the batch's composition and order
    _, again = run(eng, gids, m0_of, engine_hparams(eng, tag, E))
    assert np.array_equal(again, out)
    sub = [7, 2, 11]
    eo, o2 = run(eng, sub, m0_of, engine_hparams(eng, tag, E))
    for t, g in enumerate(sub):
        assert np.array_equal(o2[eo[t]:eo[t + 1]], out[edge_off[g]:edge_off[g + 1]]), g
    # num_epochs = 1 returns the sigmoid-symmetrised initial mask
    _, one = run(eng, gids, m0_of, engine_hparams(eng, tag, 1))
    for t, g in enumerate(gids):
        M0 = dense_m0(gv, gg, g).astype(np.float64)
        S = 1 / (1 + np.exp(-M0))
        ei, ej = np.nonzero(gg["adj"][g])
        assert np.abs(one[edge_off[t]:edge_off[t + 1]] - ((S + S.T) / 2)[ei, ej]).max() < 1e-6
    eng.close()


def molecule_batch(rng, G, max_nodes, sizes, d):
    """Padded molecule-like graphs: random trees plus a few extra bonds, one isolated atom in graph 0; features N(0,1)."""
    import networkx as nx
    adj = np.zeros((G, max_nodes, max_nodes), np.uint8)
    for g, n in enumerate(sizes):
        T = nx.random_labeled_tree(n, seed=int(rng.integers(1 << 30))) if hasattr(nx, "random_labeled_tree") else nx.random_tree(n, seed=int(rng.integers(1 << 30)))
        for _ in range(max(1, n // 6)):
            u, v = rng.integers(0, n, 2)
            if u != v:
                T.add_edge(int(u), int(v))
        if g == 0:
            T.remove_edges_from(list(T.edges(0)))
        adj[g, :n, :n] = nx.to_numpy_array(T, nodelist=range(n)).astype(np.uint8)
    feat = rng.normal(size=(G, max_nodes, d)).astype(np.float32)
    return adj, feat


def random_model(rng, L, hid, emb, d, C):
    sc = lambda *s: (rng.normal(size=s) * 0.5).astype(np.float32)
    dims = [d] + [hid] * (L - 1) + [emb]
    w = {}
    for l in range(1, L + 1):
        w["W%d" % l] = sc(dims[l - 1], dims[l])
        w["b%d" % l] = np.abs(sc(dims[l])) + 0.2      # positive biases: the edge-less constant wins some max-pools
    w["Wp"] = sc(C, hid * (L - 1) + emb); w["bp"] = sc(C)
    return w


@pytest.mark.parametrize("seed,L,bn,hid,emb,d,C", [(1, 2, True, 33, 40, 14, 2), (2, 4, True, 64, 64, 7, 3), (3, 3, False, 128, 96, 128, 6),
                                                  (4, 4, False, 48, 128, 33, 4), (5, 3, True, 20, 12, 14, 5), (6, 2, False, 128, 128, 100, 2)])
def test_random_models_match_torch_port(seed, L, bn, hid, emb, d, C):
    rng = np.random.default_rng(seed)
    G, n = 4, 40
    adj, feat = molecule_batch(rng, G, n, [int(x) for x in rng.integers(8, 36, G)], d)
    label = rng.integers(0, C, G).astype(np.int32)
    w = random_model(rng, L, hid, emb, d, C)
    eng = gnnx.Engine(0)
    eng.set_model(w, num_layers=L, bn=bn)
    eng.set_graph_batch(adj, feat, label)
    gids = list(range(G))
    dense = {g: O.draw_m0(n, seed=100 * seed + g) for g in gids}
    E = 20

    def m0_of(g):
        r, c = eng.graph_rows_cols(g)
        return dense[g][r, c]
    edge_off, out = run(eng, gids, m0_of, eng.make_hparams(num_epochs=E))
    for t, g in enumerate(gids):
        A = adj[g].astype(float)
        hp = O.default_hparams(num_epochs=E)
        ref = O.explain_dense_torch(A, feat[g], label[g], None, 0, w, dense[g], hp=hp, graph_mode=True, bn=bn)
        c64 = O.explain_closed_form(A, feat[g], label[g], None, 0, w, dense[g], hp=hp, graph_mode=True, bn=bn)
        tol = max(1e-4, 3 * O.rel_l2(c64, ref))
        r, c = eng.graph_rows_cols(g)
        assert util.rel_l2(out[edge_off[t]:edge_off[t + 1]], ref[r, c]) <= tol, (g, tol)
    eng.close()


@pytest.mark.parametrize("L,bn", [(3, False), (4, True)], ids=["default", "L4bn"])
def test_large_graphs(L, bn):
    """Graphs of several hundred to ~1000 nodes (beyond the shared-memory kernel) mixed with molecules in a batch padded to 1024."""
    rng = np.random.default_rng(11 + L)
    n, d, C = 1024, 14, 2
    sizes = [30, 900, 25, 400, 1000, 38]
    adj, feat = molecule_batch(rng, len(sizes), n, sizes, d)
    label = rng.integers(0, C, len(sizes)).astype(np.int32)
    w = random_model(rng, L, 20, 20, d, C)
    eng = gnnx.Engine(0)
    eng.set_model(w, num_layers=L, bn=bn)
    eng.set_graph_batch(adj, feat, label)
    dense = {g: O.draw_m0(n, seed=300 + g) for g in range(len(sizes))}

    def m0_of(g):
        r, c = eng.graph_rows_cols(g)
        return dense[g][r, c]
    E = 4
    full = list(range(len(sizes)))
    eo, out = run(eng, full, m0_of, eng.make_hparams(num_epochs=E))
    res = {g: out[eo[t]:eo[t + 1]] for t, g in enumerate(full)}
    for g in (1, 4, 0):
        hp = O.default_hparams(num_epochs=E)
        ref = O.explain_dense_torch(adj[g].astype(float), feat[g], label[g], None, 0, w, dense[g], hp=hp, graph_mode=True, bn=bn)
        r, c = eng.graph_rows_cols(g)
        assert util.rel_l2(res[g], ref[r, c]) <= 1e-4, g
    small = [0, 2, 5]
    eo2, out2 = run(eng, small, m0_of, eng.make_hparams(num_epochs=E))
    for t, g in enumerate(small):
        assert np.array_equal(out2[eo2[t]:eo2[t + 1]], res[g]), g
    eo3, out3 = run(eng, [4, 2, 1], m0_of, eng.make_hparams(num_epochs=E))
    assert np.array_equal(out3[eo3[0]:eo3[1]], res[4]) and np.array_equal(out3[eo3[2]:eo3[3]], res[1])
    eng.close()


def _args(tmp_path, **over):
    d = dict(num_gc_layers=3, num_epochs=30, lr=0.1, opt="adam", opt_scheduler="none", mask_act="sigmoid", mask_bias=False, gpu=False,
             bias=True, method="base", dataset="graphs", bmname=None, hidden_dim=20, output_dim=20, name_suffix="", explainer_suffix="",
             logdir=str(tmp_path))
    d.update(over)
    return types.SimpleNamespace(**d)


def _load_model(model, w, L):
    keys = ["conv_first"] + ["conv_block.%d" % i for i in range(L - 2)] + ["conv_last"]
    sd = {}
    for l, k in enumerate(keys, 1):
        sd[k + ".weight"] = torch.tensor(w["W%d" % l]); sd[k + ".bias"] = torch.tensor(w["b%d" % l])
    sd["pred_model.weight"] = torch.tensor(w["Wp"]); sd["pred_model.bias"] = torch.tensor(w["bp"])
    model.load_state_dict(sd)


@pytest.mark.parametrize("tag", ["bn", "L4bn", "sgd"])
def test_explainer_dropin_graph_variants(tag, tmp_path):
    """GcnEncoderGraph built with its own defaults (bn=True), 3 or 4 layers, and the default model with --opt sgd, through
    Explainer(graph_mode=True), under torch.manual_seed like the reference."""
    gv, gg = load()
    w, L, bn = case_weights(gv, gg, tag)
    over = dict(OPT_CASES).get(tag, {})
    args = _args(tmp_path, num_gc_layers=L, num_epochs=int(gv["num_epochs"]), **over)
    if bn:
        model = gnnx.models.GcnEncoderGraph(14, 20, 20, 2, L, args=args)      # bn defaults to True, as in the reference
        assert model.bn
    else:
        model = gnnx.models.GcnEncoderGraph(14, 20, 20, 2, L, bn=False, args=args)
    _load_model(model, w, L)
    ex = gnnx.Explainer(model=model, adj=torch.tensor(gg["adj"], dtype=torch.float), feat=torch.tensor(gg["feat"]),
                        label=torch.tensor(gg["label"]), pred=gg["pred"], train_idx=[], args=args, writer=None,
                        print_training=False, graph_mode=True, graph_idx=0)
    n = int(gg["max_nodes"])
    for g in (1, 3, 8):
        torch.manual_seed(int(gv["g%d_seed" % g]))
        masked = ex.explain(node_idx=0, graph_idx=g, graph_mode=True)
        assert masked.shape == (n, n) and masked.dtype == np.float64
        ei, ej = np.nonzero(gg["adj"][g])
        assert util.rel_l2(masked[ei, ej], gv["%s_g%d_mask" % (tag, g)]) <= 1e-4, g
        off = masked.copy(); off[ei, ej] = 0
        assert np.all(off == 0)
    torch.manual_seed(1)
    a = [ex.explain(0, graph_idx=g, graph_mode=True) for g in (4, 6)]
    torch.manual_seed(1)
    b = ex.explain_graphs([4, 6])
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    torch.manual_seed(2)
    c = ex.explain_graphs(range(12))
    assert len(c) == 12 and all(np.isfinite(x).all() for x in c)


def test_refuses_trace_and_state_on_variant_graphs():
    gv, gg = load()
    w, L, bn = case_weights(gv, gg, "L4bn")
    eng = gnnx.Engine(0)
    eng.set_model(w, num_layers=L, bn=bn)
    eng.set_graph_batch(gg["adj"], gg["feat"], gg["label"])
    edge_off = eng.plan_graphs([0, 1])
    te = int(edge_off[-1])
    m0 = np.concatenate([gv["g0_m0"], gv["g1_m0"]]).astype(np.float32)
    out = np.zeros(te, np.float32)
    with pytest.raises(_abi.GnnxError):
        eng.explain_nodes_ex(eng.make_hparams(num_epochs=3), m0, out, trace=np.zeros((2, 3, _abi.GX_TRACE_COLS), np.float32), graphs=True)
    st = dict(m=np.zeros(te, np.float32), v=np.zeros(te, np.float32), feat=np.zeros((2, 3, 14), np.float32))
    with pytest.raises(_abi.GnnxError):
        eng.explain_nodes_ex(eng.make_hparams(num_epochs=3, init=_abi.GX_INIT_STATE), m0, out, state_in=st, graphs=True)
    with pytest.raises(_abi.GnnxError):
        eng.explain_nodes_ex(eng.make_hparams(num_epochs=3), m0, out, state_out=dict(m=np.zeros(te, np.float32)), graphs=True)
    # the default model with an optimiser other than Adam runs in the same kernel: the same refusals
    eng.set_model({k: gg[k] for k in util.WKEYS})
    eng.plan_graphs([0, 1])
    hp = eng.make_hparams(num_epochs=3); hp.opt = _abi.GX_OPT["sgd"]
    with pytest.raises(_abi.GnnxError):
        eng.explain_nodes_ex(hp, m0, out, trace=np.zeros((2, 3, _abi.GX_TRACE_COLS), np.float32), graphs=True)
    eng.explain_graphs_host(hp, m0, out)          # without them it runs
    assert np.isfinite(out).all()
    eng.close()
