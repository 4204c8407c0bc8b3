"""CPU: host-side marshalling logic of the drop-in package (no GPU needed)."""
import types

import numpy as np
import pytest

import gnnx
from gnnx import explain as gx_explain
from gnnx import graph_utils as gx_gu
from gnnx.dist import shard_indices
from gnnx.engine import Plan
import gnnx_oracle as O
import os
import util


def test_csr_from_dense_matches_oracle():
    rng = np.random.default_rng(0)
    A = (rng.random((40, 40)) < 0.1).astype(float)
    A = np.maximum(A, A.T)
    np.fill_diagonal(A, 0)
    rp, col = gx_gu.csr_from_dense(A)
    rp2, col2 = O.csr_from_dense(A)
    assert np.array_equal(rp, rp2) and np.array_equal(col, col2)
    with pytest.raises(NotImplementedError):
        gx_gu.csr_from_dense(A * 0.5)


def test_plan_densify_roundtrip():
    # two tasks: a triangle and a path
    node_off = np.array([0, 3, 6]); edge_off = np.array([0, 6, 10])
    srp = np.array([0, 2, 4, 6, 0, 1, 3, 4], np.int32)
    scol = np.array([1, 2, 0, 2, 0, 1, 1, 0, 2, 1], np.int32)
    plan = Plan(np.array([5, 9]), node_off, edge_off, np.arange(6, dtype=np.int32), np.array([0, 1], np.int32), srp, scol)
    vals = np.arange(1, 11, dtype=np.float32)
    d0, d1 = plan.dense_of(0, vals), plan.dense_of(1, vals)
    assert d0.dtype == np.float64 and d0.shape == (3, 3) and d0[0, 1] == 1 and d0[2, 1] == 6 and d0[0, 0] == 0
    assert d1[0, 1] == 7 and d1[1, 0] == 8 and d1[1, 2] == 9 and d1[2, 1] == 10 and d1.sum() == 34


def test_explainer_prefix_matches_reference_naming():
    args = types.SimpleNamespace(bmname=None, dataset="syn1", method="base", hidden_dim=20, output_dim=20,
                                 bias=True, name_suffix="", explainer_suffix="")
    assert gx_explain.gen_explainer_prefix(args) == "syn1_base_h20_o20_explain"   # io_utils.py:37-60
    args.bias = False; args.name_suffix = "x"; args.explainer_suffix = "y"
    assert gx_explain.gen_explainer_prefix(args) == "syn1_base_h20_o20_nobias_x_explain_y"


def test_model_state_dict_keys_match_reference_checkpoints():
    args = types.SimpleNamespace(gpu=False, bias=True, method="base")
    m = gnnx.models.GcnEncoderNode(10, 20, 20, 4, 3, bn=False, args=args)
    keys = set(m.state_dict().keys())
    assert keys == {"conv_first.weight", "conv_first.bias", "conv_block.0.weight", "conv_block.0.bias",
                    "conv_last.weight", "conv_last.bias", "pred_model.weight", "pred_model.bias"}
    w, L = gx_explain.model_weights(m)
    assert L == 3 and w["W1"].shape == (10, 20) and w["Wp"].shape == (4, 60)
    # forward agrees with the oracle's statement of the architecture
    import torch
    x = torch.randn(1, 7, 10); adj = (torch.rand(1, 7, 7) < 0.4).float()
    adj = ((adj + adj.transpose(1, 2)) > 0).float()
    y, _ = m(x, adj)
    y2 = O._gcn_forward_torch(x, adj, O.weights_to_torch(w, False), False)
    assert torch.allclose(y, y2, atol=1e-6)


def test_shard_indices_partition():
    for world in (1, 2, 3, 8):
        costs = np.random.default_rng(1).integers(1, 100, 37)
        seen = np.concatenate([shard_indices(37, world, r, costs) for r in range(world)])
        assert sorted(seen) == list(range(37))
        loads = [costs[shard_indices(37, world, r, costs)].sum() for r in range(world)]
        assert max(loads) - min(loads) <= costs.max()


def test_make_pred_real_matches_reference():
    """explain.py:535-579 restated table-driven: identical (pred, real) and AUC to what the reference's own
    make_pred_real produced on its golden masks (oracle/gen_golden.py --only auc)."""
    import os
    from sklearn.metrics import roc_auc_score
    import util
    au = np.load(os.path.join(util.GOLDEN, "auc_golden.npz"))
    for which in ("syn1", "syn4"):
        fx = util.load_fixture(which)
        A = O.dense_from_csr(fx.rowptr, fx.col)
        ex = gx_explain.Explainer.__new__(gx_explain.Explainer)
        ex.args = types.SimpleNamespace(dataset=which)
        preds, reals = [], []
        for node in au[which + "_nodes"]:
            nbrs = fx.gold["n%d_nbrs" % node]
            sub = A[nbrs][:, nbrs]
            ei, ej = np.nonzero(sub)
            M = np.zeros_like(sub); M[ei, ej] = fx.gold["n%d_mask" % node]
            pred, real = ex.make_pred_real(M, int(fx.gold["n%d_idx_new" % node]))
            assert np.array_equal(real.astype(np.uint8), au["%s_n%d_real" % (which, node)])
            assert np.array_equal(pred.astype(np.float32), au["%s_n%d_pred" % (which, node)])
            preds.append(pred); reals.append(real)
        assert abs(roc_auc_score(np.concatenate(reals), np.concatenate(preds)) - float(au[which + "_auc"])) < 1e-12


def test_tu_reader_matches_reference(tmp_path):
    """gnnx.io_utils.read_tu_dataset against what the reference's read_graphfile + padding returned on the same toy dataset
    (tests/golden/tu_golden.npz, oracle/gen_golden.py --only tu)."""
    from gnnx.io_utils import read_tu_dataset
    rng = np.random.default_rng(4)
    sizes = util.write_tu_toy(str(tmp_path), "TOY", rng)
    out = read_tu_dataset(str(tmp_path), "TOY", max_nodes=10)
    assert out["adj"].shape[1:] == (10, 10) and len(out["label"]) == 4            # the 12-node graph is dropped
    assert np.array_equal(out["adj"], out["adj"].transpose(0, 2, 1)) and out["feat"].shape[2] == 5
    assert list(out["label"]) == [0, 1, 1, 0]                                      # first-appearance renumbering of {1,-1}
    ref = np.load(os.path.join(util.GOLDEN, "tu_golden.npz"))
    assert int(ref["count"]) == len(out["label"])
    for g in range(len(out["label"])):
        assert np.array_equal(ref["g%d_adj" % g], out["adj"][g]) and int(ref["g%d_label" % g]) == int(out["label"][g])
        feat = ref["g%d_feat" % g]
        assert len(feat) == [s for s in sizes if s <= 10][g]
        assert np.array_equal(feat, out["feat"][g, :len(feat)])


def test_bench_ba_generator_is_a_simple_symmetric_graph():
    """bench.py --workload c5 builds its Barabasi-Albert graph with a numpy generator: the CSR must be what
    gx_set_graph_csr accepts (symmetric, sorted rows, no self loops, no duplicates) with the BA degree structure."""
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    N, m = 3000, 8
    rowptr, col = bench.make_ba_csr(N, m, 0)
    assert rowptr[0] == 0 and rowptr[-1] == len(col) == 2 * m * (N - m)
    deg = np.diff(rowptr)
    assert deg[m:].min() >= m and deg.max() > 10 * m                      # late nodes keep their m links, early nodes are hubs
    rows = np.repeat(np.arange(N), deg)
    assert not np.any(rows == col)                                         # no self loops
    key = rows.astype(np.int64) * N + col
    assert np.all(np.diff(key) > 0)                                        # rows sorted, no duplicate edges
    assert np.array_equal(np.sort(key), np.sort(col.astype(np.int64) * N + rows))   # symmetric


def test_iter_explain_nodes_packed_chunks_without_gpu():
    """Chunked driver for large graphs: pure host logic over _explain_batch (stubbed here, no GPU)."""
    from gnnx.explain import Explainer
    ex = Explainer.__new__(Explainer)
    calls = []
    ex._explain_batch = lambda nodes, graph_idx=0, model="exp", unconstrained=False: (calls.append(list(nodes)) or ("plan%d" % len(calls), np.zeros(len(nodes))))
    out = list(ex.iter_explain_nodes_packed(range(10), 4))
    assert [c[0] for c in out] == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]] and calls == [c[0] for c in out]
    assert [len(c[2]) for c in out] == [4, 4, 2]
    with pytest.raises(ValueError):
        list(ex.iter_explain_nodes_packed([1, 2], 0))


def test_denoise_graph_matches_reference():
    """gnnx.io_utils.denoise_graph (dense API mirror) against the UNMODIFIED reference's denoise_graph on its own golden masks
    (tests/golden/denoise_golden.npz, oracle/gen_golden.py --only denoise): thresholded edges, weights, largest component."""
    import gnnx_oracle as O
    from gnnx import io_utils
    dg = np.load(os.path.join(util.GOLDEN, "denoise_golden.npz"))
    k = int(dg["threshold_num"])
    for which in ("syn1", "syn4"):
        fx = util.load_fixture(which)
        for node in [int(x) for x in dg[which + "_nodes"]]:
            idx, srp, scol, _, _, nbrs = O.extract_neighborhood(fx.rowptr, fx.col, fx.feat, fx.label, node, 3)
            A = O.dense_from_csr(srp, scol)
            ei, ej = np.nonzero(A)
            M = np.zeros_like(A); M[ei, ej] = fx.gold["n%d_mask" % node]
            G0 = io_utils.denoise_graph(M, idx, threshold_num=k, max_component=False)
            e = np.array(sorted((min(u, v), max(u, v)) for u, v in G0.edges()), np.int32).reshape(-1, 2)
            assert np.array_equal(e, dg["%s_n%d_edges" % (which, node)]), (which, node)
            assert np.allclose([G0[u][v]["weight"] for u, v in e], dg["%s_n%d_weights" % (which, node)], rtol=0, atol=0)
            G1 = io_utils.denoise_graph(M, idx, threshold_num=k, max_component=True)
            assert sorted(G1.nodes()) == list(dg["%s_n%d_cc" % (which, node)])
            assert G1.nodes[idx].get("self") == 1 if idx in G1 else True
