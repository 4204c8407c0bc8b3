"""CPU: graph-classification mode with model and optimiser variants (2 / 4 layers, --bn, wide layers; sgd / rmsprop / adagrad and
the schedulers) -- the torch port and the closed form (the graph-variant kernel's specification) against the masks the UNMODIFIED
reference returned (tests/golden/graph_variants_golden.npz, tools/gen_graph_variants_golden.py; 30 epochs)."""
import numpy as np
import pytest

import gnnx_oracle as O
import util

MODEL_CASES = [("L2", 2, False), ("L4", 4, False), ("bn", 3, True), ("L4bn", 4, True), ("w64", 3, False), ("w128", 2, False)]
OPT_CASES = [("sgd", dict(opt="sgd")), ("rmsprop", dict(opt="rmsprop")), ("adagrad", dict(opt="adagrad")),
             ("adamstep", dict(opt="adam", opt_scheduler="step", opt_decay_step=8, opt_decay_rate=0.5)),
             ("sgdcos", dict(opt="sgd", opt_scheduler="cos", opt_restart=12))]


def load():
    return np.load(util.GOLDEN + "/graph_variants_golden.npz"), np.load(util.GOLDEN + "/graphs_golden.npz")


def case_weights(gv, gg, tag):
    """-> (weights, num_layers, bn) of a golden case: the model cases carry their own weights, the optimiser cases use the 3-layer
    20/20 model of graphs_golden.npz."""
    if (tag + "_W1") in gv.files:
        L = int(gv[tag + "_L"])
        w = {k[len(tag) + 1:]: gv[k] for k in gv.files if k.startswith(tag + "_W") or (k.startswith(tag + "_b") and k != tag + "_bn")}
        return w, L, bool(int(gv[tag + "_bn"]))
    return {k: gg[k] for k in util.WKEYS}, 3, False


def case_hparams(tag, epochs):
    over = dict(OPT_CASES).get(tag, {})
    return O.default_hparams(num_epochs=epochs, **over)


def dense_m0(gv, gg, g):
    """M0 (n, n) as the reference drew it: the golden edge entries, ones elsewhere (off-edge entries never reach the result)."""
    n = int(gv["max_nodes"])
    M0 = np.ones((n, n), np.float32)
    ei, ej = np.nonzero(gg["adj"][g])
    M0[ei, ej] = gv["g%d_m0" % g]
    return M0


def test_golden_consistent_with_graph_fixture():
    gv, gg = load()
    assert int(gv["num_graphs"]) == int(gg["num_graphs"]) and int(gv["max_nodes"]) == int(gg["max_nodes"])
    for g in range(int(gv["num_graphs"])):
        assert np.array_equal(gv["g%d_m0" % g], gg["g%d_m0" % g])     # same seeds, same padded size


@pytest.mark.parametrize("tag", [c[0] for c in MODEL_CASES] + [c[0] for c in OPT_CASES])
def test_torch_port_matches_reference(tag):
    gv, gg = load()
    w, L, bn = case_weights(gv, gg, tag)
    E = int(gv["num_epochs"])
    for g in range(int(gv["num_graphs"])):
        ei, ej = np.nonzero(gg["adj"][g])
        got = O.explain_dense_torch(gg["adj"][g].astype(float), gg["feat"][g], int(gg["label"][g]), None, 0, w, dense_m0(gv, gg, g),
                                    hp=case_hparams(tag, E), graph_mode=True, bn=bn)
        assert O.rel_l2(got[ei, ej], gv["%s_g%d_mask" % (tag, g)]) < 1e-6, (tag, g)


@pytest.mark.parametrize("tag", [c[0] for c in MODEL_CASES])
def test_closed_form_matches_reference(tag):
    """The specification the graph-variant kernel implements (fp64), on the Adam cases."""
    gv, gg = load()
    w, L, bn = case_weights(gv, gg, tag)
    E = int(gv["num_epochs"])
    for g in range(int(gv["num_graphs"])):
        ei, ej = np.nonzero(gg["adj"][g])
        got = O.explain_closed_form(gg["adj"][g].astype(float), gg["feat"][g], int(gg["label"][g]), None, 0, w, dense_m0(gv, gg, g),
                                    hp=O.default_hparams(num_epochs=E), graph_mode=True, bn=bn)
        assert O.rel_l2(got[ei, ej], gv["%s_g%d_mask" % (tag, g)]) < 2e-5, (tag, g)
