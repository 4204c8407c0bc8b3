#!/usr/bin/env python
"""Graph-classification throughput of the model / optimiser variants and of graphs beyond shared memory (explain_graph_var.cu),
next to the default model in the tuned kernel (explain_graph.cu):

    python tools/graph_variants_bench.py [--steps 3] [--warmup 1] [--out FILE]

Small-graph configurations run on bench.make_graph_batch() (4 337 molecule-like graphs padded to 100 nodes, 100 epochs, Philox
init): default, L2, L4, bn (3 layers + --bn), w64 (64/64), sgd (default model, --opt sgd).  The large-graph batch holds 148 graphs
of 1 000 - 4 000 nodes padded to 4 096 (random recursive trees + a sixth extra bonds), with the default model and with L4 + bn.
Kernel time per step = gx_last_explain_ms (device events around the launches); the L2 is overwritten between steps.  One JSON line
on stdout (and in --out) with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-model-explainer_b200"))
import gnnx  # noqa: E402
from gnnx import _abi  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:     # the numbers stay, the label says it could not be read
        return dict(name="unknown (%s)" % e)


def model(rng, d, C_, L, hid, emb):
    sc = lambda *s: (rng.normal(size=s) * 0.4).astype(np.float32)
    dims = [d] + [hid] * (L - 1) + [emb]
    w = {}
    for l in range(1, L + 1):
        w["W%d" % l] = sc(dims[l - 1], dims[l]); w["b%d" % l] = sc(dims[l])
    w["Wp"] = sc(C_, hid * (L - 1) + emb); w["bp"] = sc(C_)
    return w


def large_batch(G=148, max_nodes=4096, d=14, C_=2, seed=1):
    """CSR of G random graphs of 1 000 - 4 000 nodes (a dense (G, 4096, 4096) array would take 2.5 GB)."""
    rng = np.random.default_rng(seed)
    rows, cols = [], []
    feat = np.zeros((G * max_nodes, d), np.float32)
    for g in range(G):
        n = int(rng.integers(1000, 4001))
        par = np.array([rng.integers(0, i) for i in range(1, n)])
        u = np.arange(1, n)
        k = n // 6
        a, b = rng.integers(0, n, k), rng.integers(0, n, k)
        ok = a != b
        e = np.concatenate([np.stack([u, par], 1), np.stack([par, u], 1), np.stack([a[ok], b[ok]], 1), np.stack([b[ok], a[ok]], 1)])
        e = np.unique(e, axis=0)
        rows.append(e[:, 0] + g * max_nodes); cols.append(e[:, 1])
        feat[g * max_nodes + np.arange(n), rng.integers(0, d, n)] = 1.0
    r = np.concatenate(rows); c = np.concatenate(cols)
    order = np.lexsort((c, r))
    r, c = r[order], c[order]
    rowptr = np.zeros(G * max_nodes + 1, np.int64)
    np.add.at(rowptr, r + 1, 1)
    rowptr = np.cumsum(rowptr).astype(np.int32)
    return rowptr, c.astype(np.int32), feat, rng.integers(0, C_, G).astype(np.int32), G, max_nodes


def set_batch_csr(eng, rowptr, col, feat, label, G, n):
    _abi.check(eng._lib.gx_set_graph_batch_csr(eng._h, G, n, rowptr.ctypes.data_as(C.c_void_p), col.ctypes.data_as(C.c_void_p),
                                               feat.ctypes.data_as(C.c_void_p), feat.shape[1], label.ctypes.data_as(C.c_void_p)))
    eng.batch_rowptr, eng.batch_col, eng.batch_G, eng.batch_n = rowptr, col, G, n


def time_config(eng, G, hp, steps, warmup, flush):
    edge_off = eng.plan_graphs(list(range(G)))
    out = np.zeros(int(edge_off[-1]), np.float32)
    ms = []
    for s in range(warmup + steps):
        flush.zero_()
        eng.explain_graphs_host(hp, None, out)
        if s >= warmup:
            ms.append(eng.last_explain_ms())
    return ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bench
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")     # 256 MB > the 126 MB L2
    info = card()
    res = dict(tool="graph_variants_bench", card=info, epochs=a.epochs, steps=a.steps, warmup=a.warmup, init="philox",
               timing="gx_last_explain_ms per step, L2 overwritten between steps", configs={})
    adj, feat, label, W = bench.make_graph_batch()
    G, n, d = adj.shape[0], adj.shape[1], feat.shape[2]
    rng = np.random.default_rng(7)
    small = [("default", W, 3, False, 0), ("L2", model(rng, d, 2, 2, 20, 20), 2, False, 0), ("L4", model(rng, d, 2, 4, 20, 20), 4, False, 0),
             ("bn", model(rng, d, 2, 3, 20, 20), 3, True, 0), ("w64", model(rng, d, 2, 3, 64, 64), 3, False, 0), ("sgd", W, 3, False, 1)]
    t0 = time.time()
    for tag, w, L, bn, opt in small:
        eng = gnnx.Engine(0)
        eng.set_model(w, num_layers=L, bn=bn)
        eng.set_graph_batch(adj, feat, label)
        hp = eng.make_hparams(num_epochs=a.epochs, init=_abi.GX_INIT_PHILOX, seed=1)
        hp.opt = opt
        ms, out = time_config(eng, G, hp, a.steps, a.warmup, flush)
        med = float(np.median(ms))
        res["configs"][tag] = dict(graphs=G, max_nodes=n, layers=L, bn=bn, widths=[int(w["W1"].shape[1]), int(w["W%d" % L].shape[1])],
                                   opt=["adam", "sgd"][opt], kernel_ms=ms, graphs_per_s=G / med * 1e3, mask_checksum=float(out.sum()))
        print("%-8s %8.2f ms  %9.0f graphs/s" % (tag, med, G / med * 1e3), file=sys.stderr)
        eng.close()
    rowptr, col, lfeat, llabel, LG, ln = large_batch(d=d)
    for tag, w, L, bn in (("large_default", W, 3, False), ("large_L4bn", model(rng, d, 2, 4, 20, 20), 4, True)):
        eng = gnnx.Engine(0)
        eng.set_model(w, num_layers=L, bn=bn)
        set_batch_csr(eng, rowptr, col, lfeat, llabel, LG, ln)
        hp = eng.make_hparams(num_epochs=a.epochs, init=_abi.GX_INIT_PHILOX, seed=1)
        ms, out = time_config(eng, LG, hp, max(1, a.steps - 1), a.warmup, flush)
        med = float(np.median(ms))
        nn = np.diff(rowptr).reshape(LG, ln)
        res["configs"][tag] = dict(graphs=LG, max_nodes=ln, layers=L, bn=bn, nodes_min=int((nn > 0).sum(1).min()), nodes_max=int((nn > 0).sum(1).max()),
                                   edges=int(rowptr[-1]), kernel_ms=ms, graphs_per_s=LG / med * 1e3, mask_checksum=float(out.sum()))
        print("%-14s %8.2f ms  %9.1f graphs/s" % (tag, med, LG / med * 1e3), file=sys.stderr)
        eng.close()
    res["wall_s"] = time.time() - t0
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
