#!/usr/bin/env python
"""bench.py -- explained-nodes/sec of the GNNExplainer mask-optimisation hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: syn1 BA-House (N=700, 2055 edges, d=10, 4 classes; the graph and the trained
GcnEncoderNode(10,20,20,4,3) weights were produced by the reference's own gengraph/train code, tests/golden/syn1_graph.npz),
explain ALL 700 nodes, 100 mask-optimisation epochs each, reference defaults (Adam lr 0.1, sigmoid mask, 3-hop subgraphs).

One "step" = one pass of the hot path over the node list:
    k-hop extraction (gx_plan_nodes) + mask init + 100-epoch optimisation (gx_explain_nodes) [+ N > 1: the shard bookkeeping
    (gx_count_nodes) and ONE NCCL all-gather of the packed masks (gx_allgather_masks + gx_unshard_masks)].
  value : inputs (graph, model, node list) resident in HBM, mask init drawn on device (Philox), masks left in HBM; CUDA events.
  e2e   : the same step through the C ABI with HOST buffers (node list in, canonical subgraph description and masks out to pinned
          host memory inside the timed region); e2e_python = the drop-in Explainer.explain_nodes call (wall clock).
N = 1: the 700-node list.  N > 1 (one rank per GPU, the product path gnnx.dist.explain_nodes_sharded):
  weak   (the line's value): the list is N x 700 nodes (the 700 nodes, N times), cost-balanced shards -> per-GPU work is fixed;
  strong (reported next to it): the SAME 700-node list sharded over the N ranks, and a 5600-node list (700 x 8) likewise;
  shard_bit_identical: rank 0 explains the gathered list again on one GPU and compares every mask value bit for bit.

--impl reference times the CPU baseline ("port": oracle/gnnx_oracle.explain_dense_torch, the line-by-line restatement that is
bit-exact to the reference on the golden set; the Python reference itself cannot travel to the GPU box) on a bounded sample of the
same workload with all host cores.  extra_workloads (N = 1 only): BASELINE configs[2] syn4, configs[3] graph-mode stand-in,
configs[4] BA(100k, 32) d=128 through the streaming kernel, each with roofline / cpu_baseline / e2e.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "gnn-model-explainer_b200"))

METRIC = "explained-nodes/sec (100 mask-opt epochs each)"
WORKLOAD = "syn1 BA-House, explain all 700 nodes batched, 100 epochs, 3-hop subgraphs"
NUM_EPOCHS = 100
D_FEAT = 10


def load_syn1(name="syn1"):
    g = np.load(os.path.join(ROOT, "tests", "golden", name + "_graph.npz"))
    N = int(g["N"])
    e = g["edges"].astype(np.int64)
    src = np.concatenate([e[:, 0], e[:, 1]]); dst = np.concatenate([e[:, 1], e[:, 0]])
    order = np.lexsort((dst, src))
    src, dst = src[order], dst[order]
    rowptr = np.zeros(N + 1, np.int64)
    np.add.at(rowptr, src + 1, 1)
    rowptr = np.cumsum(rowptr).astype(np.int32)
    weights = {k: g[k] for k in ["W1", "b1", "W2", "b2", "W3", "b3", "Wp", "bp"]}
    return dict(name=name, N=N, rowptr=rowptr, col=dst.astype(np.int32), feat=g["feat"], label=g["label"].astype(np.int32), pred=g["pred"],
                pred_label=np.argmax(g["pred"], 1).astype(np.int32), weights=weights)


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port, bounded sample
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_one(node):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gnnx_oracle as O
    if "g" not in _W:
        _W["g"] = load_syn1(_W.get("name", "syn1"))
        torch.set_num_threads(_W.get("threads", 1))
    g = _W["g"]
    idx, srp, scol, sfeat, slabel, nbrs = O.extract_neighborhood(g["rowptr"], g["col"], g["feat"], g["label"], int(node), 3)
    A = O.dense_from_csr(srp, scol)
    M0 = O.draw_m0(len(nbrs), seed=1000 + int(node))
    out = O.explain_dense_torch(A, sfeat, slabel[idx], g["pred_label"][nbrs], idx, g["weights"], M0,
                                hp=O.default_hparams(num_epochs=NUM_EPOCHS))
    return float(out.sum())


def cpu_sample_nodes(k, N=700):
    """k nodes spread evenly over the N (every N/k-th node): same size mix as the full list."""
    return [int(x) for x in np.linspace(0, N - 1, k).round().astype(int)]


def run_cpu_pool(sample, procs):
    """nodes/s over `sample` with `procs` single-thread worker processes (the strongest way to run the
    reference's per-node loop on all host cores).  Must be called BEFORE torch is imported in this
    process: the pool forks, and forking after torch started its OpenMP pool can deadlock."""
    assert "torch" not in sys.modules, "fork-pool must start before torch is imported"
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        pool.map(_cpu_one, sample[:procs], chunksize=1)  # warm-up: every worker imports torch, loads the graph
        t0 = time.perf_counter()
        pool.map(_cpu_one, sample, chunksize=1)
        dt = time.perf_counter() - t0
    return len(sample) / dt, dt


def run_cpu_sequential(sample, budget_s):
    """The reference as written: sequential loop over nodes, torch intra-op threads = torch default
    (all cores).  Stops after budget_s seconds."""
    import torch
    torch.set_num_threads(min(torch.get_num_threads(), 16))  # >16 intra-op threads only slow these tiny ops down
    _W["threads"] = torch.get_num_threads()
    _cpu_one(sample[0])
    t0 = time.perf_counter()
    done = 0
    for n in sample:
        _cpu_one(n)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return done / (time.perf_counter() - t0), torch.get_num_threads(), done


def main_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = a.cpu_procs or min(cores, 64)
    _W["name"] = a.workload if a.workload == "syn4" else "syn1"
    NN = 871 if a.workload == "syn4" else 700
    workload = WORKLOAD if a.workload != "syn4" else "syn4 Tree-Cycle, explain all 871 nodes batched, 100 epochs, 3-hop subgraphs"
    sample = cpu_sample_nodes(max(2 * procs, 16), NN)
    steps = a.steps  # each step is one bounded sample; worker warm-up is inside run_cpu_pool
    vals = []
    for _ in range(steps):
        v, dt = run_cpu_pool(sample, procs)
        vals.append(v)
    v = float(np.mean(vals))
    seq_v, seq_threads, seq_done = run_cpu_sequential(cpu_sample_nodes(6, NN), 20.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "nodes/s", "n_gpus": a.gpus, "steps": steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 * len(sample) / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sample": "%d of the %d nodes (evenly spaced), %d single-thread worker processes on %d host cores" % (len(sample), NN, procs, cores)},
        "cpu_baseline": {"value": v, "unit": "nodes/s", "cores": procs, "kind": "port",
                         "sample": "%d evenly spaced nodes x 100 epochs, one single-thread worker process per core (%d procs), %.1f s" % (len(sample), procs, dt),
                         "as_written_sequential": {"value": seq_v, "torch_threads": seq_threads, "nodes": seq_done}},
        "e2e": {"value": v, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler (NVML) -- runs during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md recipe): `nvidia-smi --query-gpu=... -lms 10` in a child
    PROCESS started when the sampler is created (nvidia-smi needs a few hundred ms before its first line); begin() / end() bracket the
    timed region and only the samples stamped inside it count.  (A polling thread inside the benchmark process competes for the GIL
    with the host side of the step: +1 ms per 5 600-node sharded step at 8 GPUs.)"""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_power_brake_slowdown")

    def __init__(self, index):
        import subprocess
        self.index = index
        self.err = None
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception as e:
            self.proc, self.err = None, repr(e)

    def start(self):      # (kept for callers that mark the beginning of the timed region this way)
        self.begin()

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        if self.t1 is None:
            self.end()
        rows, sm_max = [], None
        if self.proc is not None:
            try:
                self.proc.terminate()
                out = self.proc.communicate(timeout=5)[0]
            except Exception as e:
                out, self.err = "", repr(e)
            for line in out.splitlines():
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), [v.lower().startswith("active") for v in f[3:8]]))
                    sm_max = float(f[2])
                except ValueError:
                    continue
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap", "hw_power_brake"]
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [r for r in rows if t0 - 0.005 <= r[0] <= self.t1 + 0.005]
        note = "samples stamped inside the timed region"
        if not inside and rows:      # a region shorter than the sampling period: the three samples nearest to it
            mid = 0.5 * (t0 + self.t1)
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            note = "timed region shorter than the 10 ms sampling period: the three samples nearest to it"
        reasons = sorted({nm for r in inside for nm, on in zip(names, r[2]) if on})
        return {"sm_mhz": float(np.median([r[1] for r in inside])) if inside else None, "sm_max_mhz": sm_max, "reasons": reasons, "samples": len(inside),
                "how": "nvidia-smi -lms 10 in a child process; " + note, **({"error": self.err} if self.err else {})}


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[3] stand-in (dataset absent, no network): 4337 padded molecule-like graphs, graph-level masks
# ------------------------------------------------------------------------------------------------
def make_graph_batch(G=4337, max_nodes=100, d=14, C=2, seed=0):
    rng = np.random.default_rng(seed)
    adj = np.zeros((G, max_nodes, max_nodes), np.uint8)
    feat = np.zeros((G, max_nodes, d), np.float32)
    for g in range(G):
        n = int(np.clip(rng.normal(30, 20), 4, max_nodes))
        par = np.array([rng.integers(0, i) for i in range(1, n)])          # random recursive tree
        u = np.arange(1, n)
        adj[g, u, par] = 1; adj[g, par, u] = 1
        k = max(1, n // 6)
        a, b = rng.integers(0, n, k), rng.integers(0, n, k)
        ok = a != b
        adj[g, a[ok], b[ok]] = 1; adj[g, b[ok], a[ok]] = 1
        feat[g, np.arange(n), rng.integers(0, d, n)] = 1.0
    label = rng.integers(0, C, G).astype(np.int32)
    sc = lambda *s_: (rng.normal(size=s_) * 0.4).astype(np.float32)
    W = dict(W1=sc(d, 20), b1=sc(20), W2=sc(20, 20), b2=sc(20), W3=sc(20, 20), b3=sc(20), Wp=sc(C, 60), bp=sc(C))
    return adj, feat, label, W


def _cpu_graph_one(args):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gnnx_oracle as O
    torch.set_num_threads(1)
    A, X, y, W, seed = args
    M0 = O.draw_m0(A.shape[0], seed=seed)
    return float(O.explain_dense_torch(A.astype(float), X, int(y), None, 0, W, M0, hp=O.default_hparams(num_epochs=NUM_EPOCHS), graph_mode=True).sum())


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[4]: dense BA graph (N=100k, m=32 => avg degree 64), d=128, 3-hop neighbourhood ~ the whole graph.
# Every task runs in the streaming kernel (explain_stream.cu); a step explains --c5-nodes nodes (default: one per SM).
# ------------------------------------------------------------------------------------------------
def make_ba_csr(N, m, seed=0):
    """Barabasi-Albert preferential attachment (numpy): node v attaches to m distinct earlier nodes drawn from the endpoint list."""
    rng = np.random.default_rng(seed)
    rep = np.empty(2 * m * N, np.int32)
    L = 0
    edges = np.empty((m * (N - m), 2), np.int32)
    k = 0
    targets = np.arange(m, dtype=np.int32)
    for v in range(m, N):
        edges[k:k + m, 0] = v; edges[k:k + m, 1] = targets; k += m
        rep[L:L + m] = targets; rep[L + m:L + 2 * m] = v; L += 2 * m
        t = np.unique(rep[rng.integers(0, L, 2 * m)])
        while len(t) < m:
            t = np.unique(np.concatenate([t, rep[rng.integers(0, L, m)]]))
        targets = rng.permutation(t)[:m].astype(np.int32)
    src = np.concatenate([edges[:, 0], edges[:, 1]]); dst = np.concatenate([edges[:, 1], edges[:, 0]])
    order = np.lexsort((dst, src))
    src, dst = src[order], dst[order]
    rowptr = np.zeros(N + 1, np.int64)
    np.add.at(rowptr, src + 1, 1)
    return np.cumsum(rowptr).astype(np.int32), dst.astype(np.int32)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _peak_hbm():
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        return float(json.load(open(pk)).get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _sm_metrics(tag):
    """ncu --set full readings of THIS build's kernels (profiles/r02_sm_metrics.json, written from the committed ncu capture):
    what actually bounds the shared-memory kernels (SURVEY 8 d-roof: issue/latency, not HBM)."""
    p = os.path.join(ROOT, "profiles", "r02_sm_metrics.json")
    if os.path.exists(p):
        return json.load(open(p)).get(tag)
    return None


def _c5_traffic(K):
    """DRAM bytes of one configs[4] launch, from the committed ncu capture (one 100 000-node task x 15 updates: dram__bytes_read + write
    per task-epoch) x K tasks x 99 updates; None when the capture is not there."""
    m = _sm_metrics("c5")
    try:
        return float(m["steady_state_one_task_16_epochs"]["dram_bytes_per_task_epoch"]) * K * (NUM_EPOCHS - 1)
    except Exception:
        return None


def cpu_baseline_subprocess(workload, timeout=300):
    """The CPU arm on a bounded sample, in a separate process (the worker pool must fork before torch/CUDA exist)."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", "1"],
                           capture_output=True, text=True, timeout=timeout)
        return json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as e:
        return {"error": repr(e)[:200]}


def make_explainer(g, device, init="device", num_epochs=NUM_EPOCHS, seed=1234, print_training=False):
    import types
    import torch
    import gnnx
    args = types.SimpleNamespace(num_gc_layers=3, num_epochs=num_epochs, lr=0.1, opt="adam", opt_scheduler="none", mask_act="sigmoid",
                                 mask_bias=False, gpu=False, bias=True, method="base", dataset=g["name"], bmname=None, hidden_dim=20,
                                 output_dim=20, name_suffix="", explainer_suffix="", logdir="/tmp/gnnx_bench_log",
                                 gnnx_init=init, gnnx_seed=seed)
    w = g["weights"]
    model = gnnx.models.GcnEncoderNode(w["W1"].shape[0], 20, 20, w["Wp"].shape[0], 3, bn=False, args=args)
    sd = {"conv_first.weight": w["W1"], "conv_first.bias": w["b1"], "conv_block.0.weight": w["W2"], "conv_block.0.bias": w["b2"],
          "conv_last.weight": w["W3"], "conv_last.bias": w["b3"], "pred_model.weight": w["Wp"], "pred_model.bias": w["bp"]}
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    N = g["N"]
    A = np.zeros((N, N), np.float32)
    A[np.repeat(np.arange(N), np.diff(g["rowptr"])), g["col"]] = 1
    return gnnx.Explainer(model=model, adj=A[None], feat=g["feat"][None], label=g["label"][None], pred=g["pred"][None], train_idx=[],
                          args=args, writer=None, print_training=print_training, graph_idx=-1, device=device)


class Ctx:
    pass


def gpu_ctx(a):
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.world = int(os.environ.get("WORLD_SIZE", "1")); c.rank = int(os.environ.get("RANK", "0")); c.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if c.world != a.gpus and c.world == 1 and a.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun with %d ranks" % (a.gpus, a.gpus))
    torch.cuda.set_device(c.local_rank)
    c.dev = torch.device("cuda", c.local_rank)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=c.dev)
    c.flush = torch.empty(256 << 20, dtype=torch.uint8, device=c.dev)  # > 126 MB L2
    c.stream = torch.cuda.current_stream(c.dev)
    return c


def barrier(c):
    import torch
    import torch.distributed as dist
    if c.world > 1:
        dist.barrier()
    torch.cuda.synchronize(c.dev)


def timed(c, fn, steps, warmup, sampler=None, after=None):
    """W untimed warm-up steps, then K steps bracketed by barrier + synchronize; device time from CUDA events on the launching stream
    (L2 flushed between steps, outside the event pair); MAX over ranks.  Returns (total ms, [per-step after() values], wall s, clocks)."""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        c.flush.zero_()
        fn()
    barrier(c)
    if sampler is not None:
        sampler.begin()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    extra = []
    t0 = time.perf_counter()
    for i in range(steps):
        c.flush.zero_()
        ev[i][0].record(c.stream)
        fn()
        ev[i][1].record(c.stream)
        if after is not None:
            extra.append(after())
    barrier(c)
    wall = time.perf_counter() - t0
    if sampler is not None:
        sampler.end()
    clocks = sampler.stop() if sampler is not None else None
    ms = float(sum(s.elapsed_time(e) for s, e in ev))
    t = torch.tensor([ms], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), extra, wall, clocks


DUMP_BYTES = 60 << 20      # --dump-outputs stays below 64 MB in all (npy headers included)


def write_outputs(path, arrays, seed=0):
    """--dump-outputs: arrays[name] -> path/<name>.npy, float32 arrays as float32 and every other array as float64 (exact for the
    int32 / int64 plan arrays).  When the arrays hold more than DUMP_BYTES, each keeps a share of the budget proportional to its size:
    the values at sorted, unique positions drawn from a generator seeded with `seed`, so two runs with the same arguments write the
    same positions; the positions go to path/<name>_index.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v).ravel() for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    for name, v in arrays.items():
        if total > DUMP_BYTES:
            k = int(DUMP_BYTES * v.nbytes / total) // (v.itemsize + 8)      # each kept value also stores its float64 position
            idx = np.unique(np.random.default_rng(seed).integers(0, v.size, k))
            np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))
            v = v[idx]
        np.save(os.path.join(path, name + ".npy"), v)


def bench_nodes(a, c, name, with_cpu=True, sampler=None, dump=None):
    """syn1 / syn4 on ONE GPU through the C ABI: device-resident value + host-buffer e2e."""
    import ctypes as C
    import torch
    import gnnx
    from gnnx import _abi
    g = load_syn1(name)
    workload = WORKLOAD if name == "syn1" else "syn4 Tree-Cycle, explain all %d nodes batched, 100 epochs, 3-hop subgraphs" % g["N"]
    eng = gnnx.Engine(c.local_rank)
    eng.set_model(g["weights"])
    eng.set_graph_csr(g["rowptr"], g["col"], g["feat"], g["label"], g["pred_label"])
    eng.set_stream(c.stream.cuda_stream)
    nodes = np.arange(g["N"], dtype=np.int32)
    count = len(nodes)
    plan = eng.plan_nodes(nodes, 3)
    total_e, total_n = plan.total_edges, plan.total_nodes
    sizes = np.diff(plan.edge_off); n_t = np.diff(plan.node_off)
    d_feat = g["feat"].shape[1]
    algo = float(NUM_EPOCHS * (84.0 * sizes.sum() + 8.0 * d_feat * n_t.sum()))          # SURVEY 8(d) B_epoch x 100 epochs
    out_dev = torch.empty(total_e, dtype=torch.float32, device=c.dev)
    out_host = torch.empty(total_e, dtype=torch.float32).pin_memory()
    nodes_host = torch.from_numpy(nodes.copy()).pin_memory()
    nbr_host = torch.empty(total_n, dtype=torch.int32).pin_memory()
    srp_host = torch.empty(total_n + count, dtype=torch.int32).pin_memory()
    scol_host = torch.empty(total_e, dtype=torch.int32).pin_memory()
    noff = np.empty(count + 1, np.int64); eoff = np.empty(count + 1, np.int64); idxn = np.empty(count, np.int32)
    lib = _abi.lib()
    hp = eng.make_hparams(num_epochs=NUM_EPOCHS, init=_abi.GX_INIT_PHILOX, seed=1234 + c.rank)

    def step_device():
        eng.plan_nodes(nodes_host.numpy(), 3, fetch=False)
        eng.explain_nodes_ptr(hp, _abi.GX_DEVICE, 0, out_dev.data_ptr())

    def step_e2e():
        eng.plan_nodes(nodes_host.numpy(), 3, fetch=False)
        _abi.check(lib.gx_plan_fetch(eng._h, C.c_void_p(noff.ctypes.data), C.c_void_p(eoff.ctypes.data), C.c_void_p(nbr_host.data_ptr()),
                                     C.c_void_p(idxn.ctypes.data), C.c_void_p(srp_host.data_ptr()), C.c_void_p(scol_host.data_ptr())))
        eng.explain_nodes_ptr(hp, _abi.GX_HOST, 0, out_host.data_ptr())

    l0 = eng.launch_count()
    ms_dev, kern, wall, clocks = timed(c, step_device, a.steps, a.warmup, sampler, after=eng.last_explain_ms)
    launches = (eng.launch_count() - l0) * a.steps // (a.steps + a.warmup)
    if dump:      # the masks of the last timed step and the subgraph description its plan holds
        torch.cuda.synchronize(c.dev)
        p = eng.fetch_plan(nodes)
        write_outputs(dump, {"masks": out_dev.cpu().numpy(), "node_off": p.node_off, "edge_off": p.edge_off, "neighbors": p.neighbors,
                             "node_idx_new": p.node_idx_new, "sub_rowptr": p.sub_rowptr, "sub_col": p.sub_col})
    ms_e2e, _, _, _ = timed(c, step_e2e, a.steps, max(3, a.warmup))
    kern_ms = float(np.mean(kern))
    peak, peak_src = _peak_hbm()
    achieved = algo / (kern_ms / 1e3) / 1e9
    traffic = None
    tj = os.path.join(ROOT, "profiles", "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else "r01_traffic.json")
    if os.path.exists(tj) and name == "syn1":
        traffic = float(json.load(open(tj))["traffic_bytes_per_step"])
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "kernel": "explain_node_kernel (one launch per size class, concurrent streams) + outer_pairs_kernel",
            "kernel_ms_per_step": kern_ms, "algorithmic_bytes_per_step": algo,
            "sm": _sm_metrics(name),
            "note": "EQUIVALENT bandwidth: the SURVEY 8(d) algorithmic bytes (84*E_d + 8*n*d per node-epoch, x100, summed over the nodes) are served "
                    "from shared memory; DRAM traffic (ncu) is the compulsory one-time read of the subgraphs.  The kernel is issue/latency bound: see "
                    "roofline.sm (ncu --set full of this build) and DESIGN.md section 6"}
    h2d = int(count * 4 + 8 * (NUM_EPOCHS - 1) + 24)
    d2h = int(count * 112 * 2 + (total_n + total_n + count + total_e) * 4 + total_e * 4)
    line = {
        "metric": METRIC, "value": count * a.steps / (ms_dev / 1e3), "unit": "nodes/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "nodes_per_gpu": count, "epochs": NUM_EPOCHS, "sum_E_d": int(sizes.sum()), "sum_n": int(n_t.sum()),
                   "init": "device Philox N(1,2/n)", "l2": "flushed between steps (256 MiB write)", "parallelism": "dp1"},
        "e2e": {"value": count * a.steps / (ms_e2e / 1e3), "unit": "nodes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / a.steps, "api": "C ABI, host buffers (gx_plan_nodes + gx_plan_fetch + gx_explain_nodes GX_HOST)"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
        "cpu_baseline": cpu_baseline_subprocess(name) if with_cpu else None, "wall_s_timed_region": wall,
    }
    eng.close()
    return line, g


def bench_python_dropin(c, g, reps=3):
    """e2e_python: wall clock of the drop-in call a user of the reference makes, Explainer.explain_nodes(range(N)), host arrays out."""
    import torch
    nodes = list(range(g["N"]))
    res = {"unit": "nodes/s", "call": "gnnx.Explainer.explain_nodes(range(%d)) -> list of (n,n) float64 arrays" % g["N"]}
    for key, init, kw in (("device_init_views", "device", dict(save=False, copy=False)), ("device_init", "device", dict(save=False)),
                          ("torch_init", "torch", dict(save=False)), ("torch_init_save_npy", "torch", dict(save=True))):
        ex = make_explainer(g, c.local_rank, init=init)
        ex.explain_nodes(nodes[:32], save=False)
        ts = []
        for _ in range(reps if "save" not in key else 1):
            torch.cuda.synchronize(c.dev)
            t0 = time.perf_counter()
            out = ex.explain_nodes(nodes, **kw)
            ts.append(time.perf_counter() - t0)
        res[key] = {"value": len(nodes) / min(ts), "ms_per_call": 1e3 * min(ts)}
        assert len(out) == len(nodes) and out[5].dtype == np.float64
        ex.engine.close()
    # latency of ONE Explainer.explain(node) call (the reference's unit of use) on the most expensive node, default and latency mode
    ex = make_explainer(g, c.local_rank, init="device")
    for key, lat in (("single_explain_call_ms", False), ("single_explain_call_ms_latency_mode", True)):
        ex.engine.debug_cluster(0 if lat else 1, 0)
        ex.explain(0)
        ts = []
        for _ in range(10):
            torch.cuda.synchronize(c.dev)
            t0 = time.perf_counter()
            ex.explain(0)
            ts.append(time.perf_counter() - t0)
        res[key] = {"wall_ms": 1e3 * float(np.median(ts)), "kernel_ms": ex.engine.last_explain_ms()}
    ex.engine.close()
    res["value"] = res["device_init"]["value"]
    res["note"] = ("single_explain_call: Explainer.explain(0), node 0 = the most expensive syn1 task; latency mode (args.gnnx_latency / gx_debug_set_cluster(h, 0, 0)) runs it on a 4-CTA cluster. "
                   "torch_init draws the reference's n^2 normals per node on the host (bit-compatible M0 under torch.manual_seed); save_npy writes the "
                   "reference's 700 .npy files (~0.3 GB); *_views returns views of a pinned buffer reused by the next call")
    return res


def bench_sharded(a, c, dump=None):
    """N > 1: gnnx.dist.explain_nodes_sharded (count -> cost-balanced shards -> explain -> ONE all-gather -> unshard)."""
    import torch
    import torch.distributed as dist
    from gnnx.dist import explain_nodes_sharded, ensure_comm
    g = load_syn1("syn1")
    ex = make_explainer(g, c.local_rank, init="device")
    ex.engine.set_stream(c.stream.cuda_stream)
    ensure_comm(ex.engine)
    base = np.arange(g["N"], dtype=np.int32)
    lists = {"weak": np.tile(base, c.world), "strong_700": base, "strong_5600": np.tile(base, 8)}
    res = {}
    sampler = ClockSampler(c.local_rank) if c.rank == 0 else None
    keep = {}
    for key, nodes in lists.items():
        def step():
            keep["out"] = explain_nodes_sharded(ex, nodes)
        l0 = ex.engine.launch_count()
        ms, kern, wall, clocks = timed(c, step, a.steps, a.warmup, sampler if key == "weak" else None, after=ex.engine.last_explain_ms)
        res[key] = {"nodes": int(len(nodes)), "ms_per_step": ms / a.steps, "value": len(nodes) * a.steps / (ms / 1e3),
                    "kernel_ms_per_step": float(np.mean(kern)), "launches_per_step": (ex.engine.launch_count() - l0) // (a.steps + a.warmup)}
        if key == "weak":
            res[key]["clocks"] = clocks
            res[key]["wall"] = wall
            if dump and c.rank == 0:      # every rank holds the gathered masks of the whole list
                write_outputs(dump, {"masks": keep["out"][0].cpu().numpy(), "edge_off": keep["out"][1]})
    # the strong-scaled 700-node list again in latency mode (gx_debug_set_cluster(h, 0, 0)): a shard leaves SMs idle, so its most expensive
    # tasks run on thread-block clusters; masks agree with the default mode to round-off, not bit for bit, hence opt-in
    ex.engine.debug_cluster(0, 0)
    nodes = lists["strong_700"]

    def step_lat():
        keep["out"] = explain_nodes_sharded(ex, nodes)
    l0 = ex.engine.launch_count()
    ms, kern, _w, _c = timed(c, step_lat, a.steps, a.warmup, None, after=ex.engine.last_explain_ms)
    counts, cs = ex.engine.plan_class_counts()
    res["strong_700_latency_mode"] = {"nodes": int(len(nodes)), "ms_per_step": ms / a.steps, "value": len(nodes) * a.steps / (ms / 1e3), "kernel_ms_per_step": float(np.mean(kern)),
                                      "launches_per_step": (ex.engine.launch_count() - l0) // (a.steps + a.warmup), "rank0_cluster_tasks": int(counts[6]), "rank0_cluster_size": cs}
    ex.engine.debug_cluster(1, 0)
    # e2e: the same sharded call + delivery of ALL gathered masks into pinned host memory on every rank (what explain_nodes returns)
    values, offsets, _ = explain_nodes_sharded(ex, lists["weak"])
    host = torch.empty(int(offsets[-1]), dtype=torch.float32).pin_memory()

    def step_e2e():
        v, _o, _p = explain_nodes_sharded(ex, lists["weak"])
        with torch.cuda.stream(c.stream):
            host.copy_(v, non_blocking=True)
        c.stream.synchronize()
    ms, _k, _w, _c = timed(c, step_e2e, a.steps, a.warmup)
    res["weak_e2e"] = {"ms_per_step": ms / a.steps, "value": len(lists["weak"]) * a.steps / (ms / 1e3), "d2h_bytes_per_step": int(host.numel() * 4),
                       "h2d_bytes_per_step": int(4 * len(lists["weak"]))}
    # bit identity of the sharded result against one GPU (rank 0), on the weak list
    ident = None
    if c.rank == 0:
        plan, full = ex.explain_nodes_packed(lists["weak"])
        ident = bool(np.array_equal(values.cpu().numpy(), full) and np.array_equal(offsets, plan.edge_off))
    n_all, e_all = ex.engine.count_nodes(lists["weak"], 3)
    barrier(c)
    ex.engine.comm_destroy()
    ex.engine.close()
    return g, res, ident, int(e_all.sum()), int(n_all.sum())


def main_ours(a):
    import torch.distributed as dist
    c = gpu_ctx(a)
    if a.workload in ("syn1", "syn4") and c.world == 1:
        sampler = ClockSampler(c.local_rank)
        line, g = bench_nodes(a, c, a.workload, with_cpu=not a.no_cpu, sampler=sampler, dump=a.dump_outputs)
        if a.workload == "syn1":
            try:
                line["e2e_python"] = bench_python_dropin(c, g)
            except Exception as e:  # the drop-in measurement must not take the contract line down
                line["e2e_python"] = {"error": repr(e)[:300]}
            if not a.no_extra:
                extras = {}
                small = argparse.Namespace(**{**vars(a), "steps": max(3, a.steps // 4), "warmup": 3})
                for nm, fn in (("syn4", lambda: bench_nodes(small, c, "syn4", with_cpu=not a.no_cpu)[0]), ("graphs", lambda: bench_graphs(small, c, with_cpu=not a.no_cpu)),
                               ("c5", lambda: bench_c5(argparse.Namespace(**{**vars(a), "steps": 1, "warmup": 1}), c))):
                    try:
                        extras[nm] = fn()
                    except Exception as e:
                        extras[nm] = {"error": repr(e)[:300]}
                line["extra_workloads"] = extras
        print(json.dumps(line), flush=True)
        return
    # N > 1
    g, res, ident, sum_e, sum_n = bench_sharded(a, c, dump=a.dump_outputs)
    if c.rank == 0:
        w = res["weak"]
        peak, peak_src = _peak_hbm()
        algo = float(NUM_EPOCHS * (84.0 * sum_e + 8.0 * D_FEAT * sum_n)) / c.world      # per GPU
        achieved = algo / (w["kernel_ms_per_step"] / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": w["value"], "unit": "nodes/s", "n_gpus": c.world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": w["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD + " -- x%d: the 700-node list repeated %d times, cost-balanced shards (~700 nodes per GPU)" % (c.world, c.world),
                       "nodes_total": w["nodes"], "nodes_per_gpu": w["nodes"] // c.world, "epochs": NUM_EPOCHS, "init": "device Philox N(1,2/n)",
                       "l2": "flushed between steps (256 MiB write)",
                       "parallelism": "dp%d: gnnx.dist.explain_nodes_sharded = k-hop sizes (gx_count_nodes, cached per graph) + per-rank gx_plan_nodes/gx_explain_nodes + ONE ncclAllGather (gx_allgather_masks) + gx_unshard_masks" % c.world},
            "e2e": {"value": res["weak_e2e"]["value"], "unit": "nodes/s", "h2d_bytes_per_step": res["weak_e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": res["weak_e2e"]["d2h_bytes_per_step"],
                    "ms_per_step": res["weak_e2e"]["ms_per_step"], "api": "gnnx.dist.explain_nodes_sharded(Explainer, nodes): node list from host memory in, the packed masks of ALL nodes "
                    "copied to pinned host memory on every rank inside the timed region (value: masks left in HBM)"},
            "gpu_launches": int(w["launches_per_step"] * a.steps), "clocks": w.get("clocks"),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "kernel": "explain_node_kernel, per GPU", "kernel_ms_per_step": w["kernel_ms_per_step"], "algorithmic_bytes_per_step": algo,
                         "sm": _sm_metrics("syn1"), "note": "equivalent bandwidth of rank 0's shard, see the N = 1 line"},
            "cpu_baseline": None,
            "strong": {"list_700": res["strong_700"], "list_700_latency_mode": res["strong_700_latency_mode"], "list_5600": res["strong_5600"],
                       "note": "the SAME list sharded over the N ranks (total work fixed); the 700-node list is bounded by its largest task's critical path, which latency mode (thread-block clusters for the expensive tasks of a shard that leaves SMs idle; round-off instead of bit identity) shortens"},
            "shard_bit_identical": ident,
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def bench_graphs(a, c, with_cpu=True, dump=None):
    """BASELINE configs[3] stand-in (Mutagenicity is not in the image): 4337 padded molecule-like graphs, graph-level masks."""
    import ctypes as C
    import torch
    import gnnx
    from gnnx import _abi
    adj, feat, label, W = make_graph_batch()
    G = adj.shape[0]
    eng = gnnx.Engine(c.local_rank)
    eng.set_stream(c.stream.cuda_stream)
    eng.set_model(W)
    eng.set_graph_batch(adj, feat, label)
    gids = np.arange(G, dtype=np.int32)
    edge_off = eng.plan_graphs(gids)
    te = int(edge_off[-1])
    out_host = torch.empty(te, dtype=torch.float32).pin_memory()
    out_dev = torch.empty(te, dtype=torch.float32, device=c.dev)
    hp = eng.make_hparams(num_epochs=NUM_EPOCHS, init=_abi.GX_INIT_PHILOX, seed=7)
    lib = _abi.lib()

    def step_dev():
        eng.plan_graphs(gids)
        _abi.check(lib.gx_explain_graphs(eng._h, C.byref(hp), _abi.GX_DEVICE, None, C.c_void_p(out_dev.data_ptr()), None))

    def step_e2e():
        eng.plan_graphs(gids)
        _abi.check(lib.gx_explain_graphs(eng._h, C.byref(hp), _abi.GX_HOST, None, C.c_void_p(out_host.data_ptr()), None))

    l0 = eng.launch_count()
    ms_dev, kern, _, _ = timed(c, step_dev, a.steps, a.warmup, after=eng.last_explain_ms)
    if dump:
        write_outputs(dump, {"masks": out_dev.cpu().numpy(), "edge_off": edge_off})
    launches = (eng.launch_count() - l0) * a.steps // (a.steps + a.warmup)      # this library's kernels inside the timed region (counted by the handle)
    ms_e2e, _, _, _ = timed(c, step_e2e, a.steps, a.warmup)
    kern_ms = float(np.mean(kern))
    n_act = int((adj.sum(2) > 0).sum())
    algo = float(NUM_EPOCHS * (84.0 * te + 8.0 * feat.shape[2] * n_act))
    peak, peak_src = _peak_hbm()
    line = {"metric": "explained-graphs/sec (100 mask-opt epochs each)", "value": G * a.steps / (ms_dev / 1e3), "unit": "graphs/s", "n_gpus": 1,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[3] stand-in: %d padded graphs (max_nodes 100, d=14), graph-level mask, 100 epochs" % G, "sum_E_d": te, "init": "device Philox"},
            "e2e": {"value": G * a.steps / (ms_e2e / 1e3), "unit": "graphs/s", "ms_per_step": ms_e2e / a.steps, "h2d_bytes_per_step": int(G * 4), "d2h_bytes_per_step": int(te * 4)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": algo / (kern_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": algo / (kern_ms / 1e3) / 1e9 / peak, "traffic": None,
                         "peak_source": peak_src, "kernel": "explain_graph_kernel", "kernel_ms_per_step": kern_ms, "algorithmic_bytes_per_step": algo,
                         "note": "equivalent bandwidth (shared-memory resident, latency bound), as for syn1"},
            "cpu_baseline": cpu_baseline_subprocess("graphs") if with_cpu else None}
    eng.close()
    return line


def bench_c5(a, c, dump=None):
    """BASELINE configs[4]: BA(N, m) d=128, 3-hop neighbourhood ~ the whole graph, every task in the streaming kernel; a step explains
    --c5-nodes nodes (default one per SM).  Includes a parity check AT THIS SCALE: a few epochs of one or two of the explained nodes
    against the fp64 sparse edge-list specification (oracle/kernel_spec.py, pinned to the reference through the chain in tests/test_oracle.py)."""
    import torch
    import scipy.sparse as sp
    import gnnx
    from gnnx import _abi
    N, m, d, C = a.c5_n, a.c5_m, 128, 4
    rng = np.random.default_rng(0)
    t0 = time.perf_counter()
    rowptr, col = make_ba_csr(N, m, 0)
    X = rng.normal(size=(N, d)).astype(np.float32)
    label = rng.integers(0, C, N).astype(np.int32)
    sc = lambda *s_: (rng.normal(size=s_) * 0.3).astype(np.float32)
    W = dict(W1=sc(d, 20), b1=sc(20), W2=sc(20, 20), b2=sc(20), W3=sc(20, 20), b3=sc(20), Wp=sc(C, 60), bp=sc(C))
    A = sp.csr_matrix((np.ones(len(col), np.float32), col, rowptr), shape=(N, N))
    nrm = lambda Y: Y / np.maximum(np.linalg.norm(Y, axis=1, keepdims=True), 1e-12)
    H1 = np.maximum(nrm((A @ X) @ W["W1"] + W["b1"]), 0); H2 = np.maximum(nrm((A @ H1) @ W["W2"] + W["b2"]), 0)
    H3 = nrm((A @ H2) @ W["W3"] + W["b3"])
    pred_label = np.argmax(np.concatenate([H1, H2, H3], 1) @ W["Wp"].T + W["bp"], 1).astype(np.int32)
    gen_s = time.perf_counter() - t0
    eng = gnnx.Engine(c.local_rank)
    eng.set_stream(c.stream.cuda_stream)
    eng.set_model(W)
    eng.set_graph_csr(rowptr, col, X, label, pred_label)
    K = a.c5_nodes
    nodes = np.random.default_rng(1).permutation(N)[:K].astype(np.int32)
    hp = eng.make_hparams(num_epochs=NUM_EPOCHS, init=_abi.GX_INIT_PHILOX, seed=99)
    # ---- parity at scale (before the timed run; separate small calls with host-supplied M0)
    parity = None
    if a.c5_parity > 0:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import kernel_spec as KS
        errs, pt0, spec_s, spec_ep = [], time.perf_counter(), 0.0, 0
        for node, ep in list(zip(nodes[: a.c5_parity], (4, 3, 3, 3)))[: a.c5_parity]:
            plan = eng.plan_nodes([int(node)], 3)
            rp, cl = plan.csr_of(0)
            nb = plan.neighbors_of(0)
            n = len(nb)
            m0 = (1.0 + np.sqrt(2.0 / n) * np.random.default_rng(int(node)).standard_normal(plan.total_edges)).astype(np.float32)
            got = np.zeros(plan.total_edges, np.float32)
            eng.explain_nodes_host(eng.make_hparams(num_epochs=ep), m0, got)
            ts0 = time.perf_counter()
            ref = KS.explain_pruned_edges_sparse(rp, cl, X[nb], int(label[node]), pred_label[nb], int(plan.node_idx_new[0]), W, m0, num_epochs=ep)
            spec_s += time.perf_counter() - ts0; spec_ep += ep - 1
            errs.append({"node": int(node), "n": int(n), "E_d": int(plan.total_edges), "epochs": ep,
                         "rel_l2": float(np.linalg.norm(got - ref) / np.linalg.norm(ref)), "max_abs": float(np.abs(got - ref).max())})
        parity = {"against": "oracle/kernel_spec.explain_pruned_edges_sparse (fp64 edge-list specification)", "nodes": errs,
                  "rel_l2_max": max(e["rel_l2"] for e in errs), "seconds": time.perf_counter() - pt0,
                  "spec_seconds_per_epoch": spec_s / max(spec_ep, 1)}
    tp0 = time.perf_counter()
    eng.plan_nodes(nodes, 3, fetch=False)
    torch.cuda.synchronize()
    plan_s = time.perf_counter() - tp0
    _, total_n, total_e = eng._plan_sizes
    out_dev = torch.empty(total_e, dtype=torch.float32, device=c.dev)
    out_host = torch.empty(total_e, dtype=torch.float32).pin_memory()
    sampler = ClockSampler(c.local_rank)
    kms, wall = [], []
    l0 = 0
    for i in range(a.warmup + a.steps):
        if i == a.warmup:
            sampler.start()
            l0 = eng.launch_count()
        tw = time.perf_counter()
        eng.plan_nodes(nodes, 3, fetch=False)
        eng.explain_nodes_ptr(hp, _abi.GX_DEVICE, 0, out_dev.data_ptr())
        out_host.copy_(out_dev, non_blocking=False)      # masks delivered to the host (what explain_nodes returns)
        torch.cuda.synchronize()
        if i >= a.warmup:
            wall.append(time.perf_counter() - tw); kms.append(eng.last_explain_ms())
    sampler.end()
    clocks = sampler.stop()
    c5_launches = eng.launch_count() - l0
    if dump:
        write_outputs(dump, {"masks": out_host.numpy()})
    # top-k delivery instead of the full masks (the multi-GPU gather policy for this configuration: denoise_graph(threshold_num=20))
    td0 = time.perf_counter()
    thr, cnt, slots, vals = eng.denoise_topk(out_host.numpy(), 20)
    topk_s = time.perf_counter() - td0
    kern_s = float(np.mean(kms)) / 1e3
    algo = float(NUM_EPOCHS * (84.0 * total_e + 8.0 * d * total_n))          # SURVEY 8(d), no spill term
    peak, peak_src = _peak_hbm()
    mask = out_host.numpy()
    line = {
        "metric": METRIC, "value": K / kern_s, "unit": "nodes/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * kern_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[4]: BA(N=%d, m=%d) d=128 C=4, %d explained nodes per step, 3-hop, 100 epochs, streaming kernel (explain_gang.cu, automatic gang size)" % (N, m, K),
                   "sum_n": int(total_n), "sum_E_d": int(total_e), "init": "device Philox N(1,2/n)", "graph_gen_s": gen_s, "first_plan_s": plan_s,
                   "l2": "working set (%.1f GB of per-task state) exceeds L2" % (total_e * 4 * 3 / 1e9)},
        "e2e": {"value": K / float(np.mean(wall)), "unit": "nodes/s", "ms_per_step": 1e3 * float(np.mean(wall)),
                "h2d_bytes_per_step": int(K * 4), "d2h_bytes_per_step": int(total_e * 4)},
        "gpu_launches": int(c5_launches), "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": algo / kern_s / 1e9, "peak": peak, "unit": "GB/s", "frac": algo / kern_s / 1e9 / peak, "traffic": _c5_traffic(K),
                     "peak_source": peak_src, "kernel": "explain_gang_kernel (gangs of co-resident CTAs per node, TMA-staged 3xTF32 mma.sync feature passes) + outer_pairs_kernel", "algorithmic_bytes_per_step": algo, "sm": _sm_metrics("c5"),
                     "note": "algorithmic bytes = SURVEY 8(d) fused lower bound of the UNPRUNED algorithm (84*E_d + 8*n*d per node-epoch); the kernel "
                             "prunes to the receptive field and runs outermost pairs as register recurrences, so it can move fewer bytes than that"},
        # the reference itself cannot run this configuration (dense n x n float tensors: 40 GB per temporary at n = 100 000, 120 GB of
        # mask + Adam state per node); the CPU number is the edge-list restatement (oracle/kernel_spec.py, scipy sparse, fp64, one
        # core) timed on the parity node above and extrapolated to 99 updates -- SURVEY 8(d) d-cpu asks for exactly this
        "cpu_baseline": ({"value": 1.0 / (parity["spec_seconds_per_epoch"] * (NUM_EPOCHS - 1)), "unit": "nodes/s", "cores": 1, "kind": "port",
                          "sample": "oracle/kernel_spec.explain_pruned_edges_sparse (edge-list restatement, fp64, 1 core) on %d node(s) x %d updates, extrapolated to 99 updates; the reference's dense path needs 40 GB per temporary at this n" % (len(parity["nodes"]), sum(e["epochs"] - 1 for e in parity["nodes"]))}
                         if parity else {"value": None, "unit": "nodes/s", "cores": 0, "kind": "port", "sample": "--c5-parity 0: not timed"}),
        "parity_at_scale": parity,
        "topk_delivery": {"threshold_num": 20, "seconds": topk_s, "bytes": int(cnt.sum()) * 8, "note": "gx_denoise_topk: what a multi-GPU run gathers instead of %.2f GB of full masks" % (total_e * 4 / 1e9)},
        "mask_checksum": {"mean": float(mask.mean()), "min": float(mask.min()), "max": float(mask.max()), "finite": bool(np.isfinite(mask).all())},
    }
    eng.close()
    return line


def main_reference_graphs(a):
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    adj, feat, label, W = make_graph_batch()
    G = adj.shape[0]
    procs = a.cpu_procs or min(cores, 64)
    sample = [int(x) for x in np.linspace(0, G - 1, max(2 * procs, 16)).round()]
    jobs = [(adj[g], feat[g], label[g], W, 100 + g) for g in sample]
    with mp.get_context("fork").Pool(procs) as pool:
        pool.map(_cpu_graph_one, jobs[:procs], chunksize=1)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            pool.map(_cpu_graph_one, jobs, chunksize=1)
        dt = (time.perf_counter() - t0) / a.steps
    v = len(sample) / dt
    print(json.dumps({"impl": "reference", "metric": "explained-graphs/sec (100 mask-opt epochs each)", "value": v, "unit": "graphs/s",
                      "n_gpus": 1, "steps": a.steps, "warmup": 0, "ms_per_step": 1000 * dt, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "configs[3] stand-in: %d padded graphs (max_nodes 100, d=14), graph-level mask" % G,
                                 "sample": "%d graphs, %d single-thread worker processes" % (len(sample), procs)},
                      "cpu_baseline": {"value": v, "unit": "graphs/s", "cores": procs, "kind": "port", "sample": "%d evenly spaced graphs x 100 epochs, %d single-thread worker processes, %.1f s" % (len(sample), procs, dt)},
                      "e2e": {"value": v, "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_workloads (syn4 / graphs / c5) in the default N=1 line")
    ap.add_argument("--workload", default="syn1", choices=["syn1", "syn4", "graphs", "c5"], help="syn1 = BASELINE configs[1] (default, the contract line); syn4 = configs[2]; graphs = configs[3] stand-in; c5 = configs[4] (streaming kernel)")
    ap.add_argument("--c5-n", type=int, default=100000)
    ap.add_argument("--c5-m", type=int, default=32)
    ap.add_argument("--c5-nodes", type=int, default=148, help="explained nodes per step of the c5 workload")
    ap.add_argument("--c5-parity", type=int, default=1, help="nodes checked against the fp64 sparse specification at full scale (0 = skip)")
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of the CPU baseline (default min(cores,64))")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: after the timed steps, write what the last one computed (masks, subgraph description) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.impl == "reference":
        if a.workload == "graphs":
            main_reference_graphs(a)
        else:
            main_reference(a)
    elif a.workload == "graphs":
        c = gpu_ctx(a)
        print(json.dumps(bench_graphs(a, c, with_cpu=not a.no_cpu, dump=a.dump_outputs)), flush=True)
    elif a.workload == "c5":
        c = gpu_ctx(a)
        print(json.dumps(bench_c5(a, c, dump=a.dump_outputs)), flush=True)
    else:
        main_ours(a)
