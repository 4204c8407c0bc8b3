"""GPU (-m gpu), needs >= 2 devices: Explainer.explain_nodes sharded over 2 ranks (one process per GPU,
NCCL) with ONE all-gather of the packed masks must reproduce the 1-GPU result bit for bit."""
import os
import socket
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import conftest  # noqa: F401
    import torch.distributed as dist
    import util
    import gnnx
    import gnnx_oracle as O
    from gnnx.dist import explain_nodes_sharded
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    fx = util.load_fixture("syn1")
    args = types.SimpleNamespace(num_gc_layers=3, num_epochs=30, lr=0.1, opt="adam", opt_scheduler="none", mask_act="sigmoid",
                                 mask_bias=False, gpu=False, bias=True, method="base", dataset="syn1", bmname=None, hidden_dim=20,
                                 output_dim=20, name_suffix="", explainer_suffix="", logdir="/tmp/gnnx_dist_%d" % rank,
                                 gnnx_init="device", gnnx_seed=5)
    model = gnnx.models.GcnEncoderNode(10, 20, 20, 4, 3, bn=False, args=args)
    sd = {"conv_first.weight": fx.weights["W1"], "conv_first.bias": fx.weights["b1"], "conv_block.0.weight": fx.weights["W2"],
          "conv_block.0.bias": fx.weights["b2"], "conv_last.weight": fx.weights["W3"], "conv_last.bias": fx.weights["b3"],
          "pred_model.weight": fx.weights["Wp"], "pred_model.bias": fx.weights["bp"]}
    model.load_state_dict({k: torch.tensor(v) for k, v in sd.items()})
    A = O.dense_from_csr(fx.rowptr, fx.col)
    ex = gnnx.Explainer(model=model, adj=A[None], feat=fx.feat[None], label=fx.label[None], pred=fx.pred[None],
                        train_idx=[], args=args, writer=None, print_training=False, graph_idx=-1, device=rank)
    nodes = np.arange(0, 700, 3)
    values, offsets, _ = explain_nodes_sharded(ex, nodes)                 # gx_allgather_masks: the library's own NCCL communicator
    v2, o2, _ = explain_nodes_sharded(ex, nodes, use_engine_comm=False)   # torch.distributed's NCCL, same layout
    assert torch.equal(values, v2) and np.array_equal(offsets, o2)
    if rank == 0:
        plan, full = ex.explain_nodes_packed(nodes)      # the same list on one GPU
        q.put((values.cpu().numpy(), np.asarray(offsets), full, plan.edge_off.copy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_explain_matches_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    values, offsets, full, edge_off = q.get(timeout=300)
    [p.join(120) for p in procs]
    assert np.array_equal(offsets, edge_off)
    assert np.array_equal(values, full), "sharded result differs from the single-GPU result"
