/* gnnx.h -- C ABI of libgnnx.so, the B200-native GNNExplainer mask-optimisation engine.
 *
 * The reference (RexYing/gnn-model-explainer) has NO FFI/plugin interface: its boundary for this
 * hot path is a Python surface.  Every entry point below therefore cites the reference Python
 * function it replaces; INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - C linkage, no exceptions cross the ABI.  Every call returns GX_OK (0) or a negative
 *     gx_status; gx_last_error() returns a thread-local human-readable message.
 *   - The caller owns every input/output buffer.  The library owns only the opaque gx_handle
 *     (device copies of model/graph, the extraction plan and its workspace).
 *   - Pointers are HOST pointers unless the parameter is documented "device" or the call takes a
 *     gx_memspace.  No torch types appear in any signature.
 *   - One handle per host thread / per GPU.  Calls on one handle must not overlap.
 *   - All work is issued on the stream set with gx_set_stream (default: the legacy default
 *     stream); calls that return results to host memory synchronise that stream before returning.
 *   - There is NO CPU fallback: without a CUDA device gx_create fails with GX_ERR_CUDA.
 */
#ifndef GNNX_H_
#define GNNX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GX_VERSION 211

typedef struct gx_handle gx_handle;

typedef enum gx_status {
  GX_OK = 0,
  GX_ERR_INVALID = -1,     /* bad argument / call order                         */
  GX_ERR_CUDA = -2,        /* CUDA runtime error (message has the cudaError)    */
  GX_ERR_UNSUPPORTED = -3, /* valid in the reference but not built here (yet)   */
  GX_ERR_NODE = -4,        /* a node is not inside its own k-hop neighbourhood  */
  GX_ERR_NOMEM = -5
} gx_status;

typedef enum gx_memspace { GX_HOST = 0, GX_DEVICE = 1 } gx_memspace;

/* Model dimensions: GcnEncoderNode/GcnEncoderGraph(input_dim, hidden_dim, embedding_dim, label_dim,
 * num_layers, bn=..., args.bias) -- reference models.py:84-97,332-345. */
typedef struct gx_model_dims {
  int32_t input_dim;   /* d                                             */
  int32_t hidden_dim;  /* output width of conv_first / conv_block[*]    */
  int32_t embed_dim;   /* output width of conv_last                     */
  int32_t num_classes; /* label_dim                                     */
  int32_t num_layers;  /* num_gc_layers: 2, 3 (reference default) or 4    */
  int32_t flags;       /* GX_MODEL_* bits                               */
} gx_model_dims;
#define GX_MODEL_BN 1u /* args.bn (models.py:222-228): per-node standardisation after every hidden ReLU.  num_layers != 3, bn or a
                        * hidden / output width of 33..128 select the model-variant kernel (node mode, mask optimisation only: no
                        * trace / optimiser state / grad) */

/* Optimisation hyper-parameters: explainer_main.py:143-167 defaults + ExplainModule.coeffs
 * (explainer/explain.py:624-631) + torch.optim.Adam defaults (utils/train_utils.py:10). */
typedef struct gx_hparams {
  int32_t num_epochs;    /* args.num_epochs, default 100                                  */
  float lr;              /* args.lr, default 0.1                                          */
  float beta1, beta2;    /* 0.9, 0.999                                                    */
  float eps;             /* 1e-8                                                          */
  float coef_size;       /* coeffs["size"] = 0.005                                        */
  float coef_feat_size;  /* coeffs["feat_size"] = 1.0                                     */
  float coef_ent;        /* coeffs["ent"] = 1.0                                           */
  float coef_lap;        /* coeffs["lap"] = 1.0 (forced to 0 in graph mode)               */
  int32_t mask_act;      /* 0 = sigmoid (args.mask_act default); others GX_ERR_UNSUPPORTED */
  int32_t mask_bias;     /* args.mask_bias: accepted; a no-op exactly as in the reference (bias stays 0: ReLU6'(0)=0) */
  int32_t init;          /* GX_INIT_*                                                     */
  uint64_t seed;         /* GX_INIT_PHILOX: stream seed                                   */
  int32_t start_step;    /* GX_INIT_STATE: Adam steps already taken (torch's state["step"]); else 0 */
  int32_t opt;           /* GX_OPT_*: args.opt (utils/train_utils.py:9-16); default adam                       */
  int32_t opt_scheduler; /* GX_SCHED_*: args.opt_scheduler (train_utils.py:17-23); stepped once per epoch (explain.py:145-146) */
  int32_t opt_decay_step;/* StepLR step_size                                                          */
  float opt_decay_rate;  /* StepLR gamma                                                              */
  int32_t opt_restart;   /* CosineAnnealingLR T_max                                                   */
} gx_hparams;
#define GX_OPT_ADAM 0
#define GX_OPT_SGD 1      /* torch.optim.SGD(momentum=0.95)                                    */
#define GX_OPT_RMSPROP 2  /* torch.optim.RMSprop defaults (alpha 0.99, eps 1e-8)              */
#define GX_OPT_ADAGRAD 3  /* torch.optim.Adagrad defaults (eps 1e-10)                          */
#define GX_SCHED_NONE 0
#define GX_SCHED_STEP 1
#define GX_SCHED_COS 2    /* schedulers work with every kernel; optimisers other than Adam run node tasks in the variant kernel */
#define GX_INIT_M0 0     /* caller supplies M0 at the directed-edge entries (parity with torch's RNG draw) */
#define GX_INIT_PHILOX 1 /* N(1, 2/n) drawn on device, counter = (seed, node, edge slot)                  */
#define GX_INIT_STATE 2  /* resume / teacher forcing: mask, Adam moments and feature-mask state supplied (gx_explain_io) */

/* Per-epoch log of the optimisation, one row per epoch of this call (explain.py:137-159: the values print_training
 * prints, plus the terms they are made of).  "edges" = restricted to the E_d directed-edge entries of the mask; the
 * reference's printed loss also sums size/entropy over the n^2 - E_d entries that never reach the result:
 * gx_offedge_regularisers returns that remainder so that loss = GX_TR_LOSS_EDGES + c_size*S_off + c_ent*H_off/n^2. */
#define GX_TRACE_COLS 8
#define GX_TR_LOSS_EDGES 0 /* pred + size(edges) + lap + ent(edges) + feat_size  (explain.py:808)      */
#define GX_TR_PRED 1       /* -log softmax(logits[node])[label]                  (explain.py:750-753)  */
#define GX_TR_SIZE 2       /* coef_size * sum over edges of sigmoid(M)           (explain.py:755-760)  */
#define GX_TR_ENT 3        /* coef_ent * sum over edges of H(sigmoid(M)) / n^2   (explain.py:769-770)  */
#define GX_TR_LAP 4        /* coef_lap * y^T (D - A_m) y / n^2                   (explain.py:780-793)  */
#define GX_TR_FEAT 5       /* coef_feat_size * mean sigmoid(feat_mask)           (explain.py:763-766)  */
#define GX_TR_DENSITY 6    /* mask_density(): sum(A_m) / sum(A) AFTER the epoch's Adam step (explain.py:148,680-683) */
#define GX_TR_PGT 7        /* softmax probability of the label                                          */

/* Optional inputs / outputs of gx_explain_nodes_ex and gx_explain_graphs_ex (all in the call's gx_memspace; NULL = unused).
 * Optimiser state lives at the same slots as m0_edges / edge_mask; feature-mask state is [count][3][input_dim] =
 * (feat_mask, exp_avg, exp_avg_sq).  State out = the state edge_mask was built from, i.e. after num_epochs-1 updates:
 * a run of E epochs equals a run of E1 epochs followed by GX_INIT_STATE with start_step = E1-1 and num_epochs = E-E1+1,
 * bit for bit (tests/test_gpu_state.py). */
typedef struct gx_explain_io {
  const float* m0_edges;      /* [total_edges] GX_INIT_M0: M0; GX_INIT_STATE: the mask parameter M              */
  float* edge_mask;           /* [total_edges] out, required: masked_adj at the sub_col slots                   */
  float* feat_mask;           /* [count*input_dim] out: sigmoid(feat_mask)                                      */
  float* trace;               /* [count*num_epochs*GX_TRACE_COLS] out (ExplainModule.loss / mask_density, a12)  */
  float* trace_pred;          /* [count*num_epochs*num_classes] out: the softmax row print_training prints (explain.py:714); needs trace */
  const float* adam_m_in;     /* [total_edges] GX_INIT_STATE: exp_avg of M                                      */
  const float* adam_v_in;     /* [total_edges] GX_INIT_STATE: exp_avg_sq of M                                   */
  const float* feat_state_in; /* [count*3*input_dim] GX_INIT_STATE                                              */
  float* mask_param_out;      /* [total_edges] out: M                                                            */
  float* adam_m_out;          /* [total_edges] out                                                               */
  float* adam_v_out;          /* [total_edges] out                                                               */
  float* feat_state_out;      /* [count*3*input_dim] out                                                         */
} gx_explain_io;

void gx_default_hparams(gx_hparams* hp);

const char* gx_last_error(void);
int gx_version(void);

/* Lifetime.  device = CUDA ordinal. */
int gx_create(int device, gx_handle** out);
int gx_destroy(gx_handle* h);
int gx_set_stream(gx_handle* h, void* cuda_stream);
int gx_sync(gx_handle* h);

/* Frozen model being explained.  Replaces the torch module the reference passes to
 * Explainer(model=...) (explain.py:43-57); tensors are the state_dict entries
 * conv_first.weight (d,h) / conv_block.0.weight (h,h) / conv_last.weight (h,e) as row-major
 * (in,out) float32, their biases (NULL = --nobias), pred_model.weight (C, 2h+e) row-major and
 * pred_model.bias (C).  conv_w / conv_b are arrays of num_layers pointers. */
int gx_set_model(gx_handle* h, const gx_model_dims* dims, const float* const* conv_w,
                 const float* const* conv_b, const float* pred_w, const float* pred_b);

/* Graph of a node-classification task, replacing Explainer(adj, feat, label, pred) (explain.py:43-62):
 * CSR of the (B=1) adjacency with ascending columns per row (must be symmetric 0/1; self loops are
 * honoured by gx_plan_nodes' reachability and dropped from the explained edge set exactly like the
 * reference's diag_mask, explain.py:617,678), features (N,d) float32, label (N) and
 * pred_label = argmax(pred[0], axis=1) (N) (explain.py:105). */
int gx_set_graph_csr(gx_handle* h, int64_t num_nodes, const int32_t* rowptr, const int32_t* col,
                     const float* feat, int32_t feat_dim, const int32_t* label,
                     const int32_t* pred_label);

/* graph_utils.neighborhoods (utils/graph_utils.py:147-158) for a set of rows: writes row `nodes[t]`
 * of the dense 0/1 hop matrix into out[t*num_nodes .. ] (uint8).  Integer BFS on CSR; bit-exact. */
int gx_neighborhood_rows(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops,
                         uint8_t* out_rows);

/* Explainer.extract_neighborhood (explain.py:492-501) for a batch of nodes, on device.
 * Builds the extraction plan kept inside the handle and reports the packed sizes:
 *   total_nodes = sum_t n_t,  total_edges = sum_t E_t (directed entries of the induced sub-adjacency).
 * Fails with GX_ERR_NODE if some node is outside its own neighbourhood (isolated node / n_hops=1
 * without self loop: the reference then explains a wrong row or crashes, explain.py:496-501). */
int gx_plan_nodes(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops,
                  int64_t* total_nodes, int64_t* total_edges);

/* Copies the canonical (reference-ordered) description of the planned subgraphs to the host:
 *   node_off[count+1], edge_off[count+1]      packed offsets
 *   neighbors[total_nodes]                    ascending global ids           (explain.py:497)
 *   node_idx_new[count]                       rank of the node in its set    (explain.py:496)
 *   sub_rowptr[total_nodes+count]             per task n_t+1 entries, task-local, starting at 0
 *   sub_col[total_edges]                      local column ids, ascending per row: the row-major
 *                                             nonzero order of the reference's dense sub_adj
 * Any pointer may be NULL to skip that array. */
int gx_plan_fetch(gx_handle* h, int64_t* node_off, int64_t* edge_off, int32_t* neighbors,
                  int32_t* node_idx_new, int32_t* sub_rowptr, int32_t* sub_col);

/* The hot path: Explainer.explain's optimisation loop for every planned node
 * (explain.py:97-146,209-211; ExplainModule explain.py:583-808; models.py:58-80,230-267,363-376;
 * torch.optim.Adam), one persistent CTA per node, all epochs in one launch.
 *   m0_edges    [total_edges] float32 in `space`: M0[i,j] at the sub_col slots (GX_INIT_M0), or NULL
 *   edge_mask   [total_edges] float32 in `space`: returned masked_adj[i,j] at the same slots
 *   feat_mask   optional [count*input_dim] float32 in `space`: sigmoid(feat_mask) after the last
 *               observed update (not returned by the reference API; for tests), may be NULL */
int gx_explain_nodes(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_edges,
                     float* edge_mask, float* feat_mask);

/* Same, with the optional trace / optimiser-state buffers of gx_explain_io (io->edge_mask required). */
int gx_explain_nodes_ex(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io);

/* Regulariser sums over the mask entries OUTSIDE the sub-adjacency (non-edges and the diagonal), which the reference's
 * printed loss includes (explain.py:755-770 sum over all n^2 entries) although they never influence the result: every such
 * entry follows a private scalar Adam recurrence driven by size + entropy only.  m0_dense = the full (n_t, n_t) M0 of every
 * planned node, task after task (sum_t n_t^2 floats, `space`); out[count*num_epochs*2] = per epoch (sum sigmoid(M),
 * sum H(sigmoid(M))) over those entries, in double.  Only needed to reproduce the reference's printed loss value. */
int gx_offedge_regularisers(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_dense, double* out);

/* The gradient baseline, Explainer.explain(..., model="grad") (explain.py:125-133) with ExplainModule.adj_feat_grad
 * (explain.py:717-738), for every planned node: one forward of the frozen model on the unmasked sub-adjacency and
 * features, loss = -log softmax(logits[node])[predicted label of the node], one backward to the adjacency;
 *   edge_mask [total_edges] float32 in `space`: sigmoid(|dL/dA_ij| + |dL/dA_ji|) at the sub_col slots. */
int gx_grad_nodes(gx_handle* h, gx_memspace space, float* edge_mask);

/* ---- graph-classification mode (Explainer(..., graph_mode=True), explain_graphs: explain.py:80-85,356-363) ----
 * Batch of padded graphs, replacing Explainer(adj (G,n,n), feat (G,n,d), label (G)): block CSR over
 * G*max_nodes rows (rowptr[G*max_nodes+1] with global edge offsets, col = node id inside its graph,
 * ascending per row, symmetric 0/1, no self loops), features (G*max_nodes, d), one label per graph. */
int gx_set_graph_batch_csr(gx_handle* h, int32_t num_graphs, int32_t max_nodes, const int32_t* rowptr,
                           const int32_t* col, const float* feat, int32_t feat_dim, const int32_t* label);
/* Plans the graphs to explain; edge_off[count+1] (may be NULL) receives the packed slot offsets: the slots of
 * graph t are the entries of its adjacency in row-major order (its slice of the CSR).  Every model gx_set_model accepts is
 * accepted (num_layers 2..4, GX_MODEL_BN, widths up to 128, input_dim <= 128), and every graph up to max_nodes = 4096: the default
 * model (3 layers, no bn, widths <= 32) on a graph whose state fits 226 KB of shared memory runs in the tuned graph kernel, every
 * other graph in the graph-mode variant kernel (state in a per-CTA global slab). */
int gx_plan_graphs(gx_handle* h, const int32_t* graph_ids, int32_t count, int64_t* edge_off, int64_t* total_edges);
/* Explainer.explain(node_idx=0, graph_idx=g, graph_mode=True) for every planned graph (model =
 * GcnEncoderGraph: per-layer max-pool readout, models.py:269-316; lap_loss = 0, explain.py:787-788).
 * m0_edges / edge_mask: [total_edges] in `space`, as for gx_explain_nodes.  All four optimisers and both schedulers; with an
 * optimiser other than Adam the whole batch runs in the variant kernel.  A call in which any graph runs in the variant kernel builds
 * the mask optimisation only: a trace, GX_INIT_STATE or optimiser-state outputs return GX_ERR_UNSUPPORTED. */
int gx_explain_graphs(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_edges,
                      float* edge_mask, float* feat_mask);
int gx_explain_graphs_ex(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io);

/* Expands packed edge masks to the dense (n_t, n_t) float64 arrays Explainer.explain returns
 * (explain.py:209-221), task after task, into out (sum_t n_t^2 doubles, `space`). */
int gx_densify(gx_handle* h, gx_memspace space, const float* edge_mask, double* out);

/* The thresholding step of io_utils.denoise_graph(masked_adj, node_idx, threshold_num=k) (utils/io_utils.py:193-231; called on
 * every explained node by explain.py:238-288,308) on the packed masks of the planned nodes, on device: per node
 *   out_threshold[t] = the min(2k, #positive)-th largest positive mask value ("edges are repeated twice in adj"), +inf if none
 *   out_count[t]     = number of directed slots with value >= threshold (>= 2k when values tie at the threshold)
 *   out_slots[t*cap ..] = those slots (task-local indices into the node's sub_col / edge_mask slice), ascending, first `cap`
 *   out_vals[t*cap ..]  = their mask values (may be NULL)
 * This is also what a multi-GPU run gathers when the full masks are too large to gather (BASELINE configs[4]). */
int gx_denoise_topk(gx_handle* h, gx_memspace space, const float* edge_mask, int32_t threshold_num, int32_t cap,
                    float* out_threshold, int32_t* out_count, int32_t* out_slots, float* out_vals);

/* ---- multi-GPU: one process per GPU, explained nodes dealt across ranks, ONE all-gather of the packed masks (SURVEY 8e) ----
 * The reference's node loop (explain.py:225-236) is sequential and has no exchange step; results of different nodes never
 * interact, so the only collective is the final delivery.  NCCL is loaded at run time (dlopen libnccl.so.2).
 *   gx_comm_unique_id : rank 0 creates the 128-byte bootstrap id; the caller transports it to the other ranks
 *                       (torch.distributed broadcast, MPI, a file);
 *   gx_comm_init      : ncclCommInitRank on the handle's device; gx_comm_destroy releases it;
 *   gx_count_nodes    : |k-hop set| and directed sub-adjacency entries of each node WITHOUT building a plan -- every rank
 *                       calls it for the whole node list, so shard sizes and offsets are known everywhere with no metadata exchange;
 *   gx_allgather_masks: ONE ncclAllGather on the handle's stream; every rank contributes `slot_floats` floats (its
 *                       `local_floats` packed mask values, zero padded), gathered_dev receives world*slot_floats floats (device pointers);
 *   gx_unshard_masks  : scatters the gathered slots into the caller's global item order on device: item p (sizes[p] floats)
 *                       is read at gathered_dev[src_off[p]] and written at out_dev[dst_off[p]] (offset arrays are host pointers). */
int gx_comm_unique_id(char id[128]);
int gx_comm_init(gx_handle* h, int32_t world, int32_t rank, const char id[128]);
int gx_comm_destroy(gx_handle* h);
int gx_count_nodes(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops, int32_t* n_out, int32_t* e_out);
int gx_allgather_masks(gx_handle* h, const float* local_dev, int64_t local_floats, int64_t slot_floats, float* gathered_dev);
int gx_unshard_masks(gx_handle* h, const float* gathered_dev, int32_t items, const int64_t* src_off, const int64_t* dst_off,
                     const int32_t* sizes, float* out_dev);

/* GcnEncoderNode.forward on the uploaded graph (models.py:58-80,230-267,363-376): pred[num_nodes * num_classes] = the logits the
 * reference reads from its checkpoint (`cg["pred"]`, explainer_main.py:186-193) and hands to Explainer(pred=...).  Raw adjacency
 * (self loops included), no masks; every model gx_set_model accepts (2 / 3 / 4 layers, --bn). */
int gx_model_forward(gx_handle* h, gx_memspace space, float* pred);

/* Counters for bench.py: number of kernels this handle has launched so far, and the device time
 * (CUDA events on the handle's streams) of the explainer kernels of the last gx_explain_nodes call. */
int64_t gx_launch_count(gx_handle* h);
/* Measurement only (no counterpart in the reference, which explains one node at a time and has no scheduler).
 * gx_plan_class_counts: tasks of the current node plan per launch class -- counts[0..4] = shared-memory classes by footprint
 * (13 / 27 / 55 / 112 / 226 KB), counts[5] = streaming class, counts[6] = cluster class; smem_bytes (may be NULL) = largest per-CTA
 * shared-memory footprint of each class; *cluster_size = CTAs per task of the cluster class (1 = none). */
int gx_plan_class_counts(gx_handle* h, int32_t counts[7], int32_t smem_bytes[7], int32_t* cluster_size);
/* gx_last_class_ms: device timeline of the last gx_explain_nodes call -- per launch class (indices as above) the time its stream reached
 * the launch and the time its kernel finished, in ms after the call's first event; -1 for classes without tasks.  Synchronises like
 * gx_last_explain_ms.  (tools/cluster_study.py; this timeline found the carveout serialisation, profiles/r02cl_cluster_auto.md.) */
int gx_last_class_ms(gx_handle* h, float begin_ms[7], float end_ms[7]);
int gx_last_explain_ms(gx_handle* h, float* ms);

/* ---- test / measurement knobs (used by tests/ and tools/ only; they never change what the product computes by default) ----
 * gx_debug_force_stream: plan every task into the streaming kernel (explain_stream.cu) regardless of its size;
 * gx_debug_ieee_edge:    IEEE exp / division / sqrt in the edge phase instead of the ex2/rcp/rsqrt approximations;
 * gx_debug_set_dump:     device buffer (>= 4 MiB) receiving the shared-memory slab of the first task and phase timers;
 * gx_debug_set_gang:     CTAs per task of the streaming kernel explain_gang.cu (0 = automatic: the tasks in flight keep their
 *                        scattered state L2 resident; -1 = the first-generation kernel explain_stream.cu);
 * gx_debug_set_cluster:  thread-block cluster class of the shared-memory kernel.  cluster_size 1 = never (default: a task's masks do not
 *                        depend on the batch it is explained in, bit for bit); 0 = latency mode: when a batch leaves SMs idle (one
 *                        explain() call, a shard of a strong-scaled list) gx_plan_nodes runs its most expensive tasks on clusters of
 *                        2 / 4 CTAs (one syn1 hub node 2.85 -> 1.56 ms); 2 / 4 = every shared-memory task whose cost exceeds min_cost.
 *                        The gang size never changes a bit of the result (tests/test_gpu_stream.py); a cluster sums the per-warp
 *                        dL/dsF partials in another order, so it agrees with the single-CTA run to round-off
 *                        (tests/test_gpu_cluster.py).  Environment: GNNX_CLUSTER_SIZE. */
int gx_debug_set_gang(gx_handle* h, int ctas_per_task);
int gx_debug_set_cluster(gx_handle* h, int cluster_size, int64_t min_cost);
int gx_debug_force_stream(gx_handle* h, int on);
int gx_debug_ieee_edge(gx_handle* h, int on);
int gx_debug_set_dump(gx_handle* h, float* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* GNNX_H_ */
