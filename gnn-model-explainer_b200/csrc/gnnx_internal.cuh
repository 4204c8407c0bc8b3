// gnnx_internal.cuh -- structures shared by the plan (k-hop extraction) kernels, the persistent
// explainer kernel and the C-ABI host code.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gnnx.h"

#define GX_MAX_LEVELS 8  // n_hops <= 7
#define GX_NONE16 0xFFFFu
#define GX_MAX_LAYERS 4  // num_gc_layers of a model variant (explain_var.cu); the tuned kernels build the reference default 3
#define GX_MAX_GANG 160   // CTAs that may share one task in explain_gang.cu (<= number of SMs)
#define GX_WP_SMEM_MAX 2048  // floats: pred_model (C x (2h+e) + C) is kept in shared memory up to this size

// One explained node ("task").  Counts are produced by khop_count_kernel, offsets by the host
// prefix sums, the packed arrays by khop_fill_kernel.
struct GxTask {
  int32_t node;     // global node id
  int32_t n;        // |k-hop set|
  int32_t e_d;      // directed entries of the induced sub-adjacency (self loops dropped)
  int32_t npairs;   // e_d / 2 undirected edges
  int32_t npairs_in;  // pairs with at least one endpoint in a row the forward computes (< n2): listed first
  int32_t idx_new;  // rank of `node` among its ascending neighbours (explain.py:496)
  int32_t gt_label; // label[node]
  int32_t n1, n2;   // level-order prefix sizes: |dist<=L-2|, |dist<=L-1| for L=3 -> |dist<=1|, |dist<=2|
  int32_t e1;       // directed entries whose source row is < n2 (what the forward ever gathers)
  int32_t status;   // 0 ok; 1 node not inside its own neighbourhood
  int32_t n_norm;   // the n of the reference's dense tensors (1/n^2 factors, M0 std): n in node mode, max_nodes in graph mode
  int32_t flags;    // graph mode: bit 0 = some row of the padded graph has no edge (its constant embedding joins the max-pool)
  int32_t cum[GX_MAX_LEVELS + 1];  // cum[t] = #nodes with dist <= t (dist measured from `node`)
  int32_t smem_bytes;              // shared-memory footprint of this task in the explainer kernel
  int64_t node_off;  // into nbrs / lo2gid
  int64_t rp_off;    // into sub_rowptr / irowptr (= node_off + task index: n+1 entries per task)
  int64_t edge_off;  // into sub_col / icol / m0 / edge_mask
  int64_t pair_off;  // into the pair arrays
};

// Device-resident plan arrays (all int32).
struct GxPlanArrays {
  GxTask* tasks;
  int32_t* nbrs;        // [total_n] ascending global ids (canonical order)
  int32_t* lo2gid;      // [total_n] global id of the node with level-order id i
  int32_t* sub_rowptr;  // [total_n + count] canonical CSR, task-local
  int32_t* sub_col;     // [total_e]
  int32_t* irowptr;     // [total_n + count] level-order CSR, task-local
  int32_t* icol;        // [total_e] level-order ids; per row partitioned by level of the neighbour
  int32_t* cs2is;       // [total_e] canonical slot -> internal slot (task-local)
  int32_t* is2cs;       // [total_e] internal slot -> canonical slot
  int32_t* pair_i;      // [total_e/2] i < j, level-order ids
  int32_t* pair_j;
  int32_t* pair_pij;    // position of j in internal row i (absolute, task-local)
  int32_t* pair_pji;
  int32_t* pair_oij;    // canonical edge slot of (i,j) (task-local index into the edge arrays)
  int32_t* pair_oji;
};

struct GxGraphDev {
  int64_t N;
  int32_t nnz;
  const int32_t* rowptr;
  const int32_t* col;
  const float* feat;  // [N*d]
  int32_t d;
  const int32_t* label;
  const int32_t* pred_label;
};

struct GxModelDev {
  int32_t d, hid, emb, C, L;
  int32_t bn;          // --bn: per-node standardisation after every hidden ReLU (models.py:222-228)
  int32_t variant;     // 1: num_layers != 3 or bn -> every task runs in explain_var.cu with the UNPADDED widths hid / emb
  const float* W[GX_MAX_LAYERS];   // row-major (in,out)
  const float* Wt[GX_MAX_LAYERS];  // row-major (out,in) (default model only)
  const float* b[GX_MAX_LAYERS];   // never NULL on device (zeros when --nobias)
  const float* Wp;     // (C, 2*hid+emb)
  const float* bp;
};

struct GxHparamsDev {
  int32_t iters;     // forward/backward/update iterations executed: num_epochs - 1 (the last epoch's backward is unobservable), num_epochs when a trace is requested
  int32_t out_iter;  // the mask (and the optimiser state) is emitted after this many updates: num_epochs - 1
  float one_minus_b1, b2, one_minus_b2, eps;
  float c_size, c_feat_size, c_ent, c_lap;
  const float2* adam_tab;  // [iters] Adam: (step_size_t = lr_t/(1-b1^t), sqrt(1-b2^t)) for t = start_step + 1 .., computed in double on the host; other optimisers: (lr_t, 0).  lr_t follows the scheduler
  int32_t init;
  int32_t flags;  // GX_HP_* bits
  int32_t opt;    // GX_OPT_*; the tuned kernels build Adam only (others: explain_var.cu + outer_pairs_kernel)
  int32_t mode;   // 0: mask optimisation; 1: gradient baseline (explain(model="grad")): one forward/backward on the unmasked subgraph
  uint64_t seed;
};

#define GX_HP_IEEE_EDGE 1  // edge phase with IEEE exp/div/sqrt instead of the hardware approximations (test knob)

// Optional trace / optimiser-state buffers of gx_explain_io (device pointers, nullptr = unused).
struct GxExtra {
  float* trace;        // [count][epochs][GX_TRACE_COLS]: the explainer kernels write raw per-epoch terms, trace_finalize_kernel assembles the columns
  float* trace_pred;   // [count][epochs][C]
  double* tr_outer;    // [count][epochs][4]: (sum S, sum H(S), sum a (y_i-y_j)^2, sum 2a after the step) over the outer pairs
  int32_t epochs;      // trace rows per task (= num_epochs of the call)
  const float* adam_m_in; const float* adam_v_in; const float* feat_state_in;
  float* mask_param_out; float* adam_m_out; float* adam_v_out; float* feat_state_out;
};

// ---------------------------------------------------------------------------------------------
// Shared-memory layout of one task in the explainer kernel.  Computed identically on host
// (classification of tasks into launch classes) and device (carve-up).
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline int gx_round_up(int x, int m) { return (x + m - 1) / m * m; }

struct GxLayout {
  // float arrays (offsets in 4-byte words)
  int X, U, Yh1, q1, Yh2, q2, dZ2, a, y, W1s, W1t, W2s, W2t, W3s, bs, sF, F, mF, vF, gFp, zs, dE, dZ3, logit, Wp;
  // index arrays (offsets in 4-byte words; element type IdxT)
  int icol, irp, pi, pj, ppij, ppji, llist, cnt1, llistB;
  int total_words;
  int dp;
};

// Shared-memory footprint of one task.  np_in = pairs with an endpoint in rows < n2 (their indices live in
// shared memory, their optimiser state in a per-CTA global slab that stays in L2); pairs between two
// outermost nodes never touch the forward and are optimised by a separate elementwise kernel.
// idx_bytes = sizeof(IdxT) (2 or 4).  hid/emb must be multiples of 4.
__host__ __device__ inline GxLayout gx_make_layout(int n, int n1, int n2, int e1, int np_in, int d,
                                                   int hid, int emb, int C, int nwarps,
                                                   int idx_bytes, int cs = 1) {
  GxLayout L;
  const int dp = gx_round_up(d, 4);
  L.dp = dp;
  int o = 0;
  auto takef = [&](int words) { int r = o; o += gx_round_up(words, 4); return r; };
  auto takei = [&](int elems) { int r = o; o += gx_round_up((elems * idx_bytes + 3) / 4, 4); return r; };
  L.X = takef(n * dp);
  L.U = takef(n2 * dp);      // A_m X in the forward; overwritten row by row with dZ1 (.) sF in the backward
  L.Yh1 = takef(n2 * hid);
  L.q1 = takef(n2);
  L.Yh2 = takef(n1 * hid);
  L.q2 = takef(n1);
  L.dZ2 = takef(n1 * hid);
  L.a = takef(e1);
  L.y = takef(n);            // float(pred_label) per node (Laplacian regulariser)
  L.W1s = takef(dp * hid);   // [dp][hid]   rows >= d are zero
  L.W1t = takef(hid * dp);   // [hid][dp]   transposed
  L.W2s = takef(hid * hid);
  L.W2t = takef(hid * hid);
  L.W3s = takef(hid * emb);
  L.bs = takef(2 * hid + emb);
  L.sF = takef(dp);
  L.F = takef(dp);
  L.mF = takef(dp);
  L.vF = takef(dp);
  L.gFp = takef(nwarps * cs * dp);   // per-warp dL/dsF partials of every CTA of the cluster (cs = cluster size)
  L.zs = takef(nwarps * 128);
  L.dE = takef(2 * hid);
  L.dZ3 = takef(hid);
  L.logit = takef(C < 32 ? 32 : C);
  L.Wp = takef(C * (2 * hid + emb + 1) <= GX_WP_SMEM_MAX ? C * (2 * hid + emb + 1) : 0);  // pred_model weights + bias when small
  L.icol = takei(e1);
  L.irp = takei(n2 + 1);
  L.pi = takei(np_in);
  L.pj = takei(np_in);
  L.ppij = takei(np_in);
  L.ppji = takei(np_in);
  L.llist = takei(n2);
  L.cnt1 = takei(n2);        // per row: number of leading columns < n1 (the only ones that carry dZ2)
  L.llistB = takei(n2);      // rows whose < n1 prefix is long (split across a whole warp in the backward)
  L.total_words = o;
  return L;
}

// Global-memory slab of one task in the streaming kernel (explain_stream.cu: tasks whose state does not fit
// shared memory).  Offsets in 4-byte words; the CSR / pair index arrays are read straight from the plan.
struct GxStreamLayout {
  int64_t a, gE, P, dP, Yh1, q1, dY1, Yh2, q2, dZ2, lapg, cnt1, cnt2, gFp, gFb, longlist, trw, xlo;
  int64_t total_words;
  int dp;
};
__host__ __device__ inline GxStreamLayout gx_make_stream_layout(int n, int n1, int n2, int e_d, int np_in, int d, int hid, int nwarps) {
  GxStreamLayout L;
  const int dp = gx_round_up(d, 4);
  L.dp = dp;
  int64_t o = 0;
  auto take = [&](int64_t words) { int64_t r = o; o += (words + 3) / 4 * 4; return r; };
  L.a = take(e_d);                     // masked-adjacency value of every internal slot (rows >= n2: only their < n2 prefix is live)
  L.gE = take(e_d);                    // layer-1 edge-gradient dot <dY1[col], P[row]> of every live slot (0 elsewhere)
  L.P = take((int64_t)n * hid);        // (X . sF) W1 of every node
  L.dP = take((int64_t)n * hid);       // A_m^T dY1 of every node
  L.Yh1 = take((int64_t)n2 * hid); L.q1 = take(n2); L.dY1 = take((int64_t)n2 * hid);
  L.Yh2 = take((int64_t)n1 * hid); L.q2 = take(n1); L.dZ2 = take((int64_t)n1 * hid);
  L.lapg = take(np_in);               // per inner pair: its (epoch-invariant) Laplacian-regulariser gradient
  L.cnt1 = take(n2);                   // per row < n2: leading columns < n1
  L.cnt2 = take(n);                    // per row: leading columns < n2
  L.gFp = take((int64_t)nwarps * dp);
  // explain_gang.cu: dL/dsF partials of the 128-node blocks, rows sliced over a whole CTA, per-warp trace partials of a gang
  L.gFb = take((int64_t)((n + 127) / 128) * dp);
  L.longlist = take(n);
  L.trw = take(GX_MAX_GANG * 32 * 4);
  L.xlo = take((int64_t)(n + 16) * (gx_round_up(d, 8) + 4));   // the task's feature rows in level order, padded to the shared-memory tile pitch
  L.total_words = o;
  return L;
}

// Global-memory slab of one task in the model-variant kernel (explain_var.cu); every hidden-width array has row stride 32.
struct GxVarLayout {
  int64_t a, U, dZ1, lapg, Yh, H, dZ, q, istd;
  int64_t total_words;
};
__host__ __device__ inline GxVarLayout gx_make_var_layout(int n, int n2, int e1, int np_in, int d, int L, int vw = 32) {
  GxVarLayout Lo;
  const int dp = gx_round_up(d, 4);
  int64_t o = 0;
  auto take = [&](int64_t words) { int64_t r = o; o += (words + 3) / 4 * 4; return r; };
  (void)n;
  Lo.a = take(e1);                            // masked adjacency of the rows the forward visits (level-order rows < n2)
  Lo.U = take((int64_t)n2 * dp);              // A_m X
  Lo.dZ1 = take((int64_t)n2 * dp);            // dL/d(A_m X') (.) sigmoid(feat_mask)
  Lo.lapg = take(np_in);
  Lo.Yh = take((int64_t)L * n2 * vw);         // per layer: normalised pre-activations (row stride vw = 32 * ceil(width / 32))
  Lo.H = take((int64_t)L * n2 * vw);          // per layer: relu (+ standardisation) output = input of the next layer / the readout
  Lo.dZ = take((int64_t)(L - 1) * n2 * vw);   // layers 2..L: dL/d(A_m H_{l-1})
  Lo.q = take((int64_t)L * n2);
  Lo.istd = take((int64_t)L * n2);
  Lo.total_words = o;
  return Lo;
}

// Global-memory slab of one graph-mode task in explain_graph_var.cu (model variants, optimisers other than Adam, graphs beyond
// shared memory): every one of the `na` rows with an edge at every layer; hidden-width arrays have row stride vw = 32 * ceil(width / 32).
struct GxGraphVarLayout {
  int64_t a, U, dZ1, Yh, H, dZ, q, istd, P;
  int64_t total_words;
};
__host__ __device__ inline GxGraphVarLayout gx_make_graph_var_layout(int na, int e_d, int np, int d, int L, int vw) {
  GxGraphVarLayout Lo;
  const int dp = gx_round_up(d, 4);
  int64_t o = 0;
  auto take = [&](int64_t words) { int64_t r = o; o += (words + 3) / 4 * 4; return r; };
  Lo.a = take(e_d);                             // masked adjacency of every internal slot
  Lo.U = take((int64_t)na * dp);                // A_m X
  Lo.dZ1 = take((int64_t)na * dp);              // dL/d(A_m X') (.) sigmoid(feat_mask)
  Lo.Yh = take((int64_t)L * na * vw);           // per layer: normalised pre-activations
  Lo.H = take((int64_t)L * na * vw);            // per layer: relu (+ standardisation) output = input of the next layer / the max-pool
  Lo.dZ = take((int64_t)(L - 1) * na * vw);     // layers 2..L: dL/d(A_m H_{l-1})
  Lo.q = take((int64_t)L * na);
  Lo.istd = take((int64_t)L * na);
  Lo.P = take((int64_t)np * 8);                 // per undirected edge: (M, m, v, S) of both directions
  Lo.total_words = o;
  return Lo;
}

// Shared-memory footprint of one graph-mode task (all `na` rows with at least one edge are computed at every layer).
struct GxLayoutG {
  int X, U, Yh1, Yh2, Yh3, q, dZ2, dZ3, a, W1s, W1t, W2s, W2t, W3s, W3t, bs, cst, emb, dE, sF, F, mF, vF, gFp, zs, logit, Wp;
  int arg, icol, irp, pi, pj, ppij, ppji;
  int total_words;
  int dp;
};
__host__ __device__ inline GxLayoutG gx_make_layout_graph(int na, int e_d, int np, int d, int hid, int emb, int C, int nwarps) {
  GxLayoutG L;
  const int dp = gx_round_up(d, 4);
  L.dp = dp;
  int o = 0;
  auto takef = [&](int words) { int r = o; o += gx_round_up(words, 4); return r; };
  auto takei = [&](int elems) { int r = o; o += gx_round_up((elems * 2 + 3) / 4, 4); return r; };
  L.X = takef(na * dp); L.U = takef(na * dp);
  L.Yh1 = takef(na * hid); L.Yh2 = takef(na * hid); L.Yh3 = takef(na * emb);
  L.q = takef(3 * na);
  L.dZ2 = takef(na * hid); L.dZ3 = takef(na * hid);
  L.a = takef(e_d);
  L.W1s = takef(dp * hid); L.W1t = takef(hid * dp); L.W2s = takef(hid * hid); L.W2t = takef(hid * hid);
  L.W3s = takef(hid * emb); L.W3t = takef(emb * hid);
  L.bs = takef(2 * hid + emb);
  L.cst = takef(2 * hid + emb);   // embedding of an edge-less row: relu(normalize(b_l)) / normalize(b_3)
  L.emb = takef(2 * hid + emb);
  L.dE = takef(2 * hid + emb);
  L.sF = takef(dp); L.F = takef(dp); L.mF = takef(dp); L.vF = takef(dp);
  L.gFp = takef(nwarps * dp);
  L.zs = takef(nwarps * 128);
  L.logit = takef(C < 32 ? 32 : C);
  L.Wp = takef(C * (2 * hid + emb + 1) <= GX_WP_SMEM_MAX ? C * (2 * hid + emb + 1) : 0);
  L.arg = takef(2 * hid + emb);   // int: arg-max row of every pooled feature (-1: the edge-less constant)
  L.icol = takei(e_d); L.irp = takei(na + 1);
  L.pi = takei(np); L.pj = takei(np); L.ppij = takei(np); L.ppji = takei(np);
  L.total_words = o;
  return L;
}

// ---------------------------------------------------------------------------------------------
#define GX_CUDA_CHECK(expr)                                                          \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) {                                                         \
      gx_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                   __LINE__);                                                        \
      return GX_ERR_CUDA;                                                            \
    }                                                                                \
  } while (0)

void gx_set_error(const char* fmt, ...);

// kernel launchers (defined in khop.cu / explain_node.cu)
struct GxSlotWs {
  uint32_t* bm;     // [slots * W]   membership bitmap (must be all-zero between tasks)
  int32_t* wpref;   // [slots * (W+1)]
  uint8_t* dist;    // [slots * N]
  int32_t* q;       // [slots * (N+1)]
  int32_t* loc;     // [slots * N]  level-order id by canonical id
  int32_t* cof;     // [slots * N]  canonical id by level-order id
  int32_t* pbase;   // [slots * (N+1)]
  int32_t W;        // words per bitmap
  int32_t slots;
};

cudaError_t gx_launch_khop_count(const GxGraphDev& g, const int32_t* nodes_dev, int count, int k,
                                 int row_lvl, GxSlotWs ws, GxTask* tasks, cudaStream_t s);
cudaError_t gx_launch_khop_fill(const GxGraphDev& g, int count, int k, GxSlotWs ws, GxPlanArrays plan,
                                cudaStream_t s);
cudaError_t gx_launch_hop_rows(const GxGraphDev& g, const int32_t* nodes_dev, int count, int k,
                               GxSlotWs ws, uint8_t* out_rows, cudaStream_t s);

struct GxExplainLaunch {
  const int32_t* order;  // [ntasks] task ids of this launch class, most expensive first
  int32_t ntasks;
  int32_t* counter;      // device work-queue counter (zeroed)
  int32_t smem_bytes;    // dynamic shared memory per CTA (shared-memory classes)
  int32_t threads;
  int32_t grid;
  int32_t cluster = 1;   // CTAs per task (thread-block cluster size): 1, 2 or 4 (explain_node.cu cluster class)
  int32_t gang = 1;      // explain_gang.cu: co-resident CTAs per task (grid = gangs * gang)
  unsigned long long* gang_bars = nullptr;   // [gangs] barrier counters, zeroed
  int32_t* gang_mail = nullptr;              // [gangs * 2]
  float* gws;            // per-CTA global slab of the streaming class
  int64_t gws_stride_words;
  float* pws;            // per-CTA pair-state slab: 8 floats per inner pair (M,m,v,S of both directions)
  int64_t pws_stride_words;
  float* dbg;            // debug dump buffer (device) or NULL
  GxExtra x;             // optional trace / optimiser-state buffers
};
cudaError_t gx_launch_explain(const GxExplainLaunch& cfg, const GxGraphDev& g, const GxModelDev& m,
                              const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0,
                              float* out_mask, float* out_feat, cudaStream_t s);
cudaError_t gx_launch_explain_stream(const GxExplainLaunch& cfg, const GxGraphDev& g, const GxModelDev& m,
                                     const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0,
                                     float* out_mask, float* out_feat, cudaStream_t s);
cudaError_t gx_launch_explain_gang(const GxExplainLaunch& cfg, const GxGraphDev& g, const GxModelDev& m,
                                   const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0,
                                   float* out_mask, float* out_feat, cudaStream_t s);
int gx_gang_smem_bytes(int d, int hid, int C);
cudaError_t gx_launch_explain_var(const GxExplainLaunch& cfg, const GxGraphDev& g, const GxModelDev& m,
                                  const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0,
                                  float* out_mask, float* out_feat, cudaStream_t s);
int gx_var_smem_bytes(int d, int L, int hid, int emb, int C);
int gx_var_row_stride(int hid, int emb);
cudaError_t gx_launch_model_forward(const GxGraphDev& g, const GxModelDev& m, float* H, float* pred, float* emb_out, cudaStream_t s);
constexpr int GX_STREAM_THREADS = 768;  // 24 warps: 80 registers per thread, 5 KB of cp.async staging per warp
int gx_explain_max_smem();
struct GxGraphBatchDev {
  int32_t num_graphs, max_nodes, d;
  const int32_t* rowptr;  // [G*max_nodes+1], global edge offsets
  const int32_t* col;     // node id within the graph
  const float* feat;      // [G*max_nodes*d]
  const int32_t* label;   // [G]
};
cudaError_t gx_launch_graph_plan(const GxGraphBatchDev& gb, int count, GxPlanArrays plan, cudaStream_t s);
cudaError_t gx_launch_explain_graphs(const GxExplainLaunch& cfg, const GxGraphBatchDev& gb, const GxModelDev& m,
                                     const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0, float* out_mask,
                                     float* out_feat, cudaStream_t s);
// explain_graph_var.cu: cfg.gws / gws_stride_words = the per-CTA slabs (gx_make_graph_var_layout of the launch's largest task)
cudaError_t gx_launch_explain_graph_var(const GxExplainLaunch& cfg, const GxGraphBatchDev& gb, const GxModelDev& m,
                                        const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0, float* out_mask,
                                        float* out_feat, cudaStream_t s);
int gx_graph_var_smem_bytes(int d, int L, int hid, int emb, int C);
int gx_graph_var_row_stride(int hid, int emb);
cudaError_t gx_launch_outer_pairs(const GxHparamsDev& hp, const GxGraphDev& g, const GxPlanArrays& plan, int count,
                                  const float* m0, float* out_mask, const GxExtra& x, cudaStream_t s);
cudaError_t gx_launch_denoise_topk(const GxPlanArrays& plan, int count, const float* edge_mask, int k2, int cap, float* out_thr,
                                   int32_t* out_cnt, int32_t* out_slots, float* out_vals, cudaStream_t s);
// comm.cu
struct GxComm;
int gx_comm_impl_unique_id(char* id128);
int gx_comm_impl_init(GxComm** out, int world, int rank, const char* id128);
void gx_comm_impl_destroy(GxComm* c);
int gx_comm_impl_world(const GxComm* c);
int gx_comm_impl_rank(const GxComm* c);
int gx_comm_impl_allgather(GxComm* c, const float* send, float* recv, size_t slot_floats, cudaStream_t s);
cudaError_t gx_launch_unshard(const float* gathered, int items, const int64_t* src, const int64_t* dst, const int32_t* sz, float* out, cudaStream_t s);
// trace.cu
cudaError_t gx_launch_trace_finalize(const GxHparamsDev& hp, const GxPlanArrays& plan, int count, const GxExtra& x, cudaStream_t s);
cudaError_t gx_launch_offedge(const GxHparamsDev& hp, const GxPlanArrays& plan, int count, int epochs, const int64_t* dense_off,
                              const float* m0_dense, double* out, cudaStream_t s);
cudaError_t gx_launch_densify(const GxPlanArrays& plan, int count, const int64_t* dense_off,
                              const float* edge_mask, double* out, cudaStream_t s);
