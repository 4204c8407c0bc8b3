// api.cu -- C-ABI host side of libgnnx.so (see include/gnnx.h for the contract and the reference
// call sites each entry point replaces).  Owns the handle: device copies of graph/model, the
// extraction plan, launch classes and workspaces.  No CPU compute path exists here: every
// algorithmic step is a kernel in khop.cu / explain_node.cu.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <numeric>
#include <vector>

#include "gnnx_internal.cuh"

static thread_local char g_err[1024] = "";

void gx_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct LaunchClass {
  int cap_bytes;  // dynamic shared memory per CTA (0: the streaming class, explain_stream.cu)
  int threads;
  int ctas_per_sm;
};
// k CTAs per SM share 227 KB (1 KB per CTA is reserved by the system)
static LaunchClass kClasses[] = {
    {13 * 1024, 128, 16}, {27 * 1024, 256, 8}, {55 * 1024, 256, 4},
    {112 * 1024, 512, 2}, {226 * 1024, 512, 1}, {0, 512, 1}, {226 * 1024, 512, 1}};
constexpr int kNumClasses = sizeof(kClasses) / sizeof(kClasses[0]);
constexpr int kStreamClass = 5;    // explain_stream.cu: state in a global slab
constexpr int kClusterClass = 6;   // explain_node.cu with a thread-block cluster per task: the most expensive shared-memory tasks
constexpr int kOneClass = 4, kTwoClass = 3;
constexpr int64_t kGraphVarSmallWords = 64 * 1024;   // explain_graph_var.cu: slabs up to 256 KB form the small-slab class
// Cluster class (gx_debug_set_cluster / GNNX_CLUSTER_SIZE): off by default, so that a task's masks never depend on the batch it is in;
// 0 = latency mode, gx_plan_nodes moves the most expensive tasks of a batch that leaves SMs idle to clusters; 2 / 4 = every task above
// cluster_cost.  A full 700-node batch is throughput bound: splitting its tasks only adds barrier and DSMEM overhead
// (profiles/r02a_bench_cluster_default_on_REJECTED.json), so the latency mode gives it none.
constexpr int kNumStreams = kNumClasses + 1;   // graph mode: 6 shared-memory classes + 2 classes of explain_graph_var.cu

}  // namespace

static inline double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static inline bool host_timing() { static const bool on = [] { const char* v = getenv("GNNX_HOST_TIMING"); return v && v[0] == '1'; }(); return on; }   // stderr breakdown of the host side (tools/)

struct AdamKey { float lr, b1, b2, decay_rate; int32_t opt, sched, decay_step, restart, iters, start; };

struct gx_handle {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t side[kNumStreams] = {};
  cudaEvent_t ev_fork = nullptr;
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
  bool timed = false;
  float* dbg = nullptr;
  bool ieee_edge = false;     // test knob (gx_debug_ieee_edge / GNNX_IEEE_EDGE): IEEE arithmetic in the edge phase
  int gang_override = 0;      // test knob (gx_debug_set_gang / GNNX_GANG): CTAs per task of explain_gang.cu, 0 = automatic, -1 = explain_stream.cu
  int cluster_size = 1;       // gx_debug_set_cluster / GNNX_CLUSTER_SIZE: 1 = never (default: results independent of the batch composition), 0 = automatic, 2 / 4 = forced
  int64_t cluster_cost = 0;
  int plan_cluster = 1;       // cluster size the current plan was classified with
  bool force_stream = false;  // test knob (gx_debug_force_stream / GNNX_FORCE_STREAM): every task goes to the streaming class
  cudaEvent_t ev_join[kNumStreams] = {}, ev_begin[kNumStreams] = {};
  bool class_used[kNumStreams] = {};   // launch classes of the last gx_explain_nodes call (gx_last_class_ms)
  int64_t launches = 0;

  // graph
  bool has_graph = false;
  GxGraphDev g{};
  DevBuf g_rowptr, g_col, g_feat, g_label, g_pred;
  // model
  bool has_model = false;
  GxModelDev m{};
  DevBuf m_buf;
  // plan
  bool has_plan = false;
  int count = 0, n_hops = 0;
  int64_t total_n = 0, total_e = 0;
  std::vector<GxTask> tasks;
  AdamKey adam_key{};
  bool adam_valid = false;
  bool tasks_fetched = true;   // false: idx_new of the host copy is stale (filled on the device by khop_fill, fetched by gx_plan_fetch)
  std::vector<int32_t> class_order[kNumClasses];
  int64_t gws_stride_words = 0;
  DevBuf d_nodes, d_tasks, d_nbrs, d_lo2gid, d_srp, d_scol, d_irp, d_icol, d_pairs, d_order, d_counters;
  DevBuf d_pws, d_gws, d_adam, d_m0, d_out, d_feat, d_dense_off, d_dense, d_rows;
  DevBuf d_trace, d_trpred, d_trouter, d_min, d_vin, d_fsin, d_Mout, d_mout, d_vout, d_fsout, d_m0dense, d_offedge;   // gx_explain_io staging (GX_HOST)
  DevBuf d_dn_thr, d_dn_cnt, d_dn_slots, d_dn_vals, d_send, d_us, d_gang, d_fwd;
  GxComm* comm = nullptr;
  int32_t label_min = 0, label_max = 0, pred_min = 0, pred_max = 0;   // ranges of the uploaded labels (checked against num_classes at plan time)
  bool has_label = false;
  GxPlanArrays plan{};
  // graph-classification mode
  bool has_batch = false, has_gplan = false;
  GxGraphBatchDev gb{};
  DevBuf gb_rowptr, gb_col, gb_feat, gb_label;
  std::vector<int32_t> gb_h_rowptr, gb_h_label;
  int g_count = 0;
  int64_t g_total_e = 0;
  int g_max_smem = 0, g_max_np = 0;
  // graph mode launch classes (by shared-memory footprint, like node mode): tasks per class, the class's largest footprint / pair count
  int g_class_n[6] = {}, g_class_smem[6] = {}, g_class_np[6] = {};
  // explain_graph_var.cu classes (small / large slab) per routing: [0] the batch with Adam (tasks the shared-memory kernel does not
  // take), [1] the whole batch (optimisers other than Adam); their task ids follow the shared-memory classes in d_order ([0]) or
  // fill d_order[count, 2 count) ([1]); words = the class's largest slab
  int gv_n[2][2] = {}, gv_off[2] = {};
  int64_t gv_words[2][2] = {};
  // slot workspace
  DevBuf ws_buf;
  GxSlotWs ws{};
};

namespace {

int ensure_slot_ws(gx_handle* h) {
  const int64_t N = h->g.N;
  const int W = (int)((N + 31) / 32);
  int slots = h->num_sms * 8;
  const size_t per_slot = (size_t)W * 4 + (size_t)(W + 1) * 4 + (size_t)N + (size_t)(N + 1) * 4 * 2 + (size_t)N * 4 * 2 + 64;
  const size_t budget = (size_t)4 << 30;
  while (slots > 1 && per_slot * slots > budget) slots /= 2;
  if (h->ws.slots == slots && h->ws.W == W && h->ws_buf.p) return GX_OK;
  // carve (each array 16B aligned)
  auto al = [](size_t x) { return (x + 15) / 16 * 16; };
  size_t o = 0;
  const size_t o_bm = o; o += al((size_t)slots * W * 4);
  const size_t o_wp = o; o += al((size_t)slots * (W + 1) * 4);
  const size_t o_q = o; o += al((size_t)slots * (N + 1) * 4);
  const size_t o_loc = o; o += al((size_t)slots * N * 4);
  const size_t o_cof = o; o += al((size_t)slots * N * 4);
  const size_t o_pb = o; o += al((size_t)slots * (N + 1) * 4);
  const size_t o_dist = o; o += al((size_t)slots * N);
  GX_CUDA_CHECK(h->ws_buf.reserve(o));
  char* b = h->ws_buf.as<char>();
  h->ws.bm = (uint32_t*)(b + o_bm);
  h->ws.wpref = (int32_t*)(b + o_wp);
  h->ws.q = (int32_t*)(b + o_q);
  h->ws.loc = (int32_t*)(b + o_loc);
  h->ws.cof = (int32_t*)(b + o_cof);
  h->ws.pbase = (int32_t*)(b + o_pb);
  h->ws.dist = (uint8_t*)(b + o_dist);
  h->ws.W = W;
  h->ws.slots = slots;
  GX_CUDA_CHECK(cudaMemsetAsync(h->ws.bm, 0, (size_t)slots * W * 4, h->stream));
  return GX_OK;
}

int task_smem_class(const GxTask& T, const GxModelDev& m, bool force_stream, int* bytes_out) {
  // shared-memory classes always use 16-bit indices: a task with n or e1 >= 65535 cannot fit 227 KB anyway
  const bool small_idx = !force_stream && T.n < 65535 && T.e1 < 65535;
  for (int c = 0; small_idx && c < kStreamClass; ++c) {
    const int nwarps = kClasses[c].threads / 32;
    const GxLayout L = gx_make_layout(T.n, T.n1, T.n2, T.e1, T.npairs_in, m.d, m.hid, m.emb, m.C, nwarps, 2);
    const int64_t bytes = (int64_t)L.total_words * 4;
    if (bytes <= kClasses[c].cap_bytes) {
      *bytes_out = (int)bytes;
      return c;
    }
  }
  *bytes_out = 0;  // streaming class (explain_stream.cu): state in a global slab, sized by gx_make_stream_layout
  return kStreamClass;
}

}  // namespace

extern "C" {

const char* gx_last_error(void) { return g_err; }
int gx_version(void) { return GX_VERSION; }

void gx_default_hparams(gx_hparams* hp) {
  if (!hp) return;
  hp->num_epochs = 100;
  hp->lr = 0.1f;
  hp->beta1 = 0.9f;
  hp->beta2 = 0.999f;
  hp->eps = 1e-8f;
  hp->coef_size = 0.005f;
  hp->coef_feat_size = 1.0f;
  hp->coef_ent = 1.0f;
  hp->coef_lap = 1.0f;
  hp->mask_act = 0;
  hp->mask_bias = 0;
  hp->init = GX_INIT_M0;
  hp->seed = 0;
  hp->start_step = 0;
  hp->opt = GX_OPT_ADAM;
  hp->opt_scheduler = GX_SCHED_NONE;
  hp->opt_decay_step = 0;
  hp->opt_decay_rate = 1.0f;
  hp->opt_restart = 0;
}

int gx_create(int device, gx_handle** out) {
  if (!out) { gx_set_error("gx_create: out is NULL"); return GX_ERR_INVALID; }
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    gx_set_error("gx_create: no CUDA device (%s); libgnnx has no CPU fallback",
                 e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return GX_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) { gx_set_error("gx_create: device %d out of range [0,%d)", device, ndev); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(device));
  cudaDeviceProp prop;
  GX_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    gx_set_error("gx_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return GX_ERR_CUDA;
  }
  if (const char* env = getenv("GNNX_CLASS_THREADS")) {   // tuning knob: threads per launch class, comma separated
    int v[kNumClasses], k = 0;
    const char* p = env;
    while (*p && k < kNumClasses) { v[k++] = atoi(p); while (*p && *p != ',') ++p; if (*p == ',') ++p; }
    // (a class runs the 256-thread kernel with up to 256 threads or the 512-thread kernel with exactly 512)
    for (int c = 0; c < k; ++c) if (v[c] >= 32 && v[c] % 32 == 0 && (v[c] <= 256 || v[c] == 512)) kClasses[c].threads = v[c];
  }
  gx_handle* h = new gx_handle();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  if (const char* env = getenv("GNNX_FORCE_STREAM")) h->force_stream = atoi(env) != 0;
  if (const char* env = getenv("GNNX_GANG")) h->gang_override = atoi(env);
  if (const char* env = getenv("GNNX_CLUSTER_SIZE")) { const int v = atoi(env); if (v == 0 || v == 1 || v == 2 || v == 4) h->cluster_size = v; }
  if (const char* env = getenv("GNNX_CLUSTER_COST")) { const long long v = atoll(env); if (v > 0) h->cluster_cost = v; }
  if (const char* env = getenv("GNNX_IEEE_EDGE")) h->ieee_edge = atoi(env) != 0;
  for (int i = 0; i < kNumStreams; ++i) {
    GX_CUDA_CHECK(cudaStreamCreateWithFlags(&h->side[i], cudaStreamNonBlocking));
    GX_CUDA_CHECK(cudaEventCreate(&h->ev_join[i]));
    GX_CUDA_CHECK(cudaEventCreate(&h->ev_begin[i]));
  }
  GX_CUDA_CHECK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  GX_CUDA_CHECK(cudaEventCreate(&h->ev_t0));
  GX_CUDA_CHECK(cudaEventCreate(&h->ev_t1));
  *out = h;
  return GX_OK;
}

int gx_destroy(gx_handle* h) {
  if (!h) return GX_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  DevBuf* bufs[] = {&h->g_rowptr, &h->g_col, &h->g_feat, &h->g_label, &h->g_pred, &h->m_buf, &h->d_nodes,
                    &h->d_tasks, &h->d_nbrs, &h->d_lo2gid, &h->d_srp, &h->d_scol, &h->d_irp, &h->d_icol,
                    &h->d_pairs, &h->d_order, &h->d_counters, &h->gb_rowptr, &h->gb_col, &h->gb_feat, &h->gb_label, &h->d_pws, &h->d_gws, &h->d_adam, &h->d_m0, &h->d_out,
                    &h->d_feat, &h->d_dense_off, &h->d_dense, &h->d_rows, &h->ws_buf, &h->d_trace, &h->d_trpred, &h->d_trouter, &h->d_min, &h->d_vin,
                    &h->d_fsin, &h->d_Mout, &h->d_mout, &h->d_vout, &h->d_fsout, &h->d_m0dense, &h->d_offedge,
                    &h->d_dn_thr, &h->d_dn_cnt, &h->d_dn_slots, &h->d_dn_vals, &h->d_send, &h->d_us, &h->d_gang, &h->d_fwd};
  gx_comm_impl_destroy(h->comm);
  h->comm = nullptr;
  for (DevBuf* b : bufs) b->release();
  for (int i = 0; i < kNumStreams; ++i) {
    if (h->side[i]) cudaStreamDestroy(h->side[i]);
    if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
    if (h->ev_begin[i]) cudaEventDestroy(h->ev_begin[i]);
  }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_t0) cudaEventDestroy(h->ev_t0);
  if (h->ev_t1) cudaEventDestroy(h->ev_t1);
  delete h;
  return GX_OK;
}

int gx_set_stream(gx_handle* h, void* cuda_stream) {
  if (!h) { gx_set_error("gx_set_stream: NULL handle"); return GX_ERR_INVALID; }
  h->stream = (cudaStream_t)cuda_stream;
  return GX_OK;
}

int gx_sync(gx_handle* h) {
  if (!h) { gx_set_error("gx_sync: NULL handle"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return GX_OK;
}

int64_t gx_launch_count(gx_handle* h) { return h ? h->launches : 0; }
int gx_plan_class_counts(gx_handle* h, int32_t counts[7], int32_t smem_bytes[7], int32_t* cluster_size) {
  if (!h || !counts || !h->has_plan) { gx_set_error("gx_plan_class_counts: no plan (call gx_plan_nodes)"); return GX_ERR_INVALID; }
  for (int c = 0; c < kNumClasses; ++c) {
    counts[c] = (int32_t)h->class_order[c].size();
    if (smem_bytes) {
      smem_bytes[c] = 0;
      for (int32_t t : h->class_order[c]) smem_bytes[c] = std::max(smem_bytes[c], h->tasks[t].smem_bytes);
    }
  }
  if (cluster_size) *cluster_size = h->plan_cluster;
  return GX_OK;
}

/* debug only (not in gnnx.h): device buffer receiving the shared-memory slab of the first task of each class */
int gx_debug_set_dump(gx_handle* h, float* dev_buf) { if (!h) return GX_ERR_INVALID; h->dbg = dev_buf; return GX_OK; }

/* debug only: IEEE exp/div/sqrt in the edge phase instead of the hardware approximations (parity measurements) */
int gx_debug_ieee_edge(gx_handle* h, int on) { if (!h) return GX_ERR_INVALID; h->ieee_edge = on != 0; return GX_OK; }

/* debug only (not in gnnx.h): plan every task into the streaming class (explain_stream.cu) regardless of its size */
int gx_model_forward(gx_handle* h, gx_memspace space, float* pred) {
  if (!h || !pred) { gx_set_error("gx_model_forward: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_graph || !h->has_model) { gx_set_error("gx_model_forward: call gx_set_model and gx_set_graph_csr first"); return GX_ERR_INVALID; }
  if (h->g.d != h->m.d) { gx_set_error("gx_model_forward: graph feat_dim %d != model input_dim %d", h->g.d, h->m.d); return GX_ERR_INVALID; }
  if (h->m.hid > 32 || h->m.emb > 32) { gx_set_error("gx_model_forward: widths > 32 are not built (pass pred to the Explainer)"); return GX_ERR_UNSUPPORTED; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const size_t np_ = (size_t)h->g.N * h->m.C;
  GX_CUDA_CHECK(h->d_fwd.reserve(((size_t)h->m.L * h->g.N * 32 + np_) * 4));
  float* H = h->d_fwd.as<float>();
  float* pd = space == GX_DEVICE ? pred : H + (size_t)h->m.L * h->g.N * 32;
  GX_CUDA_CHECK(gx_launch_model_forward(h->g, h->m, H, pd, nullptr, h->stream));
  h->launches += h->m.L + 1;
  if (space != GX_DEVICE) {
    GX_CUDA_CHECK(cudaMemcpyAsync(pred, pd, np_ * 4, cudaMemcpyDeviceToHost, h->stream));
    GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  }
  return GX_OK;
}
int gx_debug_set_gang(gx_handle* h, int ctas_per_task) { if (!h) return GX_ERR_INVALID; h->gang_override = ctas_per_task; return GX_OK; }
int gx_debug_set_cluster(gx_handle* h, int cluster_size, int64_t min_cost) {
  if (!h || !(cluster_size == 0 || cluster_size == 1 || cluster_size == 2 || cluster_size == 4)) return GX_ERR_INVALID;
  h->cluster_size = cluster_size; h->cluster_cost = min_cost; h->has_plan = false;
  return GX_OK;
}
int gx_debug_force_stream(gx_handle* h, int on) { if (!h) return GX_ERR_INVALID; h->force_stream = on != 0; h->has_plan = false; return GX_OK; }

int gx_last_explain_ms(gx_handle* h, float* ms) {
  if (!h || !ms) { gx_set_error("gx_last_explain_ms: NULL argument"); return GX_ERR_INVALID; }
  if (!h->timed) { gx_set_error("gx_last_explain_ms: no gx_explain_nodes call yet"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  GX_CUDA_CHECK(cudaEventSynchronize(h->ev_t1));
  GX_CUDA_CHECK(cudaEventElapsedTime(ms, h->ev_t0, h->ev_t1));
  return GX_OK;
}

int gx_last_class_ms(gx_handle* h, float begin_ms[7], float end_ms[7]) {
  if (!h || !begin_ms || !end_ms) { gx_set_error("gx_last_class_ms: NULL argument"); return GX_ERR_INVALID; }
  if (!h->timed) { gx_set_error("gx_last_class_ms: no gx_explain_nodes call yet"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  GX_CUDA_CHECK(cudaEventSynchronize(h->ev_t1));
  for (int c = 0; c < kNumClasses; ++c) {
    begin_ms[c] = end_ms[c] = -1.f;
    if (!h->class_used[c]) continue;
    GX_CUDA_CHECK(cudaEventElapsedTime(&begin_ms[c], h->ev_t0, h->ev_begin[c]));
    GX_CUDA_CHECK(cudaEventElapsedTime(&end_ms[c], h->ev_t0, h->ev_join[c]));
  }
  return GX_OK;
}

int gx_set_model(gx_handle* h, const gx_model_dims* dims, const float* const* conv_w,
                 const float* const* conv_b, const float* pred_w, const float* pred_b) {
  if (!h || !dims || !conv_w || !pred_w || !pred_b) { gx_set_error("gx_set_model: NULL argument"); return GX_ERR_INVALID; }
  if (dims->num_layers < 2 || dims->num_layers > GX_MAX_LAYERS) {
    gx_set_error("gx_set_model: num_layers=%d outside [2,%d]", dims->num_layers, GX_MAX_LAYERS);
    return GX_ERR_UNSUPPORTED;
  }
  if (dims->hidden_dim < 1 || dims->embed_dim < 1 || dims->hidden_dim > 128 || dims->embed_dim > 128) {
    gx_set_error("gx_set_model: hidden_dim=%d output_dim=%d; this build supports widths up to 128 (tuned kernels up to 32, the variant kernel beyond)", dims->hidden_dim, dims->embed_dim);
    return GX_ERR_UNSUPPORTED;
  }
  if (dims->input_dim < 1 || dims->input_dim > 128) {
    gx_set_error("gx_set_model: input_dim=%d outside [1,128] supported by the shared-memory kernel", dims->input_dim);
    return GX_ERR_UNSUPPORTED;
  }
  if (dims->num_classes < 1) { gx_set_error("gx_set_model: num_classes < 1"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  if (dims->num_layers != 3 || (dims->flags & GX_MODEL_BN) || dims->hidden_dim > 32 || dims->embed_dim > 32) {
    // Model variant (num_gc_layers 2 / 4, --bn, widths 33..128): explain_var.cu, true widths (a zero-padded column would enter the bn statistics).
    const int L = dims->num_layers, d = dims->input_dim, hid0 = dims->hidden_dim, emb0 = dims->embed_dim, C = dims->num_classes;
    if (gx_var_smem_bytes(d, L, hid0, emb0, C) > gx_explain_max_smem()) { gx_set_error("gx_set_model: model variant does not fit shared memory"); return GX_ERR_UNSUPPORTED; }
    std::vector<float> host;
    size_t offW[GX_MAX_LAYERS], offb[GX_MAX_LAYERS];
    auto al4 = [&]() { while (host.size() % 4) host.push_back(0.f); };
    for (int l = 0; l < L; ++l) {
      if (!conv_w[l]) { gx_set_error("gx_set_model: conv_w[%d] is NULL", l); return GX_ERR_INVALID; }
      const int win = l == 0 ? d : hid0, wout = l == L - 1 ? emb0 : hid0;
      al4(); offW[l] = host.size();
      host.insert(host.end(), conv_w[l], conv_w[l] + (size_t)win * wout);
      al4(); offb[l] = host.size();
      for (int c = 0; c < wout; ++c) host.push_back((conv_b && conv_b[l]) ? conv_b[l][c] : 0.f);
    }
    const int PD0 = hid0 * (L - 1) + emb0;
    al4(); const size_t offWp = host.size();
    host.insert(host.end(), pred_w, pred_w + (size_t)C * PD0);
    al4(); const size_t offbp = host.size();
    host.insert(host.end(), pred_b, pred_b + C);
    GX_CUDA_CHECK(h->m_buf.reserve(host.size() * 4));
    GX_CUDA_CHECK(cudaMemcpyAsync(h->m_buf.p, host.data(), host.size() * 4, cudaMemcpyHostToDevice, h->stream));
    GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
    float* b = h->m_buf.as<float>();
    h->m = GxModelDev{};
    h->m.d = d; h->m.hid = hid0; h->m.emb = emb0; h->m.C = C; h->m.L = L;
    h->m.bn = (dims->flags & GX_MODEL_BN) ? 1 : 0; h->m.variant = 1;
    for (int l = 0; l < L; ++l) { h->m.W[l] = b + offW[l]; h->m.Wt[l] = nullptr; h->m.b[l] = b + offb[l]; }
    h->m.Wp = b + offWp; h->m.bp = b + offbp;
    h->has_model = true; h->has_plan = false;
    return GX_OK;
  }
  // The kernels are instantiated for the reference default 20/20 and for 32/32; any other width <= 32 is
  // zero-padded to 32.  Padding is exact: a padded output column is 0*W + 0 = 0, contributes nothing to the
  // row norm, stays 0 through normalise/ReLU, and its pred_model column is 0 (forward and backward).
  const int d = dims->input_dim, hid0 = dims->hidden_dim, emb0 = dims->embed_dim, C = dims->num_classes;
  const bool native = hid0 == 20 && emb0 == 20;
  const int hid = native ? 20 : 32, emb = native ? 20 : 32;
  const int in0[3] = {d, hid0, hid0}, out0[3] = {hid0, hid0, emb0};
  const int in_dim[3] = {d, hid, hid}, out_dim[3] = {hid, hid, emb};
  const int PD0 = 2 * hid0 + emb0, PD = 2 * hid + emb;
  std::vector<float> host;
  size_t offW[3], offWt[3], offb[3], offWp, offbp;
  auto al4 = [&]() { while (host.size() % 4) host.push_back(0.f); };
  for (int l = 0; l < 3; ++l) {
    if (!conv_w[l]) { gx_set_error("gx_set_model: conv_w[%d] is NULL", l); return GX_ERR_INVALID; }
    auto Wat = [&](int f, int c) -> float { return (f < in0[l] && c < out0[l]) ? conv_w[l][(size_t)f * out0[l] + c] : 0.f; };
    al4(); offW[l] = host.size();
    for (int f = 0; f < in_dim[l]; ++f) for (int c = 0; c < out_dim[l]; ++c) host.push_back(Wat(f, c));
    al4(); offWt[l] = host.size();
    for (int c = 0; c < out_dim[l]; ++c) for (int f = 0; f < in_dim[l]; ++f) host.push_back(Wat(f, c));
    al4(); offb[l] = host.size();
    for (int c = 0; c < out_dim[l]; ++c) host.push_back((conv_b && conv_b[l] && c < out0[l]) ? conv_b[l][c] : 0.f);
  }
  al4(); offWp = host.size();
  for (int c = 0; c < C; ++c)
    for (int k = 0; k < PD; ++k) {
      const int part = k / hid >= 2 ? 2 : k / hid, within = k - part * hid;     // padded column -> (layer, feature)
      const int w0 = part == 2 ? emb0 : hid0;
      host.push_back(within < w0 ? pred_w[(size_t)c * PD0 + part * hid0 + within] : 0.f);
    }
  al4(); offbp = host.size();
  host.insert(host.end(), pred_b, pred_b + C);
  GX_CUDA_CHECK(h->m_buf.reserve(host.size() * 4));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->m_buf.p, host.data(), host.size() * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  float* b = h->m_buf.as<float>();
  h->m = GxModelDev{};
  h->m.d = d; h->m.hid = hid; h->m.emb = emb; h->m.C = C; h->m.L = 3;
  for (int l = 0; l < 3; ++l) { h->m.W[l] = b + offW[l]; h->m.Wt[l] = b + offWt[l]; h->m.b[l] = b + offb[l]; }
  h->m.Wp = b + offWp;
  h->m.bp = b + offbp;
  h->has_model = true;
  h->has_plan = false;
  return GX_OK;
}

int gx_set_graph_csr(gx_handle* h, int64_t N, const int32_t* rowptr, const int32_t* col,
                     const float* feat, int32_t d, const int32_t* label, const int32_t* pred_label) {
  if (!h || !rowptr || !col || !feat || !pred_label) { gx_set_error("gx_set_graph_csr: NULL argument"); return GX_ERR_INVALID; }
  if (N < 1 || N > 0x7fffffff - 64) { gx_set_error("gx_set_graph_csr: num_nodes out of range"); return GX_ERR_INVALID; }
  if (rowptr[0] != 0) { gx_set_error("gx_set_graph_csr: rowptr[0] != 0"); return GX_ERR_INVALID; }
  const int64_t nnz = rowptr[N];
  for (int64_t i = 0; i < N; ++i) {
    if (rowptr[i + 1] < rowptr[i]) { gx_set_error("gx_set_graph_csr: rowptr not monotone at %lld", (long long)i); return GX_ERR_INVALID; }
    for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
      if (col[e] < 0 || col[e] >= N) { gx_set_error("gx_set_graph_csr: col out of range in row %lld", (long long)i); return GX_ERR_INVALID; }
      if (e > rowptr[i] && col[e] <= col[e - 1]) { gx_set_error("gx_set_graph_csr: row %lld columns not strictly ascending", (long long)i); return GX_ERR_INVALID; }
    }
  }
  // symmetric pattern (the reference's datasets are undirected 0/1 adjacency)
  for (int64_t i = 0; i < N; ++i)
    for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
      const int32_t j = col[e];
      if (!std::binary_search(col + rowptr[j], col + rowptr[j + 1], (int32_t)i)) {
        gx_set_error("gx_set_graph_csr: adjacency not symmetric: (%lld,%d) present, (%d,%lld) absent", (long long)i, j, j, (long long)i);
        return GX_ERR_UNSUPPORTED;
      }
    }
  h->has_label = label != nullptr;
  h->label_min = h->label_max = label ? label[0] : 0;
  h->pred_min = h->pred_max = pred_label[0];
  for (int64_t i = 0; i < N; ++i) {
    if (label) { h->label_min = std::min(h->label_min, label[i]); h->label_max = std::max(h->label_max, label[i]); }
    h->pred_min = std::min(h->pred_min, pred_label[i]); h->pred_max = std::max(h->pred_max, pred_label[i]);
  }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  GX_CUDA_CHECK(h->g_rowptr.reserve((size_t)(N + 1) * 4));
  GX_CUDA_CHECK(h->g_col.reserve((size_t)std::max<int64_t>(nnz, 1) * 4));
  GX_CUDA_CHECK(h->g_feat.reserve((size_t)N * d * 4));
  GX_CUDA_CHECK(h->g_label.reserve((size_t)N * 4));
  GX_CUDA_CHECK(h->g_pred.reserve((size_t)N * 4));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->g_rowptr.p, rowptr, (size_t)(N + 1) * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->g_col.p, col, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->g_feat.p, feat, (size_t)N * d * 4, cudaMemcpyHostToDevice, h->stream));
  if (label) GX_CUDA_CHECK(cudaMemcpyAsync(h->g_label.p, label, (size_t)N * 4, cudaMemcpyHostToDevice, h->stream));
  else GX_CUDA_CHECK(cudaMemsetAsync(h->g_label.p, 0, (size_t)N * 4, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->g_pred.p, pred_label, (size_t)N * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->g.N = N; h->g.nnz = (int32_t)nnz;
  h->g.rowptr = h->g_rowptr.as<int32_t>(); h->g.col = h->g_col.as<int32_t>();
  h->g.feat = h->g_feat.as<float>(); h->g.d = d;
  h->g.label = h->g_label.as<int32_t>(); h->g.pred_label = h->g_pred.as<int32_t>();
  h->has_graph = true;
  h->has_plan = false;
  h->ws.slots = 0;
  return GX_OK;
}

int gx_neighborhood_rows(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops, uint8_t* out_rows) {
  if (!h || !nodes || !out_rows) { gx_set_error("gx_neighborhood_rows: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_graph) { gx_set_error("gx_neighborhood_rows: call gx_set_graph_csr first"); return GX_ERR_INVALID; }
  if (n_hops < 1 || n_hops >= GX_MAX_LEVELS) { gx_set_error("gx_neighborhood_rows: n_hops=%d outside [1,%d]", n_hops, GX_MAX_LEVELS - 1); return GX_ERR_INVALID; }
  if (count <= 0) return GX_OK;
  for (int t = 0; t < count; ++t)
    if (nodes[t] < 0 || nodes[t] >= h->g.N) { gx_set_error("gx_neighborhood_rows: node %d out of range", nodes[t]); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  int rc = ensure_slot_ws(h);
  if (rc != GX_OK) return rc;
  const size_t bytes = (size_t)count * h->g.N;
  GX_CUDA_CHECK(h->d_nodes.reserve((size_t)count * 4));
  GX_CUDA_CHECK(h->d_rows.reserve(bytes));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_nodes.p, nodes, (size_t)count * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemsetAsync(h->d_rows.p, 0, bytes, h->stream));
  GX_CUDA_CHECK(gx_launch_hop_rows(h->g, h->d_nodes.as<int32_t>(), count, n_hops, h->ws, h->d_rows.as<uint8_t>(), h->stream));
  h->launches += 1;
  GX_CUDA_CHECK(cudaMemcpyAsync(out_rows, h->d_rows.p, bytes, cudaMemcpyDeviceToHost, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return GX_OK;
}

int gx_plan_nodes(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops,
                  int64_t* total_nodes, int64_t* total_edges) {
  if (!h || !nodes) { gx_set_error("gx_plan_nodes: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_graph || !h->has_model) { gx_set_error("gx_plan_nodes: call gx_set_model and gx_set_graph_csr first"); return GX_ERR_INVALID; }
  if (h->g.d != h->m.d) { gx_set_error("gx_plan_nodes: graph feat_dim %d != model input_dim %d", h->g.d, h->m.d); return GX_ERR_INVALID; }
  if (n_hops < 1 || n_hops >= GX_MAX_LEVELS) { gx_set_error("gx_plan_nodes: n_hops=%d outside [1,%d]", n_hops, GX_MAX_LEVELS - 1); return GX_ERR_INVALID; }
  if (n_hops < 2) { gx_set_error("gx_plan_nodes: n_hops=1 never contains the node itself without a self loop"); return GX_ERR_UNSUPPORTED; }
  if (count <= 0) { gx_set_error("gx_plan_nodes: count <= 0"); return GX_ERR_INVALID; }
  for (int t = 0; t < count; ++t)
    if (nodes[t] < 0 || nodes[t] >= h->g.N) { gx_set_error("gx_plan_nodes: node %d out of range [0,%lld)", nodes[t], (long long)h->g.N); return GX_ERR_INVALID; }
  // the reference indexes pred[gt_label] / a float pred_label vector (explain.py:750-753,789): a label outside [0,C) is an IndexError there
  if (h->has_label && (h->label_min < 0 || h->label_max >= h->m.C)) { gx_set_error("gx_plan_nodes: label values span [%d,%d], model has %d classes", h->label_min, h->label_max, h->m.C); return GX_ERR_INVALID; }
  if (h->pred_min < 0 || h->pred_max >= h->m.C) { gx_set_error("gx_plan_nodes: pred_label values span [%d,%d], model has %d classes", h->pred_min, h->pred_max, h->m.C); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const double t0 = host_timing() ? now_us() : 0.0;
  h->has_plan = false;
  h->has_gplan = false;
  int rc = ensure_slot_ws(h);
  if (rc != GX_OK) return rc;
  GX_CUDA_CHECK(h->d_nodes.reserve((size_t)count * 4));
  GX_CUDA_CHECK(h->d_tasks.reserve((size_t)count * sizeof(GxTask)));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_nodes.p, nodes, (size_t)count * 4, cudaMemcpyHostToDevice, h->stream));
  const int row_lvl = h->m.L - 1;
  GX_CUDA_CHECK(gx_launch_khop_count(h->g, h->d_nodes.as<int32_t>(), count, n_hops, row_lvl, h->ws, h->d_tasks.as<GxTask>(), h->stream));
  h->launches += 1;
  h->tasks.resize(count);
  GX_CUDA_CHECK(cudaMemcpyAsync(h->tasks.data(), h->d_tasks.p, (size_t)count * sizeof(GxTask), cudaMemcpyDeviceToHost, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  const double t1 = host_timing() ? now_us() : 0.0;
  // host, step 1: status checks and the offsets the fill kernel needs
  int64_t tn = 0, te = 0, tp = 0;
  for (int t = 0; t < count; ++t) {
    GxTask& T = h->tasks[t];
    if (T.status != 0) {
      gx_set_error("gx_plan_nodes: node %d is not inside its own %d-hop neighbourhood (isolated node?)", T.node, n_hops);
      return GX_ERR_NODE;
    }
    if (T.e_d % 2 != 0) { gx_set_error("gx_plan_nodes: induced sub-adjacency of node %d is not symmetric", T.node); return GX_ERR_INVALID; }
    T.node_off = tn; T.rp_off = tn + t; T.edge_off = te; T.pair_off = tp;
    tn += T.n; te += T.e_d; tp += T.npairs;
  }
  h->count = count; h->n_hops = n_hops; h->total_n = tn; h->total_e = te;
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_tasks.p, h->tasks.data(), (size_t)count * sizeof(GxTask), cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(h->d_counters.reserve(kNumClasses * 4));
  GX_CUDA_CHECK(h->d_nbrs.reserve((size_t)std::max<int64_t>(tn, 1) * 4));
  GX_CUDA_CHECK(h->d_lo2gid.reserve((size_t)std::max<int64_t>(tn, 1) * 4));
  GX_CUDA_CHECK(h->d_srp.reserve((size_t)(tn + count) * 4));
  GX_CUDA_CHECK(h->d_irp.reserve((size_t)(tn + count) * 4));
  GX_CUDA_CHECK(h->d_scol.reserve((size_t)std::max<int64_t>(te, 1) * 4));
  GX_CUDA_CHECK(h->d_icol.reserve((size_t)std::max<int64_t>(te, 1) * 4 * 3));
  GX_CUDA_CHECK(h->d_pairs.reserve((size_t)std::max<int64_t>(tp, 1) * 4 * 6));
  h->plan.tasks = h->d_tasks.as<GxTask>();
  h->plan.nbrs = h->d_nbrs.as<int32_t>();
  h->plan.lo2gid = h->d_lo2gid.as<int32_t>();
  h->plan.sub_rowptr = h->d_srp.as<int32_t>();
  h->plan.irowptr = h->d_irp.as<int32_t>();
  h->plan.sub_col = h->d_scol.as<int32_t>();
  h->plan.icol = h->d_icol.as<int32_t>();
  h->plan.cs2is = h->plan.icol + te;
  h->plan.is2cs = h->plan.icol + 2 * te;
  int32_t* pb = h->d_pairs.as<int32_t>();
  h->plan.pair_i = pb; h->plan.pair_j = pb + tp; h->plan.pair_pij = pb + 2 * tp;
  h->plan.pair_pji = pb + 3 * tp; h->plan.pair_oij = pb + 4 * tp; h->plan.pair_oji = pb + 5 * tp;
  const double t2 = host_timing() ? now_us() : 0.0;
  GX_CUDA_CHECK(gx_launch_khop_fill(h->g, count, n_hops, h->ws, h->plan, h->stream));
  h->launches += 1;
  // host, step 2 (while the fill kernel runs): launch classes and work order.  Nothing here is read by the device: T.smem_bytes and the
  // class lists stay on the host, only the order array is uploaded.
  for (int c = 0; c < kNumClasses; ++c) h->class_order[c].clear();
  int64_t gws_words = 0;
  auto cost = [&](int32_t t) { const GxTask& T = h->tasks[t]; return (int64_t)T.e1 * (h->m.d + 2 * h->m.hid) + (int64_t)T.n2 * 600 + (int64_t)T.npairs * 60; };
  const int g_cluster_size = h->cluster_size > 1 ? h->cluster_size : 1;
  const int64_t g_cluster_cost = h->cluster_cost;
  h->plan_cluster = g_cluster_size;
  for (int t = 0; t < count; ++t) {
    GxTask& T = h->tasks[t];
    int bytes = 0;
    int cls = h->m.variant ? kStreamClass : task_smem_class(T, h->m, h->force_stream, &bytes);
    if (h->m.variant) bytes = 0;
    if (cls < kStreamClass && g_cluster_size > 1 && cost(t) > g_cluster_cost) {
      // expensive task: one thread-block cluster (explain_node.cu, CS CTAs share the rows and pairs); decided by the task alone
      const GxLayout L = gx_make_layout(T.n, T.n1, T.n2, T.e1, T.npairs_in, h->m.d, h->m.hid, h->m.emb, h->m.C, kClasses[kClusterClass].threads / 32, 2, g_cluster_size);
      if ((int64_t)L.total_words * 4 <= kClasses[kClusterClass].cap_bytes) { cls = kClusterClass; bytes = L.total_words * 4; }
    }
    T.smem_bytes = bytes;
    if (cls == kStreamClass && h->m.variant)
      gws_words = std::max<int64_t>(gws_words, gx_make_var_layout(T.n, T.n2, T.e1, T.npairs_in, h->m.d, h->m.L, gx_var_row_stride(h->m.hid, h->m.emb)).total_words);
    else if (cls == kStreamClass)
      gws_words = std::max<int64_t>(gws_words, gx_make_stream_layout(T.n, T.n1, T.n2, T.e_d, T.npairs_in, h->m.d, h->m.hid, GX_STREAM_THREADS / 32).total_words);
    h->class_order[cls].push_back(t);
  }
  h->gws_stride_words = (gws_words + 3) / 4 * 4;
  if (h->cluster_size == 0 && !h->m.variant && !h->force_stream && h->class_order[kStreamClass].empty()) {
    // Latency mode (cluster_size 0): a batch that leaves SMs idle (one explain() call, a shard of a strong-scaled list) is bounded by the
    // latency of its most expensive tasks, so those run on thread-block clusters of the spare SMs.  A full batch (700 syn1 nodes on one
    // GPU needs ~180 SM-slots) has no spare SM and stays as it is.  A cluster sums the per-warp dL/dsF partials of its 32 / 64 warps in
    // another order than one CTA's 16 warps: the masks agree with the single-CTA run to round-off (2e-6 after 10 epochs), not bit for
    // bit -- which is why this mode is opt-in.
    // Latency model from profiles/r02b_cluster_study_syn1.json: 6 us per 1000 cost units on one CTA; a cluster divides that by its
    // size and adds 0.55 ms (2 CTAs) / 0.8 ms (4 CTAs) of cluster-barrier time per 100 epochs.
    double demand = 0;
    for (int c = 0; c < kStreamClass; ++c) demand += (double)h->class_order[c].size() / kClasses[c].ctas_per_sm;
    const int spare = h->num_sms - (int)(demand + 0.999);
    std::vector<int32_t> cand;
    for (int c : {kTwoClass, kOneClass}) for (int32_t t : h->class_order[c]) cand.push_back(t);
    std::stable_sort(cand.begin(), cand.end(), [&](int32_t x, int32_t y) { return cost(x) > cost(y); });
    auto lat = [&](int32_t t) { return 6e-6 * (double)cost(t); };
    int best_cs = 1, best_k = 0;
    if (!cand.empty() && spare >= 2) {
      double best = lat(cand[0]);
      for (int cs : {2, 4}) {
        const double ovh = cs == 2 ? 0.55 : 0.8;
        // the k most expensive tasks on clusters: every one of them must gain, and all of them must fit the class and the spare SMs
        int k = 0;
        while (k < (int)cand.size() && (k + 1) * cs <= spare && lat(cand[k]) / cs + ovh < lat(cand[k])) {
          const GxTask& T = h->tasks[cand[k]];
          const GxLayout L = gx_make_layout(T.n, T.n1, T.n2, T.e1, T.npairs_in, h->m.d, h->m.hid, h->m.emb, h->m.C, kClasses[kClusterClass].threads / 32, 2, cs);
          if ((int64_t)L.total_words * 4 > kClasses[kClusterClass].cap_bytes) break;
          ++k;
        }
        if (k == 0) continue;
        const double span = std::max(lat(cand[0]) / cs + ovh, k < (int)cand.size() ? lat(cand[k]) : 0.0);
        if (span < best * 0.95) { best = span; best_cs = cs; best_k = k; }
      }
    }
    if (best_cs > 1) {
      h->plan_cluster = best_cs;
      for (int i = 0; i < best_k; ++i) {
        const int32_t t = cand[i];
        GxTask& T = h->tasks[t];
        const GxLayout L = gx_make_layout(T.n, T.n1, T.n2, T.e1, T.npairs_in, h->m.d, h->m.hid, h->m.emb, h->m.C, kClasses[kClusterClass].threads / 32, 2, best_cs);
        T.smem_bytes = L.total_words * 4;
        for (int c : {kTwoClass, kOneClass}) {
          auto& v = h->class_order[c];
          v.erase(std::remove(v.begin(), v.end(), t), v.end());
        }
        h->class_order[kClusterClass].push_back(t);
      }
    }
  }
  std::vector<int32_t> order_all;
  for (int c = 0; c < kNumClasses; ++c) {
    auto& v = h->class_order[c];
    std::stable_sort(v.begin(), v.end(), [&](int32_t x, int32_t y) { return cost(x) > cost(y); });
  }
  {
    // The batch makespan is the latency of its most expensive tasks (one wave; a 512-thread task is ~15 % slower
    // when it shares the SM with a second one: profiles/r01d_timeline.md).  The top-K tasks of the 2-per-SM
    // class therefore run alone on an SM (moved to the 1-per-SM class, which requests the whole shared memory).
    static int topk = -1;
    if (topk < 0) { const char* e = getenv("GNNX_EXCLUSIVE_TOPK"); topk = e ? atoi(e) : 12; }
    auto& two = h->class_order[kTwoClass];
    auto& one = h->class_order[kOneClass];
    // only when the 2-per-SM class really pairs up tasks, and the exclusive SMs still leave everything in one wave
    int k = 0;
    if ((int)two.size() > h->num_sms) {
      k = topk;
      while (k > 0 && (int)one.size() + k + ((int)two.size() - k + 1) / 2 > (h->num_sms * 17) / 20) --k;
    }
    if (k > 0 && (int)two.size() > k) {
      one.insert(one.end(), two.begin(), two.begin() + k);
      two.erase(two.begin(), two.begin() + k);
      std::stable_sort(one.begin(), one.end(), [&](int32_t x, int32_t y) { return cost(x) > cost(y); });
    }
  }
  for (int c = 0; c < kNumClasses; ++c) {
    auto& v = h->class_order[c];
    order_all.insert(order_all.end(), v.begin(), v.end());
  }
  GX_CUDA_CHECK(h->d_order.reserve((size_t)count * 4));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_order.p, order_all.data(), (size_t)count * 4, cudaMemcpyHostToDevice, h->stream));
  // idx_new (the canonical description's position of the node) is copied back by gx_plan_fetch on demand.  The host still waits for the
  // fill kernel: explainer launches queued BEHIND it all become runnable at the same instant and the block scheduler interleaves the
  // launch classes arbitrarily, which costs the batch 0.5 ms (kernels 2.9 -> 3.5 ms, profiles/r02cl_cluster_auto.md); issued one by
  // one onto an idle GPU the most expensive class is placed first.
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->tasks_fetched = false;
  h->has_plan = true;
  if (host_timing()) {
    const double t3 = now_us();
    fprintf(stderr, "[gnnx] gx_plan_nodes(%d): count kernel + copy %.0f us, offsets + uploads %.0f us, fill kernel (host classes / order underneath) %.0f us\n", count, t1 - t0, t2 - t1, t3 - t2);
  }
  if (total_nodes) *total_nodes = tn;
  if (total_edges) *total_edges = te;
  return GX_OK;
}

int gx_plan_fetch(gx_handle* h, int64_t* node_off, int64_t* edge_off, int32_t* neighbors,
                  int32_t* node_idx_new, int32_t* sub_rowptr, int32_t* sub_col) {
  if (!h || !h->has_plan) { gx_set_error("gx_plan_fetch: no plan (call gx_plan_nodes)"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->count;
  if (node_off) { for (int t = 0; t < count; ++t) node_off[t] = h->tasks[t].node_off; node_off[count] = h->total_n; }
  if (edge_off) { for (int t = 0; t < count; ++t) edge_off[t] = h->tasks[t].edge_off; edge_off[count] = h->total_e; }
  if (node_idx_new) {
    if (!h->tasks_fetched) {   // only idx_new comes from the device copy (the host copy carries the launch classes)
      std::vector<GxTask> dev(count);
      GX_CUDA_CHECK(cudaMemcpyAsync(dev.data(), h->d_tasks.p, (size_t)count * sizeof(GxTask), cudaMemcpyDeviceToHost, h->stream));
      GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
      for (int t = 0; t < count; ++t) h->tasks[t].idx_new = dev[t].idx_new;
      h->tasks_fetched = true;
    }
    for (int t = 0; t < count; ++t) node_idx_new[t] = h->tasks[t].idx_new;
  }
  if (neighbors) GX_CUDA_CHECK(cudaMemcpyAsync(neighbors, h->d_nbrs.p, (size_t)h->total_n * 4, cudaMemcpyDeviceToHost, h->stream));
  if (sub_rowptr) GX_CUDA_CHECK(cudaMemcpyAsync(sub_rowptr, h->d_srp.p, (size_t)(h->total_n + count) * 4, cudaMemcpyDeviceToHost, h->stream));
  if (sub_col) GX_CUDA_CHECK(cudaMemcpyAsync(sub_col, h->d_scol.p, (size_t)h->total_e * 4, cudaMemcpyDeviceToHost, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return GX_OK;
}

}  // extern "C"

namespace {

// Device views of a gx_explain_io: identity for GX_DEVICE, staged through handle-owned buffers for GX_HOST.
struct IoDev {
  const float* m0 = nullptr;
  float* out = nullptr;
  float* feat = nullptr;
  GxExtra x{};
};

cudaError_t stage_in(gx_handle* h, DevBuf& b, const float* host, size_t n, const float** dev) {
  *dev = nullptr;
  if (!host || n == 0) return cudaSuccess;
  cudaError_t e = b.reserve(n * 4);
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(b.p, host, n * 4, cudaMemcpyHostToDevice, h->stream);
  *dev = b.as<float>();
  return e;
}
cudaError_t stage_out(DevBuf& b, float* host, size_t n, float** dev) {
  *dev = nullptr;
  if (!host) return cudaSuccess;
  cudaError_t e = b.reserve(std::max<size_t>(n, 1) * 4);
  *dev = b.as<float>();
  return e;
}

// Validates the optional buffers, stages them (GX_HOST) and fills the kernels' GxExtra.  epochs = num_epochs of the call.
int io_prepare(gx_handle* h, const char* who, const gx_hparams* hp, int mode, gx_memspace space, const gx_explain_io* io, int count,
               int64_t te, int d, int C, IoDev* D) {
  if (!io || !io->edge_mask) { gx_set_error("%s: io->edge_mask is NULL", who); return GX_ERR_INVALID; }
  const bool state = mode == 0 && hp->init == GX_INIT_STATE;
  if (mode == 0 && hp->init != GX_INIT_PHILOX && !io->m0_edges) { gx_set_error("%s: init %d needs m0_edges", who, hp->init); return GX_ERR_INVALID; }
  if (state && (!io->adam_m_in || !io->adam_v_in)) { gx_set_error("%s: GX_INIT_STATE needs adam_m_in and adam_v_in", who); return GX_ERR_INVALID; }
  if (state && hp->start_step < 0) { gx_set_error("%s: start_step < 0", who); return GX_ERR_INVALID; }
  if (!state && hp->start_step != 0) { gx_set_error("%s: start_step != 0 without GX_INIT_STATE", who); return GX_ERR_INVALID; }
  if (io->trace_pred && !io->trace) { gx_set_error("%s: trace_pred needs trace", who); return GX_ERR_INVALID; }
  if (io->trace && mode != 0) { gx_set_error("%s: no trace for the gradient baseline", who); return GX_ERR_INVALID; }
  if (io->trace && hp->num_epochs > 1536) { gx_set_error("%s: a trace supports at most 1536 epochs per call", who); return GX_ERR_UNSUPPORTED; }
  const size_t ne = (size_t)std::max<int64_t>(te, 1), nf = (size_t)count * d, nfs = (size_t)count * 3 * d;
  const size_t ntr = (size_t)count * hp->num_epochs * GX_TRACE_COLS, ntp = (size_t)count * hp->num_epochs * C;
  GxExtra& x = D->x;
  x.epochs = hp->num_epochs;
  if (space == GX_DEVICE) {
    D->m0 = io->m0_edges; D->out = io->edge_mask; D->feat = io->feat_mask;
    x.trace = io->trace; x.trace_pred = io->trace_pred;
    x.adam_m_in = io->adam_m_in; x.adam_v_in = io->adam_v_in; x.feat_state_in = io->feat_state_in;
    x.mask_param_out = io->mask_param_out; x.adam_m_out = io->adam_m_out; x.adam_v_out = io->adam_v_out; x.feat_state_out = io->feat_state_out;
  } else {
    const bool need_m0 = mode == 0 && hp->init != GX_INIT_PHILOX;
    GX_CUDA_CHECK(stage_in(h, h->d_m0, need_m0 ? io->m0_edges : nullptr, (size_t)te, &D->m0));
    GX_CUDA_CHECK(stage_out(h->d_out, io->edge_mask, ne, &D->out));
    GX_CUDA_CHECK(stage_out(h->d_feat, io->feat_mask, nf, &D->feat));
    GX_CUDA_CHECK(stage_out(h->d_trace, io->trace, ntr, &x.trace));
    GX_CUDA_CHECK(stage_out(h->d_trpred, io->trace_pred, ntp, &x.trace_pred));
    GX_CUDA_CHECK(stage_in(h, h->d_min, state ? io->adam_m_in : nullptr, (size_t)te, &x.adam_m_in));
    GX_CUDA_CHECK(stage_in(h, h->d_vin, state ? io->adam_v_in : nullptr, (size_t)te, &x.adam_v_in));
    GX_CUDA_CHECK(stage_in(h, h->d_fsin, state ? io->feat_state_in : nullptr, nfs, &x.feat_state_in));
    GX_CUDA_CHECK(stage_out(h->d_Mout, io->mask_param_out, ne, &x.mask_param_out));
    GX_CUDA_CHECK(stage_out(h->d_mout, io->adam_m_out, ne, &x.adam_m_out));
    GX_CUDA_CHECK(stage_out(h->d_vout, io->adam_v_out, ne, &x.adam_v_out));
    GX_CUDA_CHECK(stage_out(h->d_fsout, io->feat_state_out, nfs, &x.feat_state_out));
  }
  if (!state) { x.adam_m_in = nullptr; x.adam_v_in = nullptr; x.feat_state_in = nullptr; }
  if (x.trace) {
    GX_CUDA_CHECK(h->d_trouter.reserve((size_t)count * hp->num_epochs * 4 * sizeof(double)));
    GX_CUDA_CHECK(cudaMemsetAsync(h->d_trouter.p, 0, (size_t)count * hp->num_epochs * 4 * sizeof(double), h->stream));
    x.tr_outer = h->d_trouter.as<double>();
  }
  return GX_OK;
}

// copies the staged outputs back (GX_HOST) and synchronises
int io_finish(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io, int count, int64_t te, int d, int C, const IoDev& D) {
  if (space != GX_HOST) return GX_OK;
  auto back = [&](float* host, const float* dev, size_t n) -> cudaError_t {
    if (!host || !dev || n == 0) return cudaSuccess;
    return cudaMemcpyAsync(host, dev, n * 4, cudaMemcpyDeviceToHost, h->stream);
  };
  GX_CUDA_CHECK(back(io->edge_mask, D.out, (size_t)te));
  GX_CUDA_CHECK(back(io->feat_mask, D.feat, (size_t)count * d));
  GX_CUDA_CHECK(back(io->trace, D.x.trace, (size_t)count * hp->num_epochs * GX_TRACE_COLS));
  GX_CUDA_CHECK(back(io->trace_pred, D.x.trace_pred, (size_t)count * hp->num_epochs * C));
  GX_CUDA_CHECK(back(io->mask_param_out, D.x.mask_param_out, (size_t)te));
  GX_CUDA_CHECK(back(io->adam_m_out, D.x.adam_m_out, (size_t)te));
  GX_CUDA_CHECK(back(io->adam_v_out, D.x.adam_v_out, (size_t)te));
  GX_CUDA_CHECK(back(io->feat_state_out, D.x.feat_state_out, (size_t)count * 3 * d));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  return GX_OK;
}

// Per-step table for steps start+1 .. start+iters, in double like torch's python scalars: the epoch's learning rate under the
// scheduler (StepLR / CosineAnnealingLR are stepped once per epoch AFTER the optimiser, explain.py:144-146, so step t runs with the
// rate after t-1 scheduler steps) and, for Adam, the bias corrections (torch/optim/adam.py): (lr_t / (1-b1^t), sqrt(1-b2^t)).
int check_optimiser(const char* who, const gx_hparams* hp) {
  if (hp->opt < GX_OPT_ADAM || hp->opt > GX_OPT_ADAGRAD) { gx_set_error("%s: unknown optimiser %d", who, hp->opt); return GX_ERR_INVALID; }
  if (hp->opt_scheduler < GX_SCHED_NONE || hp->opt_scheduler > GX_SCHED_COS) { gx_set_error("%s: unknown scheduler %d", who, hp->opt_scheduler); return GX_ERR_INVALID; }
  if (hp->opt_scheduler == GX_SCHED_STEP && hp->opt_decay_step < 1) { gx_set_error("%s: step scheduler needs opt_decay_step >= 1", who); return GX_ERR_INVALID; }
  if (hp->opt_scheduler == GX_SCHED_COS && hp->opt_restart < 1) { gx_set_error("%s: cos scheduler needs opt_restart >= 1", who); return GX_ERR_INVALID; }
  return GX_OK;
}
int upload_adam_table(gx_handle* h, const gx_hparams* hp, int iters, int start) {
  // the table on the device is reused while the optimiser settings do not change (one explain call per step in a serving loop)
  AdamKey key{hp->lr, hp->beta1, hp->beta2, hp->opt_decay_rate, hp->opt, hp->opt_scheduler, hp->opt_decay_step, hp->opt_restart, iters, start};
  if (h->adam_valid && memcmp(&key, &h->adam_key, sizeof(key)) == 0 && h->d_adam.p) return GX_OK;
  std::vector<float2> tab(std::max(iters, 1));
  for (int k = 1; k <= iters; ++k) {
    const double t = (double)(start + k);
    const double e = t - 1.0;   // scheduler steps taken so far
    double lr = (double)hp->lr;
    if (hp->opt_scheduler == GX_SCHED_STEP) lr *= std::pow((double)hp->opt_decay_rate, std::floor(e / (double)hp->opt_decay_step));
    else if (hp->opt_scheduler == GX_SCHED_COS) lr *= 0.5 * (1.0 + std::cos(3.14159265358979323846 * e / (double)hp->opt_restart));
    if (hp->opt == GX_OPT_ADAM) {
      const double bc1 = 1.0 - std::pow((double)hp->beta1, t);
      const double bc2 = 1.0 - std::pow((double)hp->beta2, t);
      tab[k - 1].x = (float)(lr / bc1);
      tab[k - 1].y = (float)std::sqrt(bc2);
    } else {
      tab[k - 1].x = (float)lr;
      tab[k - 1].y = 1.0f;
    }
  }
  GX_CUDA_CHECK(h->d_adam.reserve(tab.size() * sizeof(float2)));
  // pageable source: the copy is staged before the call returns, the vector may go out of scope
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_adam.p, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  h->adam_key = key; h->adam_valid = true;
  return GX_OK;
}

void fill_hparams(const gx_handle* h, const gx_hparams* hp, int mode, bool trace, GxHparamsDev* hd) {
  hd->out_iter = mode == 1 ? 1 : hp->num_epochs - 1;
  hd->iters = (trace && mode == 0) ? hp->num_epochs : hd->out_iter;   // a trace also needs the last epoch's loss and the density after its step
  hd->one_minus_b1 = 1.0f - hp->beta1;
  hd->b2 = hp->beta2;
  hd->one_minus_b2 = 1.0f - hp->beta2;
  hd->eps = hp->eps;
  hd->c_size = hp->coef_size; hd->c_feat_size = hp->coef_feat_size; hd->c_ent = hp->coef_ent; hd->c_lap = hp->coef_lap;
  hd->adam_tab = h->d_adam.as<float2>();
  hd->init = hp->init;
  hd->flags = h->ieee_edge ? GX_HP_IEEE_EDGE : 0;
  hd->mode = mode;
  hd->opt = hp->opt;
  hd->seed = hp->seed;
}

}  // namespace

// mode 0: Explainer.explain's optimisation loop; mode 1: its model="grad" baseline (one forward/backward, explain.py:125-133,717-738)
static int explain_nodes_impl(gx_handle* h, const gx_hparams* hp, int mode, gx_memspace space, const gx_explain_io* io) {
  if (!h || !hp) { gx_set_error("gx_explain_nodes: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_plan) { gx_set_error("gx_explain_nodes: no plan (call gx_plan_nodes)"); return GX_ERR_INVALID; }
  const double t_entry = host_timing() ? now_us() : 0.0;
  // mask_act "ReLU": the reference's entropy term takes log(1 - relu(M)) with M ~ N(1, 2/n) -> NaN masks from step 1 (explain.py:755-770;
  // pinned by tests/test_oracle.py): nothing to reproduce.  mask_bias: the bias parameter starts at 0 where ReLU6'(0) = 0, so Adam never
  // moves it and the result equals the default run bit for bit (explain.py:657-660,673-676; same test): accepted, no extra state.
  if (hp->mask_act != 0) { gx_set_error("gx_explain_nodes: mask_act != sigmoid is not built (the reference's ReLU variant returns NaN masks)"); return GX_ERR_UNSUPPORTED; }
  if (hp->num_epochs < 1) { gx_set_error("gx_explain_nodes: num_epochs < 1"); return GX_ERR_INVALID; }
  { const int orc = check_optimiser("gx_explain_nodes", hp); if (orc != GX_OK) return orc; }
  const bool all_var = h->m.variant || hp->opt != GX_OPT_ADAM;   // every task through explain_var.cu
  if (all_var && (mode != 0 || hp->init == GX_INIT_STATE || (io && (io->trace || io->trace_pred || io->adam_m_out || io->adam_v_out || io->mask_param_out || io->feat_state_out)))) {
    gx_set_error("gx_explain_nodes: model variants (num_layers != 3 / --bn) and optimisers other than Adam build the mask optimisation only (no trace, optimiser state or gradient baseline)");
    return GX_ERR_UNSUPPORTED;
  }
  if (hp->init != GX_INIT_M0 && hp->init != GX_INIT_PHILOX && hp->init != GX_INIT_STATE) { gx_set_error("gx_explain_nodes: unknown init %d", hp->init); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->count;
  const int64_t te = h->total_e;
  IoDev D;
  int rc = io_prepare(h, "gx_explain_nodes", hp, mode, space, io, count, te, h->m.d, h->m.C, &D);
  if (rc != GX_OK) return rc;
  GxHparamsDev hd;
  fill_hparams(h, hp, mode, D.x.trace != nullptr, &hd);
  rc = upload_adam_table(h, hp, hd.iters, mode == 0 ? hp->start_step : 0);
  if (rc != GX_OK) return rc;
  hd.adam_tab = h->d_adam.as<float2>();   // (the buffer may have been (re)allocated by the upload)
  const float* m0_dev = D.m0;
  float* out_dev = D.out;
  float* feat_dev = D.feat;
  GX_CUDA_CHECK(cudaMemsetAsync(h->d_counters.p, 0, kNumClasses * 4, h->stream));
  if (all_var && !h->m.variant) {
    // default model, optimiser other than Adam: the whole batch in one launch of the variant kernel (+ the outer-pair recurrences)
    if (gx_var_smem_bytes(h->m.d, h->m.L, h->m.hid, h->m.emb, h->m.C) > gx_explain_max_smem()) { gx_set_error("gx_explain_nodes: model does not fit the variant kernel"); return GX_ERR_UNSUPPORTED; }
    int64_t words = 4; int maxnp = 0;
    for (const GxTask& T : h->tasks) {
      words = std::max<int64_t>(words, gx_make_var_layout(T.n, T.n2, T.e1, T.npairs_in, h->m.d, h->m.L, gx_var_row_stride(h->m.hid, h->m.emb)).total_words);
      maxnp = std::max(maxnp, T.npairs_in);
    }
    const int grid = std::min(count, h->num_sms * 4);
    const int64_t pstride = ((int64_t)maxnp * 8 + 3) / 4 * 4 + 4;
    GX_CUDA_CHECK(h->d_gws.reserve((size_t)grid * words * 4));
    GX_CUDA_CHECK(h->d_pws.reserve((size_t)grid * pstride * 4));
    GX_CUDA_CHECK(cudaEventRecord(h->ev_t0, h->stream));
    GxExplainLaunch cfg;
    cfg.order = h->d_order.as<int32_t>(); cfg.ntasks = count; cfg.counter = h->d_counters.as<int32_t>();
    cfg.smem_bytes = 0; cfg.threads = 0; cfg.grid = grid;
    cfg.gws = h->d_gws.as<float>(); cfg.gws_stride_words = words;
    cfg.pws = h->d_pws.as<float>(); cfg.pws_stride_words = pstride;
    cfg.dbg = nullptr; cfg.x = D.x;
    GX_CUDA_CHECK(gx_launch_explain_var(cfg, h->g, h->m, hd, h->plan, m0_dev, out_dev, feat_dev, h->stream));
    GX_CUDA_CHECK(gx_launch_outer_pairs(hd, h->g, h->plan, count, m0_dev, out_dev, D.x, h->stream));
    h->launches += 2;
    GX_CUDA_CHECK(cudaEventRecord(h->ev_t1, h->stream));
    h->timed = true;
    return io_finish(h, hp, space, io, count, te, h->m.d, h->m.C, D);
  }
  int stream_grid = 0;   // slabs of the streaming class = tasks in flight (CTAs of explain_stream.cu / gangs of explain_gang.cu)
  int gang = 0;          // > 0: explain_gang.cu with this many CTAs per task
  if (!h->class_order[kStreamClass].empty()) {
    // streaming class: one CTA per SM, fewer when the per-CTA slabs (node/edge state + 32 B per inner pair) would not fit
    stream_grid = std::min<int>((int)h->class_order[kStreamClass].size(), h->num_sms);
    int maxnp = 0;
    for (int32_t t : h->class_order[kStreamClass]) maxnp = std::max(maxnp, h->tasks[t].npairs_in);
    const int gang_env = h->gang_override;
    if (!h->m.variant && gang_env >= 0 && h->m.d <= 128 && gx_gang_smem_bytes(h->m.d, h->m.hid, h->m.C) <= gx_explain_max_smem()) {
      // explain_gang.cu: G co-resident CTAs per task.  As many tasks in flight as keep their randomly accessed state
      // (a, gE: 8 B per directed edge; P, dP, dY1: 240 B per node) inside the L2, the SMs divided evenly among them.
      int64_t ws = 1;
      for (int32_t t : h->class_order[kStreamClass]) ws = std::max<int64_t>(ws, (int64_t)h->tasks[t].e_d * 8 + (int64_t)h->tasks[t].n * 240);
      const int64_t l2_budget = (int64_t)80 << 20;
      int ngangs = (int)std::max<int64_t>(1, std::min<int64_t>(stream_grid, l2_budget / ws));
      gang = std::max(1, std::min(h->num_sms / ngangs, GX_MAX_GANG));
      if (gang_env > 0) gang = std::min(std::min(gang_env, h->num_sms), GX_MAX_GANG);
      ngangs = std::max(1, std::min(ngangs, h->num_sms / gang));
      stream_grid = std::min(stream_grid, ngangs);
    }
    const int64_t per_cta = (h->gws_stride_words + (int64_t)maxnp * 8 + 4) * 4;
    size_t free_b = 0, total_b = 0;
    GX_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const int64_t budget = (int64_t)(free_b + h->d_gws.cap + h->d_pws.cap) * 8 / 10;
    if (per_cta > budget) { gx_set_error("gx_explain_nodes: a task needs %lld MB of device workspace, %lld MB are free", (long long)(per_cta >> 20), (long long)(budget >> 20)); return GX_ERR_CUDA; }
    stream_grid = (int)std::max<int64_t>(1, std::min<int64_t>(stream_grid, budget / per_cta));
    GX_CUDA_CHECK(h->d_gws.reserve((size_t)stream_grid * h->gws_stride_words * 4));
  }
  // per-CTA pair-state slabs (one region per launch class, 8 floats per inner pair of its largest task)
  int64_t pws_off[kNumClasses + 1], pws_stride[kNumClasses];
  int grids[kNumClasses];
  {
    int64_t acc_words = 0;
    for (int c = 0; c < kNumClasses; ++c) {
      const int nt = (int)h->class_order[c].size();
      int maxnp = 0;
      for (int32_t t : h->class_order[c]) maxnp = std::max(maxnp, h->tasks[t].npairs_in);
      pws_stride[c] = ((int64_t)maxnp * 8 + 3) / 4 * 4;
      grids[c] = c == kStreamClass ? stream_grid : std::min<int>(nt, h->num_sms * kClasses[c].ctas_per_sm);
      const int g_cluster_size = h->plan_cluster;
      if (c == kClusterClass) grids[c] = std::min<int>(nt, h->num_sms / g_cluster_size) * g_cluster_size;   // CTAs; one pair slab per cluster
      pws_off[c] = acc_words;
      acc_words += pws_stride[c] * std::max(c == kClusterClass ? grids[c] / g_cluster_size : grids[c], 0);
    }
    pws_off[kNumClasses] = acc_words;
    GX_CUDA_CHECK(h->d_pws.reserve((size_t)std::max<int64_t>(acc_words, 4) * 4));
  }
  GX_CUDA_CHECK(cudaEventRecord(h->ev_t0, h->stream));
  GX_CUDA_CHECK(cudaEventRecord(h->ev_fork, h->stream));
  int off = 0;
  std::vector<int> used;
  for (int c = 0; c < kNumClasses; ++c) h->class_used[c] = false;
  // most expensive class first so that its long tasks start at t=0 and the small ones fill around them
  std::vector<int> offs(kNumClasses);
  for (int c = 0; c < kNumClasses; ++c) { offs[c] = off; off += (int)h->class_order[c].size(); }
  for (int c = kNumClasses - 1; c >= 0; --c) {
    const int nt = (int)h->class_order[c].size();
    if (nt == 0) continue;
    GxExplainLaunch cfg;
    cfg.order = h->d_order.as<int32_t>() + offs[c];
    cfg.ntasks = nt;
    cfg.counter = h->d_counters.as<int32_t>() + c;
    cfg.smem_bytes = kClasses[c].cap_bytes;
    cfg.threads = kClasses[c].threads;
    cfg.gws = h->d_gws.as<float>();
    cfg.gws_stride_words = h->gws_stride_words;
    cfg.dbg = h->dbg;
    cfg.x = D.x;
    cfg.pws = h->d_pws.as<float>() + pws_off[c];
    cfg.pws_stride_words = pws_stride[c];
    cfg.grid = grids[c];
    cfg.cluster = c == kClusterClass ? h->plan_cluster : 1;
    if (c != kStreamClass) {
      // shrink the dynamic smem request to what the class actually needs (more CTAs can co-reside)
      int need = 0;
      for (int32_t t : h->class_order[c]) need = std::max(need, h->tasks[t].smem_bytes);
      // the 1-per-SM class and the cluster class request the whole SM: a CTA of another class next to them would take the room the
      // scheduler's breadth-first placement needs for the small classes launched last (profiles/r02cl_cluster_auto.md)
      // (2 KB short of the class limit: kernels with a trace carry 1.2 KB of static shared memory)
      cfg.smem_bytes = (c == kOneClass || c == kClusterClass) ? std::max(need, kClasses[c].cap_bytes - 2048) : std::max(need, 1024);
    }
    GX_CUDA_CHECK(cudaStreamWaitEvent(h->side[c], h->ev_fork, 0));
    GX_CUDA_CHECK(cudaEventRecord(h->ev_begin[c], h->side[c]));
    if (c == kStreamClass && h->m.variant) {
      GX_CUDA_CHECK(gx_launch_explain_var(cfg, h->g, h->m, hd, h->plan, m0_dev, out_dev, feat_dev, h->side[c]));
    } else if (c == kStreamClass && gang > 0) {
      cfg.gang = gang;
      cfg.grid = stream_grid * gang;
      GX_CUDA_CHECK(h->d_gang.reserve((size_t)stream_grid * 16));
      GX_CUDA_CHECK(cudaMemsetAsync(h->d_gang.p, 0, (size_t)stream_grid * 16, h->side[c]));
      cfg.gang_bars = h->d_gang.as<unsigned long long>();
      cfg.gang_mail = reinterpret_cast<int32_t*>(h->d_gang.as<char>() + (size_t)stream_grid * 8);
      GX_CUDA_CHECK(gx_launch_explain_gang(cfg, h->g, h->m, hd, h->plan, m0_dev, out_dev, feat_dev, h->side[c]));
    } else if (c == kStreamClass) GX_CUDA_CHECK(gx_launch_explain_stream(cfg, h->g, h->m, hd, h->plan, m0_dev, out_dev, feat_dev, h->side[c]));
    else GX_CUDA_CHECK(gx_launch_explain(cfg, h->g, h->m, hd, h->plan, m0_dev, out_dev, feat_dev, h->side[c]));
    h->launches += 1;
    GX_CUDA_CHECK(cudaEventRecord(h->ev_join[c], h->side[c]));
    used.push_back(c);
    h->class_used[c] = true;
  }
  // pairs between two outermost nodes: independent scalar recurrences, whole batch in one launch
  GX_CUDA_CHECK(gx_launch_outer_pairs(hd, h->g, h->plan, count, m0_dev, out_dev, D.x, h->stream));
  h->launches += 1;
  for (int c : used) GX_CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_join[c], 0));
  if (D.x.trace) {
    GX_CUDA_CHECK(gx_launch_trace_finalize(hd, h->plan, count, D.x, h->stream));
    h->launches += 1;
  }
  GX_CUDA_CHECK(cudaEventRecord(h->ev_t1, h->stream));
  h->timed = true;
  if (host_timing()) fprintf(stderr, "[gnnx] gx_explain_nodes: host %.0f us from entry to the last launch\n", now_us() - t_entry);
  return io_finish(h, hp, space, io, count, te, h->m.d, h->m.C, D);
}

extern "C" {

int gx_explain_nodes(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_edges,
                     float* edge_mask, float* feat_mask) {
  gx_explain_io io;
  memset(&io, 0, sizeof(io));
  io.m0_edges = m0_edges; io.edge_mask = edge_mask; io.feat_mask = feat_mask;
  return explain_nodes_impl(h, hp, 0, space, &io);
}

int gx_explain_nodes_ex(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io) {
  return explain_nodes_impl(h, hp, 0, space, io);
}

int gx_grad_nodes(gx_handle* h, gx_memspace space, float* edge_mask) {
  gx_hparams hp;
  gx_default_hparams(&hp);
  gx_explain_io io;
  memset(&io, 0, sizeof(io));
  io.edge_mask = edge_mask;
  return explain_nodes_impl(h, &hp, 1, space, &io);
}

int gx_offedge_regularisers(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_dense, double* out) {
  if (!h || !hp || !m0_dense || !out) { gx_set_error("gx_offedge_regularisers: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_plan) { gx_set_error("gx_offedge_regularisers: no plan (call gx_plan_nodes)"); return GX_ERR_INVALID; }
  if (hp->num_epochs < 1 || hp->num_epochs > 3072) { gx_set_error("gx_offedge_regularisers: num_epochs outside [1,3072]"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->count, E = hp->num_epochs;
  std::vector<int64_t> doff(count + 1);
  int64_t acc = 0;
  for (int t = 0; t < count; ++t) { doff[t] = acc; acc += (int64_t)h->tasks[t].n * h->tasks[t].n; }
  doff[count] = acc;
  GX_CUDA_CHECK(h->d_dense_off.reserve((size_t)(count + 1) * 8));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_dense_off.p, doff.data(), (size_t)(count + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  GxHparamsDev hd;
  fill_hparams(h, hp, 0, false, &hd);
  if (hp->opt != GX_OPT_ADAM) { gx_set_error("gx_offedge_regularisers: the off-edge trajectories are built for Adam only"); return GX_ERR_UNSUPPORTED; }
  int rc = check_optimiser("gx_offedge_regularisers", hp);
  if (rc != GX_OK) return rc;
  rc = upload_adam_table(h, hp, E, 0);
  if (rc != GX_OK) return rc;
  hd.adam_tab = h->d_adam.as<float2>();
  const float* m0d = m0_dense;
  double* od = out;
  const size_t nout = (size_t)count * E * 2;
  if (space == GX_HOST) {
    GX_CUDA_CHECK(h->d_m0dense.reserve((size_t)std::max<int64_t>(acc, 1) * 4));
    GX_CUDA_CHECK(cudaMemcpyAsync(h->d_m0dense.p, m0_dense, (size_t)acc * 4, cudaMemcpyHostToDevice, h->stream));
    GX_CUDA_CHECK(h->d_offedge.reserve(nout * 8));
    m0d = h->d_m0dense.as<float>();
    od = h->d_offedge.as<double>();
  }
  GX_CUDA_CHECK(cudaMemsetAsync(od, 0, nout * 8, h->stream));
  GX_CUDA_CHECK(gx_launch_offedge(hd, h->plan, count, E, h->d_dense_off.as<int64_t>(), m0d, od, h->stream));
  h->launches += 1;
  if (space == GX_HOST) GX_CUDA_CHECK(cudaMemcpyAsync(out, od, nout * 8, cudaMemcpyDeviceToHost, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));   // doff (host vector) was copied asynchronously
  return GX_OK;
}

int gx_set_graph_batch_csr(gx_handle* h, int32_t G, int32_t max_nodes, const int32_t* rowptr, const int32_t* col,
                           const float* feat, int32_t d, const int32_t* label) {
  if (!h || !rowptr || !col || !feat || !label) { gx_set_error("gx_set_graph_batch_csr: NULL argument"); return GX_ERR_INVALID; }
  if (G < 1 || max_nodes < 1 || max_nodes > 4096) { gx_set_error("gx_set_graph_batch_csr: num_graphs/max_nodes out of range (max_nodes <= 4096)"); return GX_ERR_INVALID; }
  const int64_t R = (int64_t)G * max_nodes;
  if (rowptr[0] != 0) { gx_set_error("gx_set_graph_batch_csr: rowptr[0] != 0"); return GX_ERR_INVALID; }
  for (int64_t r = 0; r < R; ++r) {
    if (rowptr[r + 1] < rowptr[r]) { gx_set_error("gx_set_graph_batch_csr: rowptr not monotone"); return GX_ERR_INVALID; }
    const int64_t g0 = r / max_nodes * max_nodes;
    const int32_t i = (int32_t)(r - g0);
    for (int64_t e = rowptr[r]; e < rowptr[r + 1]; ++e) {
      const int32_t j = col[e];
      if (j < 0 || j >= max_nodes) { gx_set_error("gx_set_graph_batch_csr: col out of range"); return GX_ERR_INVALID; }
      if (e > rowptr[r] && col[e] <= col[e - 1]) { gx_set_error("gx_set_graph_batch_csr: columns not strictly ascending"); return GX_ERR_INVALID; }
      if (j == i) { gx_set_error("gx_set_graph_batch_csr: self loops are not supported in graph mode"); return GX_ERR_UNSUPPORTED; }
      if (!std::binary_search(col + rowptr[g0 + j], col + rowptr[g0 + j + 1], i)) { gx_set_error("gx_set_graph_batch_csr: adjacency not symmetric"); return GX_ERR_UNSUPPORTED; }
    }
  }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int64_t nnz = rowptr[R];
  GX_CUDA_CHECK(h->gb_rowptr.reserve((size_t)(R + 1) * 4));
  GX_CUDA_CHECK(h->gb_col.reserve((size_t)std::max<int64_t>(nnz, 1) * 4));
  GX_CUDA_CHECK(h->gb_feat.reserve((size_t)R * d * 4));
  GX_CUDA_CHECK(h->gb_label.reserve((size_t)G * 4));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->gb_rowptr.p, rowptr, (size_t)(R + 1) * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->gb_col.p, col, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->gb_feat.p, feat, (size_t)R * d * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->gb_label.p, label, (size_t)G * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->gb_h_rowptr.assign(rowptr, rowptr + R + 1);
  h->gb_h_label.assign(label, label + G);
  h->gb.num_graphs = G; h->gb.max_nodes = max_nodes; h->gb.d = d;
  h->gb.rowptr = h->gb_rowptr.as<int32_t>(); h->gb.col = h->gb_col.as<int32_t>();
  h->gb.feat = h->gb_feat.as<float>(); h->gb.label = h->gb_label.as<int32_t>();
  h->has_batch = true; h->has_gplan = false;
  return GX_OK;
}

int gx_plan_graphs(gx_handle* h, const int32_t* graph_ids, int32_t count, int64_t* edge_off, int64_t* total_edges) {
  if (!h || !graph_ids) { gx_set_error("gx_plan_graphs: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_batch || !h->has_model) { gx_set_error("gx_plan_graphs: call gx_set_model and gx_set_graph_batch_csr first"); return GX_ERR_INVALID; }
  if (h->gb.d != h->m.d) { gx_set_error("gx_plan_graphs: feat_dim %d != model input_dim %d", h->gb.d, h->m.d); return GX_ERR_INVALID; }
  if (count <= 0) { gx_set_error("gx_plan_graphs: count <= 0"); return GX_ERR_INVALID; }
  if (gx_graph_var_smem_bytes(h->m.d, h->m.L, h->m.hid, h->m.emb, h->m.C) > gx_explain_max_smem()) {
    gx_set_error("gx_plan_graphs: model does not fit the shared memory of the graph-mode variant kernel"); return GX_ERR_UNSUPPORTED;
  }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  h->has_gplan = false; h->has_plan = false;
  const int nf = h->gb.max_nodes;
  const int vw = gx_graph_var_row_stride(h->m.hid, h->m.emb);
  h->tasks.assign(count, GxTask());
  std::vector<int64_t> var_words(count);
  std::vector<char> in_smem(count);
  int64_t tn = 0, te = 0, tp = 0;
  int max_smem = 0, max_np = 0;
  const int nwarps = 128 / 32;
  for (int t = 0; t < count; ++t) {
    const int g = graph_ids[t];
    if (g < 0 || g >= h->gb.num_graphs) { gx_set_error("gx_plan_graphs: graph %d out of range", g); return GX_ERR_INVALID; }
    const int32_t* rp = h->gb_h_rowptr.data() + (int64_t)g * nf;
    GxTask& T = h->tasks[t];
    memset(&T, 0, sizeof(T));
    int na = 0;
    for (int i = 0; i < nf; ++i) na += rp[i + 1] > rp[i] ? 1 : 0;
    T.node = g; T.n = na; T.n1 = na; T.n2 = na;
    T.e_d = rp[nf] - rp[0]; T.e1 = T.e_d; T.npairs = T.e_d / 2; T.npairs_in = T.npairs;
    T.gt_label = h->gb_h_label[g]; T.n_norm = nf; T.flags = na < nf ? 1 : 0;
    T.node_off = tn; T.rp_off = tn + t; T.edge_off = te; T.pair_off = tp;
    var_words[t] = gx_make_graph_var_layout(na, T.e_d, T.npairs, h->m.d, h->m.L, vw).total_words;
    // the tuned shared-memory kernel takes the default model's graphs that fit its layout (16-bit indices, 226 KB); the rest goes to
    // explain_graph_var.cu
    in_smem[t] = !h->m.variant && na < 65535 && T.e_d < 65535;
    if (in_smem[t]) {
      const GxLayoutG L = gx_make_layout_graph(na, T.e_d, T.npairs, h->m.d, h->m.hid, h->m.emb, h->m.C, nwarps);
      T.smem_bytes = L.total_words * 4;
      in_smem[t] = T.smem_bytes <= 226 * 1024;
    }
    if (!in_smem[t]) T.smem_bytes = 0;
    else max_smem = std::max(max_smem, T.smem_bytes);
    max_np = std::max(max_np, T.npairs);
    tn += na; te += T.e_d; tp += T.npairs;
  }
  // Launch classes by footprint: a batch padded to 100 nodes mostly holds 20-40-node molecules; one launch sized for the largest graph
  // left 3 CTAs per SM where 5-11 fit (~12 KB of every footprint are the weights).  Classes <= 18 / 27 / 36 / 44 / 80 / 226 KB ->
  // 11 / 8 / 6 / 5 / 2 / 1 CTAs per SM (each launch requests its class's largest footprint), most expensive first inside a class.
  static const int kGraphCap[6] = {18 * 1024, 27 * 1024, 36 * 1024, 44 * 1024, 80 * 1024, 226 * 1024};
  std::vector<int32_t> cls_tasks[6];
  for (int c = 0; c < 6; ++c) { h->g_class_n[c] = 0; h->g_class_smem[c] = 0; h->g_class_np[c] = 0; }
  for (int t = 0; t < count; ++t) {
    if (!in_smem[t]) continue;
    int c = 0;
    while (c < 5 && h->tasks[t].smem_bytes > kGraphCap[c]) ++c;
    cls_tasks[c].push_back(t);
    h->g_class_smem[c] = std::max(h->g_class_smem[c], h->tasks[t].smem_bytes);
    h->g_class_np[c] = std::max(h->g_class_np[c], h->tasks[t].npairs);
  }
  auto costlier = [&](int32_t x, int32_t y) { return h->tasks[x].e_d + 4 * h->tasks[x].n > h->tasks[y].e_d + 4 * h->tasks[y].n; };
  std::vector<int32_t> order;
  order.reserve(2 * (size_t)count);
  for (int c = 0; c < 6; ++c) {
    std::stable_sort(cls_tasks[c].begin(), cls_tasks[c].end(), costlier);
    h->g_class_n[c] = (int)cls_tasks[c].size();
    order.insert(order.end(), cls_tasks[c].begin(), cls_tasks[c].end());
  }
  // explain_graph_var.cu: a small-slab class (molecules: many CTAs per SM, slabs in L2) and a large-slab class (a few hundred nodes and
  // more: few CTAs, so that one 4 000-node graph does not size the slab of every CTA of the grid).  Routing [0]: the tasks above;
  // routing [1]: every task (optimisers other than Adam).
  for (int r = 0; r < 2; ++r) {
    std::vector<int32_t> cv[2];
    for (int t = 0; t < count; ++t)
      if (r == 1 || !in_smem[t]) cv[var_words[t] > kGraphVarSmallWords ? 1 : 0].push_back(t);
    h->gv_off[r] = (int)order.size();
    for (int c = 0; c < 2; ++c) {
      std::stable_sort(cv[c].begin(), cv[c].end(), costlier);
      h->gv_n[r][c] = (int)cv[c].size();
      h->gv_words[r][c] = 4;
      for (int32_t t : cv[c]) h->gv_words[r][c] = std::max(h->gv_words[r][c], var_words[t]);
      order.insert(order.end(), cv[c].begin(), cv[c].end());
    }
  }
  GX_CUDA_CHECK(h->d_tasks.reserve((size_t)count * sizeof(GxTask)));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_tasks.p, h->tasks.data(), (size_t)count * sizeof(GxTask), cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(h->d_order.reserve(order.size() * 4));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_order.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(h->d_counters.reserve(kNumStreams * 4));
  GX_CUDA_CHECK(h->d_lo2gid.reserve((size_t)std::max<int64_t>(tn, 1) * 4));
  GX_CUDA_CHECK(h->d_irp.reserve((size_t)(tn + count) * 4));
  GX_CUDA_CHECK(h->d_icol.reserve((size_t)std::max<int64_t>(te, 1) * 4));
  GX_CUDA_CHECK(h->d_pairs.reserve((size_t)std::max<int64_t>(tp, 1) * 4 * 6));
  h->plan = GxPlanArrays();
  h->plan.tasks = h->d_tasks.as<GxTask>();
  h->plan.lo2gid = h->d_lo2gid.as<int32_t>();
  h->plan.irowptr = h->d_irp.as<int32_t>();
  h->plan.icol = h->d_icol.as<int32_t>();
  int32_t* pb = h->d_pairs.as<int32_t>();
  h->plan.pair_i = pb; h->plan.pair_j = pb + tp; h->plan.pair_pij = pb + 2 * tp;
  h->plan.pair_pji = pb + 3 * tp; h->plan.pair_oij = pb + 4 * tp; h->plan.pair_oji = pb + 5 * tp;
  GX_CUDA_CHECK(gx_launch_graph_plan(h->gb, count, h->plan, h->stream));
  h->launches += 1;
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->g_count = count; h->g_total_e = te; h->g_max_smem = max_smem; h->g_max_np = max_np;
  h->count = count; h->total_e = te;
  h->has_gplan = true;
  if (edge_off) { for (int t = 0; t < count; ++t) edge_off[t] = h->tasks[t].edge_off; edge_off[count] = te; }
  if (total_edges) *total_edges = te;
  return GX_OK;
}

static int explain_graphs_impl(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io) {
  if (!h || !hp) { gx_set_error("gx_explain_graphs: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_gplan) { gx_set_error("gx_explain_graphs: no plan (call gx_plan_graphs)"); return GX_ERR_INVALID; }
  if (hp->mask_act != 0) { gx_set_error("gx_explain_graphs: mask_act != sigmoid is not built (the reference's ReLU variant returns NaN masks)"); return GX_ERR_UNSUPPORTED; }
  if (hp->num_epochs < 1) { gx_set_error("gx_explain_graphs: num_epochs < 1"); return GX_ERR_INVALID; }
  if (hp->init != GX_INIT_M0 && hp->init != GX_INIT_PHILOX && hp->init != GX_INIT_STATE) { gx_set_error("gx_explain_graphs: unknown init %d", hp->init); return GX_ERR_INVALID; }
  int rc = check_optimiser("gx_explain_graphs", hp);
  if (rc != GX_OK) return rc;
  // routing [1]: optimisers other than Adam run the whole batch in explain_graph_var.cu; [0]: Adam, the variant kernel takes the
  // tasks explain_graph.cu does not (model variants, graphs beyond its shared-memory layout)
  const int route = hp->opt != GX_OPT_ADAM ? 1 : 0;
  const bool any_var = h->gv_n[route][0] + h->gv_n[route][1] > 0;
  if (any_var && (hp->init == GX_INIT_STATE || (io && (io->trace || io->trace_pred || io->adam_m_out || io->adam_v_out || io->mask_param_out || io->feat_state_out)))) {
    gx_set_error("gx_explain_graphs: model variants (num_layers != 3 / --bn / widths > 32), optimisers other than Adam and graphs beyond the shared-memory kernel "
                 "build the mask optimisation only (no trace or optimiser state)");
    return GX_ERR_UNSUPPORTED;
  }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->g_count;
  const int64_t te = h->g_total_e;
  IoDev D;
  rc = io_prepare(h, "gx_explain_graphs", hp, 0, space, io, count, te, h->m.d, h->m.C, &D);
  if (rc != GX_OK) return rc;
  D.x.tr_outer = nullptr;   // graph mode has no outer pairs
  GxHparamsDev hd;
  fill_hparams(h, hp, 0, D.x.trace != nullptr, &hd);
  hd.c_lap = 0.f;           // lap_loss = 0 in graph mode (explain.py:787-788)
  rc = upload_adam_table(h, hp, hd.iters, hp->start_step);
  if (rc != GX_OK) return rc;
  hd.adam_tab = h->d_adam.as<float2>();
  // one persistent launch per footprint class, on its own stream (the classes overlap like the node-mode classes)
  int grids[6]; int64_t pstride[6], poff[7] = {};
  for (int c = 0; c < 6; ++c) {
    const int nt = route == 0 ? h->g_class_n[c] : 0;
    const int smem_c = std::max(h->g_class_smem[c], 1024);
    const int per_sm = std::max(1, std::min(16, (227 * 1024) / (smem_c + 1024)));
    grids[c] = std::min(nt, h->num_sms * per_sm);
    pstride[c] = ((int64_t)h->g_class_np[c] * 8 + 3) / 4 * 4;
    poff[c + 1] = poff[c] + pstride[c] * grids[c];
  }
  GX_CUDA_CHECK(h->d_pws.reserve((size_t)std::max<int64_t>(poff[6], 4) * 4));
  // explain_graph_var.cu: one slab per CTA, sized by the class's largest graph; 8 CTAs per SM of 128 threads (fewer when the weights
  // take the shared memory), the large-slab class 2 per SM and no more than 80% of the free device memory
  int vgrid[2] = {0, 0}; int64_t voff[3] = {0, 0, 0};
  if (any_var) {
    const int vsm = gx_graph_var_smem_bytes(h->m.d, h->m.L, h->m.hid, h->m.emb, h->m.C);
    const int per_sm = std::max(1, std::min(8, (227 * 1024) / (vsm + 1024)));
    size_t free_b = 0, total_b = 0;
    GX_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const int64_t budget = (int64_t)(free_b + h->d_gws.cap) / 4 * 8 / 10;   // words
    for (int c = 0; c < 2; ++c) {
      const int nt = h->gv_n[route][c];
      voff[c + 1] = voff[c];
      if (nt == 0) continue;
      const int64_t words = h->gv_words[route][c];
      const int64_t room = c == 0 ? budget / 2 : budget - voff[1];   // the small class leaves at least half of the budget to the large one
      const int grid = (int)std::min<int64_t>(std::min(nt, h->num_sms * (c == 0 ? per_sm : std::min(per_sm, 2))), room / words);
      if (grid < 1) { gx_set_error("gx_explain_graphs: a graph needs %lld MB of device workspace", (long long)(words * 4 >> 20)); return GX_ERR_CUDA; }
      vgrid[c] = grid;
      voff[c + 1] = voff[c] + words * grid;
    }
    GX_CUDA_CHECK(h->d_gws.reserve((size_t)std::max<int64_t>(voff[2], 4) * 4));
  }
  GX_CUDA_CHECK(cudaMemsetAsync(h->d_counters.p, 0, kNumStreams * 4, h->stream));
  GX_CUDA_CHECK(cudaEventRecord(h->ev_t0, h->stream));
  GX_CUDA_CHECK(cudaEventRecord(h->ev_fork, h->stream));
  int offs[6];
  for (int c = 0, acc = 0; c < 6; ++c) { offs[c] = acc; acc += h->g_class_n[c]; }
  for (int c = 1; c >= 0; --c) {   // large graphs first
    if (vgrid[c] == 0) continue;
    const int sidx = 6 + c;
    GxExplainLaunch cfg;
    cfg.order = h->d_order.as<int32_t>() + h->gv_off[route] + (c == 1 ? h->gv_n[route][0] : 0);
    cfg.ntasks = h->gv_n[route][c]; cfg.counter = h->d_counters.as<int32_t>() + sidx;
    cfg.smem_bytes = 0; cfg.threads = 0; cfg.grid = vgrid[c];
    cfg.gws = h->d_gws.as<float>() + voff[c]; cfg.gws_stride_words = h->gv_words[route][c];
    cfg.pws = nullptr; cfg.pws_stride_words = 0; cfg.dbg = nullptr;
    cfg.x = D.x;
    GX_CUDA_CHECK(cudaStreamWaitEvent(h->side[sidx], h->ev_fork, 0));
    GX_CUDA_CHECK(gx_launch_explain_graph_var(cfg, h->gb, h->m, hd, h->plan, D.m0, D.out, D.feat, h->side[sidx]));
    GX_CUDA_CHECK(cudaEventRecord(h->ev_join[sidx], h->side[sidx]));
    GX_CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_join[sidx], 0));
    h->launches += 1;
  }
  for (int c = 5; c >= 0; --c) {   // largest graphs first
    if (grids[c] == 0) continue;
    GxExplainLaunch cfg;
    cfg.order = h->d_order.as<int32_t>() + offs[c]; cfg.ntasks = h->g_class_n[c]; cfg.counter = h->d_counters.as<int32_t>() + c;
    cfg.smem_bytes = std::max(h->g_class_smem[c], 1024);
    cfg.threads = 128;
    cfg.grid = grids[c];
    cfg.gws = nullptr; cfg.gws_stride_words = 0; cfg.dbg = nullptr;
    cfg.x = D.x;
    cfg.pws_stride_words = pstride[c];
    cfg.pws = h->d_pws.as<float>() + poff[c];
    GX_CUDA_CHECK(cudaStreamWaitEvent(h->side[c], h->ev_fork, 0));
    GX_CUDA_CHECK(gx_launch_explain_graphs(cfg, h->gb, h->m, hd, h->plan, D.m0, D.out, D.feat, h->side[c]));
    GX_CUDA_CHECK(cudaEventRecord(h->ev_join[c], h->side[c]));
    GX_CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_join[c], 0));
    h->launches += 1;
  }
  if (D.x.trace) {
    GX_CUDA_CHECK(gx_launch_trace_finalize(hd, h->plan, count, D.x, h->stream));
    h->launches += 1;
  }
  GX_CUDA_CHECK(cudaEventRecord(h->ev_t1, h->stream));
  h->timed = true;
  return io_finish(h, hp, space, io, count, te, h->m.d, h->m.C, D);
}

int gx_explain_graphs(gx_handle* h, const gx_hparams* hp, gx_memspace space, const float* m0_edges,
                      float* edge_mask, float* feat_mask) {
  gx_explain_io io;
  memset(&io, 0, sizeof(io));
  io.m0_edges = m0_edges; io.edge_mask = edge_mask; io.feat_mask = feat_mask;
  return explain_graphs_impl(h, hp, space, &io);
}

int gx_explain_graphs_ex(gx_handle* h, const gx_hparams* hp, gx_memspace space, const gx_explain_io* io) {
  return explain_graphs_impl(h, hp, space, io);
}

int gx_comm_unique_id(char id[128]) {
  if (!id) { gx_set_error("gx_comm_unique_id: NULL argument"); return GX_ERR_INVALID; }
  return gx_comm_impl_unique_id(id);
}

int gx_comm_init(gx_handle* h, int32_t world, int32_t rank, const char id[128]) {
  if (!h || !id) { gx_set_error("gx_comm_init: NULL argument"); return GX_ERR_INVALID; }
  if (world < 1 || rank < 0 || rank >= world) { gx_set_error("gx_comm_init: rank %d outside [0,%d)", rank, world); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  gx_comm_impl_destroy(h->comm);
  h->comm = nullptr;
  return gx_comm_impl_init(&h->comm, world, rank, id);
}

int gx_comm_destroy(gx_handle* h) {
  if (!h) return GX_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  gx_comm_impl_destroy(h->comm);
  h->comm = nullptr;
  return GX_OK;
}

int gx_count_nodes(gx_handle* h, const int32_t* nodes, int32_t count, int32_t n_hops, int32_t* n_out, int32_t* e_out) {
  if (!h || !nodes) { gx_set_error("gx_count_nodes: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_graph) { gx_set_error("gx_count_nodes: call gx_set_graph_csr first"); return GX_ERR_INVALID; }
  if (n_hops < 1 || n_hops >= GX_MAX_LEVELS) { gx_set_error("gx_count_nodes: n_hops=%d outside [1,%d]", n_hops, GX_MAX_LEVELS - 1); return GX_ERR_INVALID; }
  if (count <= 0) return GX_OK;
  for (int t = 0; t < count; ++t)
    if (nodes[t] < 0 || nodes[t] >= h->g.N) { gx_set_error("gx_count_nodes: node %d out of range", nodes[t]); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  int rc = ensure_slot_ws(h);
  if (rc != GX_OK) return rc;
  h->has_plan = false;     // the task buffer is shared with the plan
  GX_CUDA_CHECK(h->d_nodes.reserve((size_t)count * 4));
  GX_CUDA_CHECK(h->d_tasks.reserve((size_t)count * sizeof(GxTask)));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_nodes.p, nodes, (size_t)count * 4, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(gx_launch_khop_count(h->g, h->d_nodes.as<int32_t>(), count, n_hops, h->has_model ? h->m.L - 1 : 2, h->ws, h->d_tasks.as<GxTask>(), h->stream));
  h->launches += 1;
  std::vector<GxTask> tk(count);
  GX_CUDA_CHECK(cudaMemcpyAsync(tk.data(), h->d_tasks.p, (size_t)count * sizeof(GxTask), cudaMemcpyDeviceToHost, h->stream));
  GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  for (int t = 0; t < count; ++t) { if (n_out) n_out[t] = tk[t].n; if (e_out) e_out[t] = tk[t].e_d; }
  return GX_OK;
}

int gx_allgather_masks(gx_handle* h, const float* local_dev, int64_t local_floats, int64_t slot_floats, float* gathered_dev) {
  if (!h || !gathered_dev || (local_floats > 0 && !local_dev)) { gx_set_error("gx_allgather_masks: NULL argument"); return GX_ERR_INVALID; }
  if (!h->comm) { gx_set_error("gx_allgather_masks: no communicator (call gx_comm_init)"); return GX_ERR_INVALID; }
  if (local_floats < 0 || slot_floats < local_floats || slot_floats < 1) { gx_set_error("gx_allgather_masks: need 0 <= local_floats <= slot_floats"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  // the send slot: this rank's values, zero padded to the common slot size (in place inside the receive buffer: NCCL's in-place all-gather)
  float* mine = gathered_dev + (int64_t)gx_comm_impl_rank(h->comm) * slot_floats;
  if (local_floats > 0 && mine != local_dev)
    GX_CUDA_CHECK(cudaMemcpyAsync(mine, local_dev, (size_t)local_floats * 4, cudaMemcpyDeviceToDevice, h->stream));
  if (slot_floats > local_floats)
    GX_CUDA_CHECK(cudaMemsetAsync(mine + local_floats, 0, (size_t)(slot_floats - local_floats) * 4, h->stream));
  return gx_comm_impl_allgather(h->comm, mine, gathered_dev, (size_t)slot_floats, h->stream);
}

int gx_unshard_masks(gx_handle* h, const float* gathered_dev, int32_t items, const int64_t* src_off, const int64_t* dst_off,
                     const int32_t* sizes, float* out_dev) {
  if (!h || !gathered_dev || !src_off || !dst_off || !sizes || !out_dev) { gx_set_error("gx_unshard_masks: NULL argument"); return GX_ERR_INVALID; }
  if (items <= 0) return GX_OK;
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const size_t b64 = (size_t)items * 8, b32 = (size_t)items * 4;
  GX_CUDA_CHECK(h->d_us.reserve(2 * b64 + b32));
  char* b = h->d_us.as<char>();
  GX_CUDA_CHECK(cudaMemcpyAsync(b, src_off, b64, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(b + b64, dst_off, b64, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(cudaMemcpyAsync(b + 2 * b64, sizes, b32, cudaMemcpyHostToDevice, h->stream));
  GX_CUDA_CHECK(gx_launch_unshard(gathered_dev, items, (const int64_t*)b, (const int64_t*)(b + b64), (const int32_t*)(b + 2 * b64), out_dev, h->stream));
  h->launches += 1;
  return GX_OK;
}

int gx_denoise_topk(gx_handle* h, gx_memspace space, const float* edge_mask, int32_t threshold_num, int32_t cap,
                    float* out_threshold, int32_t* out_count, int32_t* out_slots, float* out_vals) {
  if (!h || !edge_mask || !out_threshold || !out_count || !out_slots) { gx_set_error("gx_denoise_topk: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_plan) { gx_set_error("gx_denoise_topk: no plan (call gx_plan_nodes)"); return GX_ERR_INVALID; }
  if (threshold_num < 1 || cap < 1) { gx_set_error("gx_denoise_topk: threshold_num and cap must be >= 1"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->count;
  const float* em = edge_mask;
  float* thr = out_threshold; int32_t* cnt = out_count; int32_t* slots = out_slots; float* vals = out_vals;
  if (space == GX_HOST) {
    GX_CUDA_CHECK(h->d_out.reserve((size_t)std::max<int64_t>(h->total_e, 1) * 4));
    GX_CUDA_CHECK(cudaMemcpyAsync(h->d_out.p, edge_mask, (size_t)h->total_e * 4, cudaMemcpyHostToDevice, h->stream));
    GX_CUDA_CHECK(h->d_dn_thr.reserve((size_t)count * 4)); GX_CUDA_CHECK(h->d_dn_cnt.reserve((size_t)count * 4));
    GX_CUDA_CHECK(h->d_dn_slots.reserve((size_t)count * cap * 4));
    if (out_vals) GX_CUDA_CHECK(h->d_dn_vals.reserve((size_t)count * cap * 4));
    em = h->d_out.as<float>(); thr = h->d_dn_thr.as<float>(); cnt = h->d_dn_cnt.as<int32_t>(); slots = h->d_dn_slots.as<int32_t>();
    vals = out_vals ? h->d_dn_vals.as<float>() : nullptr;
  }
  GX_CUDA_CHECK(cudaMemsetAsync(slots, 0xFF, (size_t)count * cap * 4, h->stream));   // unused entries read as -1
  GX_CUDA_CHECK(gx_launch_denoise_topk(h->plan, count, em, 2 * threshold_num, cap, thr, cnt, slots, vals, h->stream));
  h->launches += 1;
  if (space == GX_HOST) {
    GX_CUDA_CHECK(cudaMemcpyAsync(out_threshold, thr, (size_t)count * 4, cudaMemcpyDeviceToHost, h->stream));
    GX_CUDA_CHECK(cudaMemcpyAsync(out_count, cnt, (size_t)count * 4, cudaMemcpyDeviceToHost, h->stream));
    GX_CUDA_CHECK(cudaMemcpyAsync(out_slots, slots, (size_t)count * cap * 4, cudaMemcpyDeviceToHost, h->stream));
    if (out_vals) GX_CUDA_CHECK(cudaMemcpyAsync(out_vals, vals, (size_t)count * cap * 4, cudaMemcpyDeviceToHost, h->stream));
    GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  }
  return GX_OK;
}

int gx_densify(gx_handle* h, gx_memspace space, const float* edge_mask, double* out) {
  if (!h || !edge_mask || !out) { gx_set_error("gx_densify: NULL argument"); return GX_ERR_INVALID; }
  if (!h->has_plan) { gx_set_error("gx_densify: no plan"); return GX_ERR_INVALID; }
  GX_CUDA_CHECK(cudaSetDevice(h->device));
  const int count = h->count;
  std::vector<int64_t> doff(count + 1);
  int64_t acc = 0;
  for (int t = 0; t < count; ++t) { doff[t] = acc; acc += (int64_t)h->tasks[t].n * h->tasks[t].n; }
  doff[count] = acc;
  GX_CUDA_CHECK(h->d_dense_off.reserve((size_t)(count + 1) * 8));
  GX_CUDA_CHECK(cudaMemcpyAsync(h->d_dense_off.p, doff.data(), (size_t)(count + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  const float* em = edge_mask;
  double* o = out;
  if (space == GX_HOST) {
    GX_CUDA_CHECK(h->d_out.reserve((size_t)std::max<int64_t>(h->total_e, 1) * 4));
    GX_CUDA_CHECK(cudaMemcpyAsync(h->d_out.p, edge_mask, (size_t)h->total_e * 4, cudaMemcpyHostToDevice, h->stream));
    GX_CUDA_CHECK(h->d_dense.reserve((size_t)std::max<int64_t>(acc, 1) * 8));
    em = h->d_out.as<float>();
    o = h->d_dense.as<double>();
  }
  GX_CUDA_CHECK(gx_launch_densify(h->plan, count, h->d_dense_off.as<int64_t>(), em, o, h->stream));
  h->launches += 1;
  if (space == GX_HOST) {
    GX_CUDA_CHECK(cudaMemcpyAsync(out, o, (size_t)acc * 8, cudaMemcpyDeviceToHost, h->stream));
    GX_CUDA_CHECK(cudaStreamSynchronize(h->stream));
  }
  return GX_OK;
}

}  // extern "C"
