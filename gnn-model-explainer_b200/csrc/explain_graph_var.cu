// explain_graph_var.cu -- graph-classification mode (SURVEY.md section 8 row f1) for everything explain_graph.cu does not build:
//   * the model variants of GcnEncoderGraph (models.py:84-316): num_gc_layers 2 / 3 / 4, --bn (a fresh BatchNorm1d(n) in train mode
//     after the ReLU of every hidden layer = per-node standardisation over the feature axis, eps 1e-5, biased variance), hidden /
//     output widths 1 .. 128 at their true width, d <= 128, any number of classes;
//   * the optimisers other than Adam (utils/train_utils.py:7-23), every model;
//   * graphs whose state does not fit the 226 KB shared-memory layout of explain_graph.cu (up to max_nodes = 4096).
// It computes the closed-form specification of graph mode (SURVEY.md section 8a, graph_mode=True, optional bn): no receptive-field
// pruning (every row with an edge at every layer), rows without an edge (padding, isolated atoms) represented by one constant
// post_l(normalize(b_l)) that joins every max-pool, readout = per-layer column max with first-arg-max routing of dEmb, concat, Linear,
// softmax, -log p[graph label]; every edge gets the SDDMM terms of all L layers; no Laplacian term; the 1/n^2 of the entropy term
// and the std of M0 use the PADDED size.
// One persistent CTA per graph, all epochs in one launch; the per-graph state lives in a per-CTA global slab (L2 resident for
// molecule-sized graphs), the weights in shared memory.  One warp per row with lane = feature (KW chunks of 32), one thread per
// undirected edge in the edge phase.  Phases per epoch (one __syncthreads each): F1 .. FL | pool | S | BL .. B1 | P.
#include "explain_common.cuh"

namespace {

constexpr int kGvThreads = 128;
constexpr int kGvWeightWords = 36 * 1024;   // conv weights are staged in shared memory up to this many floats (144 KB), read through L2 beyond

__host__ __device__ inline int gv_kw(int hid, int emb) { const int w = hid > emb ? hid : emb; return w <= 32 ? 1 : (w <= 64 ? 2 : 4); }

struct GvSmem { int W[GX_MAX_LAYERS], b[GX_MAX_LAYERS], Wp, sF, F, mF, vF, zs, zlen, gFp, cst, emb, dEmb, arg, logit, w_in_smem, total; };
__host__ __device__ inline GvSmem gv_smem(int d, int L, int hid, int emb, int C, int nwarps) {
  GvSmem S;
  const int dp = gx_round_up(d, 4);
  int o = 0;
  auto take = [&](int words) { int r = o; o += gx_round_up(words, 4); return r; };
  int wwords = 0;
  for (int l = 0; l < L; ++l) wwords += (l == 0 ? d : hid) * (l == L - 1 ? emb : hid);
  S.w_in_smem = wwords <= kGvWeightWords;
  for (int l = 0; l < L; ++l) {
    const int win = l == 0 ? d : hid, wout = l == L - 1 ? emb : hid;
    S.W[l] = take(S.w_in_smem ? win * wout : 0);
    S.b[l] = take(wout);
  }
  const int PD = hid * (L - 1) + emb;
  S.Wp = take(C * (PD + 1) <= GX_WP_SMEM_MAX ? C * (PD + 1) : 0);
  S.sF = take(dp); S.F = take(dp); S.mF = take(dp); S.vF = take(dp);
  S.zlen = dp > 32 * gv_kw(hid, emb) ? dp : 32 * gv_kw(hid, emb);   // per-warp scratch row: a feature row or a hidden row
  S.zs = take(nwarps * S.zlen);
  S.gFp = take(nwarps * dp);
  S.cst = take(PD); S.emb = take(PD); S.dEmb = take(PD);
  S.arg = take(PD);   // int: arg-max row of every pooled feature (-1: the edge-less constant)
  S.logit = take(C < 32 ? 32 : C);
  S.total = o;
  return S;
}

struct GraphVarArgs {
  const int32_t* order;
  int32_t ntasks;
  int32_t* counter;
  float* gws;
  int64_t gws_stride_words;
  GxGraphBatchDev gb;
  GxModelDev m;
  GxHparamsDev hp;
  GxPlanArrays plan;
  const float* m0;
  float* out_mask;
  float* out_feat;
};

// 8 CTAs per SM (64 registers) for widths <= 64; the 128-wide rows (4 chunks per lane) get 128 registers
template <bool kBn, int KW>
__global__ void __launch_bounds__(kGvThreads, KW == 4 ? 4 : 8) explain_graph_var_kernel(const GraphVarArgs A) {
  extern __shared__ __align__(16) float sm[];
  __shared__ int s_task;
  __shared__ const float* s_W[GX_MAX_LAYERS];   // per layer: conv weights (shared memory when they fit, else global, L2 resident)
  __shared__ const float* s_b[GX_MAX_LAYERS];   // per layer: bias (shared memory)
  constexpr int NT = kGvThreads, nwarps = NT / 32;
  constexpr int VW = 32 * KW;   // row stride of every hidden-width array
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const GxModelDev& m = A.m;
  const GxHparamsDev& hp = A.hp;
  const int d = m.d, C = m.C, L = m.L, hid = m.hid, embw = m.emb;
  const int dp = gx_round_up(d, 4);
  const int PD = hid * (L - 1) + embw;
  const bool ieee = (hp.flags & GX_HP_IEEE_EDGE) != 0;
  const GvSmem S = gv_smem(d, L, hid, embw, C, nwarps);
  float* const sF = sm + S.sF; float* const Fm = sm + S.F; float* const mF = sm + S.mF; float* const vF = sm + S.vF;
  float* const zs = sm + S.zs + warp * S.zlen;
  float* const gFp = sm + S.gFp;
  float* const cst = sm + S.cst; float* const emb = sm + S.emb; float* const dEmb = sm + S.dEmb; float* const logit = sm + S.logit;
  int* const arg = reinterpret_cast<int*>(sm + S.arg);
  const bool wp_smem = C * (PD + 1) <= GX_WP_SMEM_MAX;
  const float* const Wpp = wp_smem ? sm + S.Wp : m.Wp;
  const float* const bpp = wp_smem ? sm + S.Wp + C * PD : m.bp;
  auto win_of = [&](int l) { return l == 0 ? d : hid; };            // l = 0 .. L-1
  auto wout_of = [&](int l) { return l == L - 1 ? embw : hid; };

#pragma unroll
  for (int l = 0; l < GX_MAX_LAYERS; ++l) {   // (unrolled: the per-layer pointers are read by compile-time index)
    if (l >= L) break;
    const int cnt = win_of(l) * wout_of(l);
    if (S.w_in_smem)
      for (int idx = tid; idx < cnt; idx += NT) sm[S.W[l] + idx] = __ldg(m.W[l] + idx);
    for (int idx = tid; idx < wout_of(l); idx += NT) sm[S.b[l] + idx] = __ldg(m.b[l] + idx);
    if (tid == 0) { s_W[l] = S.w_in_smem ? sm + S.W[l] : m.W[l]; s_b[l] = sm + S.b[l]; }
  }
  if (wp_smem) {
    for (int idx = tid; idx < C * PD; idx += NT) sm[S.Wp + idx] = __ldg(m.Wp + idx);
    for (int idx = tid; idx < C; idx += NT) sm[S.Wp + C * PD + idx] = __ldg(m.bp + idx);
  }
  __syncthreads();
  // embedding of a row without edges: Y = 0 W + b -> normalize(b_l) (-> ReLU (-> standardisation) for hidden layers), whatever the
  // masks are: one constant per layer, the same for every graph of the batch
  if (warp == 0) {
    for (int l = 0; l < L; ++l) {
      const int wout = wout_of(l);
      float v[KW], ssl = 0.f;
#pragma unroll
      for (int k = 0; k < KW; ++k) { const int c = lane + 32 * k; v[k] = c < wout ? s_b[l][c] : 0.f; ssl += v[k] * v[k]; }
      const float qn = fmaxf(sqrtf(warp_sum(ssl)), 1e-12f);
#pragma unroll
      for (int k = 0; k < KW; ++k) v[k] = v[k] / qn;
      if (l < L - 1) {
#pragma unroll
        for (int k = 0; k < KW; ++k) v[k] = fmaxf(v[k], 0.f);
        if (kBn) {
          float sl = 0.f;
#pragma unroll
          for (int k = 0; k < KW; ++k) sl += lane + 32 * k < wout ? v[k] : 0.f;
          const float mu = warp_sum(sl) / (float)wout;
          float vl = 0.f;
#pragma unroll
          for (int k = 0; k < KW; ++k) { v[k] = lane + 32 * k < wout ? v[k] - mu : 0.f; vl += v[k] * v[k]; }
          const float is = 1.0f / sqrtf(warp_sum(vl) / (float)wout + 1e-5f);
#pragma unroll
          for (int k = 0; k < KW; ++k) v[k] *= is;
        }
      }
#pragma unroll
      for (int k = 0; k < KW; ++k) if (lane + 32 * k < wout) cst[hid * l + lane + 32 * k] = v[k];
    }
  }
  float* const slab = A.gws + (int64_t)blockIdx.x * A.gws_stride_words;
  const int nf = A.gb.max_nodes;

  for (;;) {
    __syncthreads();
    if (tid == 0) s_task = atomicAdd(A.counter, 1);
    __syncthreads();
    const int qi = s_task;
    if (qi >= A.ntasks) break;
    const int task_id = A.order[qi];
    const GxTask* __restrict__ Tp = A.plan.tasks + task_id;
    const int na = Tp->n, e_d = Tp->e_d, np = Tp->npairs, gt = Tp->gt_label, g = Tp->node;
    const bool has_const = (Tp->flags & 1) != 0;
    const int64_t node_off = Tp->node_off, rp_off = Tp->rp_off, edge_off = Tp->edge_off, pair_off = Tp->pair_off;
    const GxGraphVarLayout Lo = gx_make_graph_var_layout(na, e_d, np, d, L, VW);
    const int32_t* __restrict__ lo2gid = A.plan.lo2gid + node_off;
    const int32_t* __restrict__ irp = A.plan.irowptr + rp_off;
    const int32_t* __restrict__ icol = A.plan.icol + edge_off;
    const int32_t* __restrict__ pi = A.plan.pair_i + pair_off; const int32_t* __restrict__ pj = A.plan.pair_j + pair_off;
    const int32_t* __restrict__ ppij = A.plan.pair_pij + pair_off; const int32_t* __restrict__ ppji = A.plan.pair_pji + pair_off;
    const int32_t* __restrict__ poij = A.plan.pair_oij + pair_off; const int32_t* __restrict__ poji = A.plan.pair_oji + pair_off;
    const float* __restrict__ X = A.gb.feat + (int64_t)g * nf * d;   // the graph's padded feature rows (full ids)
    float* const a = slab + Lo.a; float* const U = slab + Lo.U; float* const dZ1 = slab + Lo.dZ1;
    auto Yh = [&](int l) { return slab + Lo.Yh + (int64_t)(l - 1) * na * VW; };     // l = 1..L: normalised pre-activation
    auto Hh = [&](int l) { return slab + Lo.H + (int64_t)(l - 1) * na * VW; };      // l = 1..L: what the next layer / the max-pool sees
    auto dZ = [&](int l) { return slab + Lo.dZ + (int64_t)(l - 2) * na * VW; };     // l = 2..L: dL/d(A_m H_{l-1}) (width hid)
    auto qn = [&](int l) { return slab + Lo.q + (int64_t)(l - 1) * na; };
    auto istd = [&](int l) { return slab + Lo.istd + (int64_t)(l - 1) * na; };
    float2* const MM = reinterpret_cast<float2*>(slab + Lo.P); float2* const mm = MM + np; float2* const vv = mm + np; float2* const SS = vv + np;
    const float nn = (float)Tp->n_norm * (float)Tp->n_norm;
    const float ent_over_nn = hp.c_ent / nn;

    for (int f = tid; f < dp; f += NT) {
      sF[f] = 0.5f; Fm[f] = 0.f; mF[f] = 0.f; vF[f] = 0.f;   // feat_mask = 0 (explain.py:633-643)
      if (hp.out_iter == 0 && f < d && A.out_feat != nullptr) A.out_feat[(int64_t)task_id * d + f] = 0.5f;
    }
    {
      const float m0_std = sqrtf(2.0f / (float)Tp->n_norm);  // gain('relu') * sqrt(2/(n+n)), n = the padded size (explain.py:647-651)
      for (int p = tid; p < np; p += NT) {
        const int oij = poij[p], oji = poji[p];
        float Mi, Mj;
        if (hp.init == GX_INIT_PHILOX) {
          Mi = 1.0f + m0_std * philox_normal(hp.seed, (uint32_t)g, (uint32_t)oij);
          Mj = 1.0f + m0_std * philox_normal(hp.seed, (uint32_t)g, (uint32_t)oji);
        } else {
          Mi = __ldg(A.m0 + edge_off + oij);
          Mj = __ldg(A.m0 + edge_off + oji);
        }
        MM[p] = make_float2(Mi, Mj);
        mm[p] = make_float2(0.f, 0.f);
        vv[p] = make_float2(0.f, 0.f);
        const float Si = sigmoid_f(Mi), Sj = sigmoid_f(Mj);
        SS[p] = make_float2(Si, Sj);
        const float a0 = 0.5f * (Si + Sj);  // explain.py:665-678
        a[ppij[p]] = a0; a[ppji[p]] = a0;
        if (hp.out_iter == 0) { A.out_mask[edge_off + oij] = a0; A.out_mask[edge_off + oji] = a0; }
      }
    }
    __syncthreads();

    for (int it = 1; it <= hp.iters; ++it) {
      // ---------------------------------------------------------------- forward, layer by layer, every row with an edge
      for (int l = 1; l <= L; ++l) {
        const int win = win_of(l - 1), wout = wout_of(l - 1);
        const float* const Ws = s_W[l - 1]; const float* const bsm = s_b[l - 1];
        for (int i = warp; i < na; i += nwarps) {
          const int r0 = irp[i], r1 = irp[i + 1];
          float y[KW];
#pragma unroll
          for (int k = 0; k < KW; ++k) y[k] = lane + 32 * k < wout ? bsm[lane + 32 * k] : 0.f;
          if (l == 1) {
            for (int f0 = 0; f0 < d; f0 += 32) {
              const int f = f0 + lane;
              float z = 0.f;
              if (f < d)
                for (int e = r0; e < r1; ++e) z = fmaf(a[e], __ldg(X + (int64_t)lo2gid[icol[e]] * d + f), z);
              if (f < d) { U[(int64_t)i * dp + f] = z; zs[f] = z * sF[f]; }   // x * sigmoid(feat_mask) (explain.py:707), linear in x
            }
          } else {
            const float* const Hp = Hh(l - 1);
#pragma unroll
            for (int k = 0; k < KW; ++k) {
              const int f = lane + 32 * k;
              float z = 0.f;
              if (f < win)
                for (int e = r0; e < r1; ++e) z = fmaf(a[e], Hp[(int64_t)icol[e] * VW + f], z);
              if (f < win) zs[f] = z;
            }
          }
          __syncwarp();
          for (int f = 0; f < win; ++f) {
            const float zf = zs[f];
#pragma unroll
            for (int k = 0; k < KW; ++k)
              if (lane + 32 * k < wout) y[k] = fmaf(zf, Ws[f * wout + lane + 32 * k], y[k]);
          }
          __syncwarp();
          float ssl = 0.f;
#pragma unroll
          for (int k = 0; k < KW; ++k) ssl += lane + 32 * k < wout ? y[k] * y[k] : 0.f;
          const float q = fmaxf(sqrtf(warp_sum(ssl)), 1e-12f);   // F.normalize(p=2, dim=2), eps 1e-12
          float yh[KW], h[KW];
#pragma unroll
          for (int k = 0; k < KW; ++k) { yh[k] = lane + 32 * k < wout ? y[k] / q : 0.f; h[k] = yh[k]; }
          if (l < L) {
#pragma unroll
            for (int k = 0; k < KW; ++k) h[k] = fmaxf(yh[k], 0.f);
            if (kBn) {   // fresh BatchNorm1d(n) in train mode: per node, over the feature axis (models.py:222-228)
              float sl = 0.f;
#pragma unroll
              for (int k = 0; k < KW; ++k) sl += lane + 32 * k < wout ? h[k] : 0.f;
              const float mu = warp_sum(sl) / (float)wout;
              float vl = 0.f;
#pragma unroll
              for (int k = 0; k < KW; ++k) { h[k] = lane + 32 * k < wout ? h[k] - mu : 0.f; vl += h[k] * h[k]; }
              const float var = warp_sum(vl) / (float)wout;
              const float is = 1.0f / sqrtf(var + 1e-5f);
#pragma unroll
              for (int k = 0; k < KW; ++k) h[k] *= is;
              if (lane == 0) istd(l)[i] = is;
            }
          }
#pragma unroll
          for (int k = 0; k < KW; ++k) {
            Yh(l)[(int64_t)i * VW + lane + 32 * k] = yh[k];
            Hh(l)[(int64_t)i * VW + lane + 32 * k] = lane + 32 * k < wout ? h[k] : 0.f;
          }
          if (lane == 0) qn(l)[i] = q;
        }
        __syncthreads();
      }
      // ---------------------------------------------------------------- pool: per-layer column max over the rows (+ the edge-less
      // constant), first arg-max like torch.max; one warp per pooled feature, lanes over the rows      (models.py:283,293,304)
      for (int k = warp; k < PD; k += nwarps) {
        const int l = k < hid * (L - 1) ? k / hid : L - 1;
        const int c = k - hid * l;
        const float* const Hl = Hh(l + 1);
        float best = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = lane; i < na; i += 32) {
          const float v = Hl[(int64_t)i * VW + c];
          if (v > best) { best = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ob = __shfl_xor_sync(0xffffffffu, best, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (has_const && !(best > cst[k])) { best = cst[k]; bi = -1; }   // ties go to the constant, as in explain_graph.cu
        if (lane == 0) { emb[k] = best; arg[k] = bi; }
      }
      __syncthreads();
      // ---------------------------------------------------------------- S: Linear, softmax, dL/dlogits = p - onehot(label), dEmb = Wp^T g
      if (warp == 0) {
        for (int c = 0; c < C; ++c) {
          float t = 0.f;
          for (int k = lane; k < PD; k += 32) t = fmaf(emb[k], Wpp[c * PD + k], t);
          t = warp_sum(t);
          if (lane == 0) logit[c] = t + bpp[c];
        }
        __syncwarp();
        float mx = -INFINITY;
        for (int c = lane; c < C; c += 32) mx = fmaxf(mx, logit[c]);
        mx = warp_max(mx);
        float se = 0.f;
        for (int c = lane; c < C; c += 32) se += expf(logit[c] - mx);
        se = warp_sum(se);
        __syncwarp();
        for (int c = lane; c < C; c += 32) logit[c] = expf(logit[c] - mx) / se - (c == gt ? 1.f : 0.f);  // explain.py:711,750-753
        __syncwarp();
        for (int k = lane; k < PD; k += 32) {
          float t = 0.f;
          for (int c = 0; c < C; ++c) t = fmaf(logit[c], Wpp[c * PD + k], t);
          dEmb[k] = t;
        }
      }
      for (int idx = tid; idx < nwarps * dp; idx += NT) gFp[idx] = 0.f;
      __syncthreads();
      // ---------------------------------------------------------------- backward, layer by layer, every row with an edge
      for (int l = L; l >= 1; --l) {
        const int win = win_of(l - 1), wout = wout_of(l - 1);
        const float* const Ws = s_W[l - 1];
        const int koff = hid * (l - 1);
        for (int i = warp; i < na; i += nwarps) {
          // dL/dH_l[i] = (A_m^T dZ_{l+1})[i] (A_m symmetric) + dEmb routed to the arg-max rows
          float g[KW], yh[KW];
#pragma unroll
          for (int k = 0; k < KW; ++k) g[k] = 0.f;
          if (l < L) {
            const int r0 = irp[i], r1 = irp[i + 1];
            const float* const dZn = dZ(l + 1);
            for (int e = r0; e < r1; ++e) {
              const int j = icol[e];
              const float ae = a[e];
#pragma unroll
              for (int k = 0; k < KW; ++k)
                if (lane + 32 * k < wout) g[k] = fmaf(ae, dZn[(int64_t)j * VW + lane + 32 * k], g[k]);
            }
          }
#pragma unroll
          for (int k = 0; k < KW; ++k) {
            const int c = lane + 32 * k;
            if (c < wout && arg[koff + c] == i) g[k] += dEmb[koff + c];
            yh[k] = Yh(l)[(int64_t)i * VW + c];
          }
          if (l < L) {
            if (kBn) {   // backward of the per-node standardisation: (g - mean(g) - Hb mean(g Hb)) * istd
              float hb[KW], s1 = 0.f, s2 = 0.f;
#pragma unroll
              for (int k = 0; k < KW; ++k) {
                hb[k] = Hh(l)[(int64_t)i * VW + lane + 32 * k];
                if (lane + 32 * k < wout) { s1 += g[k]; s2 += g[k] * hb[k]; }
              }
              const float m1 = warp_sum(s1) / (float)wout, m2 = warp_sum(s2) / (float)wout, is = istd(l)[i];
#pragma unroll
              for (int k = 0; k < KW; ++k) g[k] = lane + 32 * k < wout ? (g[k] - m1 - hb[k] * m2) * is : 0.f;
            }
#pragma unroll
            for (int k = 0; k < KW; ++k) g[k] = yh[k] > 0.f ? g[k] : 0.f;   // relu backward
          }
          float sl = 0.f;
#pragma unroll
          for (int k = 0; k < KW; ++k) sl += lane + 32 * k < wout ? yh[k] * g[k] : 0.f;
          const float sdot = warp_sum(sl);
          const float qi = qn(l)[i];
          __syncwarp();
#pragma unroll
          for (int k = 0; k < KW; ++k)
            if (lane + 32 * k < wout) zs[lane + 32 * k] = (g[k] - yh[k] * sdot) / qi;   // dY: backward of y / max(|y|, eps)
          __syncwarp();
          // dZ[f] = sum_c dY[c] W[f][c]
          if (l == 1) {
            for (int f0 = 0; f0 < d; f0 += 32) {
              const int f = f0 + lane;
              float t = 0.f;
              if (f < d)
                for (int c = 0; c < wout; ++c) t = fmaf(zs[c], Ws[f * wout + c], t);
              if (f < d) {
                gFp[warp * dp + f] = fmaf(t, U[(int64_t)i * dp + f], gFp[warp * dp + f]);   // dL/dsF partial (U = A_m X)
                dZ1[(int64_t)i * dp + f] = t * sF[f];                                        // kept masked for the edge dots
              }
            }
          } else {
#pragma unroll
            for (int k = 0; k < KW; ++k) {
              const int f = lane + 32 * k;
              float t = 0.f;
              if (f < win)
                for (int c = 0; c < wout; ++c) t = fmaf(zs[c], Ws[f * wout + c], t);
              dZ(l)[(int64_t)i * VW + f] = f < win ? t : 0.f;
            }
          }
          __syncwarp();
        }
        __syncthreads();
      }
      // ---------------------------------------------------------------- P: edge gradients (all L layers), regularisers, optimiser step
      {
        const float2 tab = __ldg(hp.adam_tab + (it - 1));
        const float step = tab.x, bc2s = tab.y, bc2s_inv = 1.0f / tab.y;
        const bool last = (it == hp.out_iter);   // the mask built after this update is the one the reference returns
        for (int f = tid; f < d; f += NT) {
          float gsum = 0.f;
          for (int w = 0; w < nwarps; ++w) gsum += gFp[w * dp + f];
          const float s = sF[f];
          const float gg = s * (1.f - s) * (gsum + hp.c_feat_size / (float)d);
          float mf = mF[f], vf = vF[f], Fv = Fm[f];
          if (hp.opt == GX_OPT_ADAM) {
            mf = mf + (gg - mf) * hp.one_minus_b1;
            vf = vf * hp.b2 + hp.one_minus_b2 * gg * gg;
            Fv = Fv - step * (mf / (sqrtf(vf) / bc2s + hp.eps));
          } else {
            opt_step_other(hp.opt, Fv, gg, mf, vf, step);
          }
          mF[f] = mf; vF[f] = vf; Fm[f] = Fv;
          const float sn = sigmoid_f(Fv);
          sF[f] = sn;   // (the edge dots below use dZ1 (.) sF stored in the backward, not this value)
          if (last && A.out_feat != nullptr) A.out_feat[(int64_t)task_id * d + f] = sn;
        }
        for (int p = tid; p < np; p += NT) {
          const int i = pi[p], j = pj[p];
          float Gd = 0.f;
          {
            float t = 0.f;
            const float* xj = X + (int64_t)lo2gid[j] * d; const float* xi = X + (int64_t)lo2gid[i] * d;
            for (int f = 0; f < d; ++f) t = fmaf(dZ1[(int64_t)i * dp + f], __ldg(xj + f), t);
            Gd += t;
            t = 0.f;
            for (int f = 0; f < d; ++f) t = fmaf(dZ1[(int64_t)j * dp + f], __ldg(xi + f), t);
            Gd += t;
          }
          for (int l = 2; l <= L; ++l) {
            const float* const dZl = dZ(l); const float* const Hp = Hh(l - 1);
            float t = 0.f;
            for (int f = 0; f < hid; ++f) t = fmaf(dZl[(int64_t)i * VW + f], Hp[(int64_t)j * VW + f], t);
            Gd += t;
            t = 0.f;
            for (int f = 0; f < hid; ++f) t = fmaf(dZl[(int64_t)j * VW + f], Hp[(int64_t)i * VW + f], t);
            Gd += t;
          }
          Gd *= 0.5f;  // sym_mask = (S + S^T)/2 (explain.py:671); no Laplacian term in graph mode (explain.py:787-788)
          float2 Mv = MM[p];
          const float2 Sv = SS[p];
          float2 m2 = mm[p], v2 = vv[p];
          const float gi = Sv.x * (1.f - Sv.x) * (Gd + hp.c_size - ent_over_nn * Mv.x);
          const float gj = Sv.y * (1.f - Sv.y) * (Gd + hp.c_size - ent_over_nn * Mv.y);
          if (hp.opt == GX_OPT_ADAM) {
            m2.x = m2.x + (gi - m2.x) * hp.one_minus_b1;
            m2.y = m2.y + (gj - m2.y) * hp.one_minus_b1;
            v2.x = v2.x * hp.b2 + hp.one_minus_b2 * gi * gi;
            v2.y = v2.y * hp.b2 + hp.one_minus_b2 * gj * gj;
            Mv.x = Mv.x - adam_delta_fast(m2.x, v2.x, step, bc2s, bc2s_inv, hp.eps, ieee);
            Mv.y = Mv.y - adam_delta_fast(m2.y, v2.y, step, bc2s, bc2s_inv, hp.eps, ieee);
          } else {
            opt_step_other(hp.opt, Mv.x, gi, m2.x, v2.x, step);
            opt_step_other(hp.opt, Mv.y, gj, m2.y, v2.y, step);
          }
          const float2 Sn = make_float2(sigmoid_fast(Mv.x, ieee), sigmoid_fast(Mv.y, ieee));
          MM[p] = Mv; mm[p] = m2; vv[p] = v2; SS[p] = Sn;
          const float an = 0.5f * (Sn.x + Sn.y);
          a[ppij[p]] = an; a[ppji[p]] = an;
          if (last) { A.out_mask[edge_off + poij[p]] = an; A.out_mask[edge_off + poji[p]] = an; }
        }
      }
      __syncthreads();
    }
  }
}

}  // namespace

int gx_graph_var_smem_bytes(int d, int L, int hid, int emb, int C) { return gv_smem(d, L, hid, emb, C, kGvThreads / 32).total * 4; }
int gx_graph_var_row_stride(int hid, int emb) { return 32 * gv_kw(hid, emb); }

cudaError_t gx_launch_explain_graph_var(const GxExplainLaunch& cfg, const GxGraphBatchDev& gb, const GxModelDev& m,
                                        const GxHparamsDev& hp, const GxPlanArrays& plan, const float* m0, float* out_mask,
                                        float* out_feat, cudaStream_t s) {
  GraphVarArgs args;
  args.order = cfg.order; args.ntasks = cfg.ntasks; args.counter = cfg.counter;
  args.gws = cfg.gws; args.gws_stride_words = cfg.gws_stride_words;
  args.gb = gb; args.m = m; args.hp = hp; args.plan = plan;
  args.m0 = m0; args.out_mask = out_mask; args.out_feat = out_feat;
  const int bytes = gx_graph_var_smem_bytes(m.d, m.L, m.hid, m.emb, m.C);
  const int kw = gv_kw(m.hid, m.emb);
  auto go = [&](auto kern) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return e;
    // the largest carveout, like every other launch class: CTAs of the shared-memory classes can share an SM with these
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    kern<<<cfg.grid, kGvThreads, bytes, s>>>(args);
    return cudaGetLastError();
  };
  if (m.bn) {
    if (kw == 1) return go(explain_graph_var_kernel<true, 1>);
    if (kw == 2) return go(explain_graph_var_kernel<true, 2>);
    return go(explain_graph_var_kernel<true, 4>);
  }
  if (kw == 1) return go(explain_graph_var_kernel<false, 1>);
  if (kw == 2) return go(explain_graph_var_kernel<false, 2>);
  return go(explain_graph_var_kernel<false, 4>);
}
