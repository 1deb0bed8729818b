// first_layer.cu - the narrow-input layer (d_in <= 8: the first layer, F = 5 node features) without tensor cores.
//
// With 5 input channels the layer is all output traffic: z = [.] W^T + b has 10-20 multiply-adds per output element,
// the gather runs in the 5-channel input space, and a 128-row MMA pipeline only adds barriers.  One CTA per subject
// (three per SM), two phases:
//   forward   input rows (+ blob) -> shared memory; a = A^ x (GCN) or the weighted mean (GraphSAGE) by the packed-blob
//             gather; then thread = (row, output-channel quad): z = b + sum_k in_k W[.][k], ReLU (GraphSAGE),
//             Welford partials for BatchNorm, 16-byte coalesced stores             (reference models.py:111-114, 146-152)
//   backward  (no input gradient - node features are data) same staging of the per-row input vector, then
//             thread = (row, quad): dz on load (dropout / ReLU / BatchNorm backward), dW += dz (x) in, dbias += dz
//                                                                       (autograd of models.py:111-114 / 151-152)
#include "agg.cuh"
#include "rowtile.cuh"
#include "tile.cuh"

namespace cgnn {
#ifndef CGNN_EMU

struct FirstArgs {
  const float* t_in; Act act_in; const float* W; const float* bias;
  const int32_t* blob; const int32_t* meta; long long B;
  int K, H, max_nodes, max_edges;
  // forward
  float* z; float* agg_out; double* stats_partials;
  // backward
  const float* du; const float* demb; const float* zin; Act act_out; BnBwdDev bn; const float* agg_in;
  float* partials; int part_stride;     // per CTA: [dW H x K2][dbias H]
};

// the per-row input vector of the contraction in shared memory: s_x = act(t_in) rows, s_a = aggregated rows, both
// [n][8] floats (zero padded); GraphSAGE backward reads the aggregate stored by forward instead of gathering
template <int SAGE, bool BWD, int NT>
__device__ __forceinline__ void stage_subject(const FirstArgs& p, const int4& m, long long g, float4* s_x, float4* s_a,
                                              int32_t* s_blob) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long nb = m.x;
  const int n = m.y, K = p.K;
  const bool need_gather = !(SAGE && BWD);
  if (need_gather) {
    const int32_t* gb = p.blob + agg_base_words(nb, m.z, g);
    const int n16 = (agg_copy_words(n, m.w) + 3) >> 2;
    for (int i = tid; i < n16; i += NT) cp_async_16(s_blob + 4 * i, gb + 4 * i);
  }
  cp_async_commit();
  const bool affine = p.act_in.scale != nullptr;
  for (int base = tid; base < 8 * n; base += 4 * NT) {     // four independent loads in flight per thread
    float v[4], g2[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = base + u * NT, r = idx >> 3, k = idx & 7;
      v[u] = 0.0f; g2[u] = 0.0f;
      if (idx < 8 * n && k < K) {
        v[u] = p.t_in[(nb + r) * K + k];
        if (!need_gather) g2[u] = p.agg_in[(nb + r) * K + k];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int idx = base + u * NT, r = idx >> 3, k = idx & 7;
      if (idx >= 8 * n) continue;
      float x = v[u];
      if (k < K) {
        const uint32_t rh = p.act_in.drop ? drop_row_hash(p.act_in, p.act_in.row_base + nb + r) : 0u;
        x = act_fwd(p.act_in, affine, x, affine ? p.act_in.scale[k] : 1.0f, affine ? p.act_in.shift[k] : 0.0f, rh, k);
      }
      reinterpret_cast<float*>(s_x)[idx] = x;
      if (!need_gather) reinterpret_cast<float*>(s_a)[idx] = g2[u];
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  if (need_gather) {
    const int4* s_desc = reinterpret_cast<const int4*>(s_blob);
    const int4* s_rec2 = reinterpret_cast<const int4*>(s_blob + 4 * n);
    for (int i0 = warp * 16; i0 < n; i0 += (NT / 32) * 16) {
      float4 acc;
      float aux;
      int row;
      if (!agg_gather_group<2>(s_desc, s_rec2, s_x, i0, n, acc, aux, row)) continue;
      if (SAGE) {
        const float den = aux + 1e-8f;
        acc.x /= den; acc.y /= den; acc.z /= den; acc.w /= den;
      }
      const int cl = lane & 1;
      s_a[row * 2 + cl] = acc;
      if (SAGE && !BWD && p.agg_out) rt::st_quad<false>(p.agg_out, nb + row, K, 4 * cl, acc);
    }
    __syncthreads();
  }
}

// QH = H / 4 output-channel quads; thread = (quad tid % QH, rows tid / QH + i * NT / QH); NT threads per CTA, two CTAs per SM
template <int SAGE, int QH, int NT, int KX>
__global__ void __launch_bounds__(NT, 2) k_first_fwd(FirstArgs p) {
  act_salt(p.act_in); act_salt(p.act_out);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  constexpr int RS = NT / QH, H = 4 * QH, KK = SAGE ? 2 * KX : KX;
  float4* s_x = reinterpret_cast<float4*>(cgnn_smem);                 // [max_nodes][2]
  float4* s_a = s_x + 2 * (size_t)p.max_nodes;                         // [max_nodes][2]
  int32_t* s_blob = reinterpret_cast<int32_t*>(s_a + 2 * (size_t)p.max_nodes);
  const int tid = threadIdx.x, q = tid % QH, rsub = tid / QH;
  const int K = p.K;
  // this thread's weights: wq[k][j] = W[4q + j][k] (GCN: k over the aggregate; GraphSAGE: 0-7 self, 8-15 neighbours)
  float wq[KK][4];
#pragma unroll
  for (int k = 0; k < KK; ++k)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int kk = k % KX, half = k / KX;
      wq[k][j] = kk < K ? p.W[(size_t)(4 * q + j) * (SAGE ? 2 * K : K) + half * K + kk] : 0.0f;
    }
  float b4[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) b4[j] = p.bias ? p.bias[4 * q + j] : 0.0f;
  const bool want_stats = p.stats_partials != nullptr;
  QuadWelford wf;
  wf.init();

  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  int4 m_next = make_int4(0, 0, 0, 0);
  if ((long long)blockIdx.x < p.B) m_next = meta[blockIdx.x];
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    int4 m = m_next;                               // loaded one subject ahead
    if (g + gridDim.x < p.B) m_next = meta[g + gridDim.x];
    m.y = min(m.y, p.max_nodes); m.w = min(m.w, p.max_edges);
    stage_subject<SAGE, false, NT>(p, m, g, s_x, s_a, s_blob);
    const long long nb = m.x;
    for (int r = rsub; r < m.y; r += RS) {
      const float4 a0 = s_a[2 * r], a1 = s_a[2 * r + 1];
      const float in_a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float4 o4 = make_float4(b4[0], b4[1], b4[2], b4[3]);
      if (SAGE) {
        const float4 x0 = s_x[2 * r], x1 = s_x[2 * r + 1];
        const float in_x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
        for (int k = 0; k < KX; ++k) fma_quad(o4, make_float4(wq[k][0], wq[k][1], wq[k][2], wq[k][3]), in_x[k]);
      }
#pragma unroll
      for (int k = 0; k < KX; ++k) {
        constexpr int O = SAGE ? KX : 0;
        fma_quad(o4, make_float4(wq[O + k][0], wq[O + k][1], wq[O + k][2], wq[O + k][3]), in_a[k]);
      }
      float o[4] = {o4.x, o4.y, o4.z, o4.w};
      if (SAGE) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = fmaxf(o[j], 0.0f);
      }
      *reinterpret_cast<float4*>(p.z + (nb + r) * H + 4 * q) = make_float4(o[0], o[1], o[2], o[3]);
      if (want_stats) wf.push(make_float4(o[0], o[1], o[2], o[3]));   // BatchNorm batch statistics: training only
    }
    __syncthreads();   // tiles and blob are rewritten by the next subject
  }

  if (p.stats_partials) {
    float* rec = reinterpret_cast<float*>(cgnn_smem);   // [NT][9]
    wf.deposit(rec + tid * 9);
    __syncthreads();
    cta_write_quad_stats(rec, NT, QH, H, tid, p.stats_partials + (size_t)blockIdx.x * (1 + 2 * H));
  }
}

template <int SAGE, int QH, int NT, int KX>
__global__ void __launch_bounds__(NT, 2) k_first_bwd(FirstArgs p) {
  act_salt(p.act_in); act_salt(p.act_out);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  constexpr int RS = NT / QH, H = 4 * QH, KK = SAGE ? 2 * KX : KX;
  float4* s_x = reinterpret_cast<float4*>(cgnn_smem);
  float4* s_a = s_x + 2 * (size_t)p.max_nodes;
  int32_t* s_blob = reinterpret_cast<int32_t*>(s_a + 2 * (size_t)p.max_nodes);
  const int tid = threadIdx.x, q = tid % QH, rsub = tid / QH;
  const int K = p.K, K2 = SAGE ? 2 * K : K;
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act_out, 4 * q, H);
  const rt::RowKey rk = rt::row_key(p.act_out);
  rt::BnQuad bq;
  rt::bn_quad_init(bq, p.bn, 4 * q, H);
  float acc[KK][4];
#pragma unroll
  for (int k = 0; k < KK; ++k)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[k][j] = 0.0f;
  float db[4] = {0.f, 0.f, 0.f, 0.f};

  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  int4 m_next = make_int4(0, 0, 0, 0);
  if ((long long)blockIdx.x < p.B) m_next = meta[blockIdx.x];
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    int4 m = m_next;                               // loaded one subject ahead
    if (g + gridDim.x < p.B) m_next = meta[g + gridDim.x];
    m.y = min(m.y, p.max_nodes); m.w = min(m.w, p.max_edges);
    stage_subject<SAGE, true, NT>(p, m, g, s_x, s_a, s_blob);
    const long long nb = m.x;
    float4 pooled = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!p.du) pooled = rt::pooled_quad<true>(p.demb, g, H, 4 * q, m.y);
    constexpr int UB = 4;     // rows in flight per thread
    for (int r = rsub; r < m.y; r += UB * RS) {
      float4 zv[UB], uv[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        uv[u] = pooled;
        if (r + u * RS < m.y) {
          zv[u] = rt::ld_quad<true>(p.zin, nb + r + u * RS, H, 4 * q);
          if (p.du) uv[u] = rt::ld_quad<true>(p.du, nb + r + u * RS, H, 4 * q);
        }
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int rr = r + u * RS;
        if (rr >= m.y) continue;
        const float4 dz = rt::dz4<SAGE>(p.act_out, cq, p.bn, bq, zv[u], uv[u], rk, (uint32_t)(nb + rr));
        const float d4[4] = {dz.x, dz.y, dz.z, dz.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) db[j] += d4[j];
        const float4 a0 = s_a[2 * rr], a1 = s_a[2 * rr + 1];
        const float in_a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        if (SAGE) {
          const float4 x0 = s_x[2 * rr], x1 = s_x[2 * rr + 1];
          const float in_x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
          for (int k = 0; k < KX; ++k)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[k][j] = fmaf(d4[j], in_x[k], acc[k][j]);
        }
#pragma unroll
        for (int k = 0; k < KX; ++k)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[SAGE ? KX + k : k][j] = fmaf(d4[j], in_a[k], acc[SAGE ? KX + k : k][j]);
      }
    }
    __syncthreads();
  }

  // per-CTA partial record [dW H x K2][dbias H]: one pass per input index through a [NT] float4 buffer
  float4* red = reinterpret_cast<float4*>(cgnn_smem);
  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
#pragma unroll 1
  for (int k = 0; k <= KK; ++k) {
    float4 v = make_float4(db[0], db[1], db[2], db[3]);
#pragma unroll
    for (int kk = 0; kk < KK; ++kk)
      if (kk == k) v = make_float4(acc[kk][0], acc[kk][1], acc[kk][2], acc[kk][3]);
    red[tid] = v;
    __syncthreads();
    const int kin = k % KX, half = k / KX;          // k == KK: the dbias pass
    const bool live = k == KK || kin < K;
    if (live && tid < H) {
      const int qq = tid >> 2, j = tid & 3;
      float s = 0.0f;
      for (int th = qq; th < NT; th += QH) s += reinterpret_cast<const float*>(&red[th])[j];
      if (k == KK) part[(size_t)H * K2 + tid] = s;
      else part[(size_t)tid * K2 + half * K + kin] = s;
    }
    __syncthreads();
  }
  (void)RS;
}

static size_t first_smem(int max_nodes, int max_edges) {
  size_t b = (size_t)max_nodes * 64 + (size_t)agg_smem_words(max_nodes, max_edges) * 4;
  if (b < (size_t)kThreads * 36) b = (size_t)kThreads * 36;
  return b;
}
static bool first_shape_ok(const cgnn_csr_t* csr, int kind, int d_in, int H, int max_nodes, int max_edges, size_t* smem) {
  if (d_in < 1 || d_in > 8 || (H != 32 && H != 64 && H != 128 && H != 256)) return false;
  if (!csr->agg_in || csr->agg_kind != kind) return false;
  *smem = first_smem(max_nodes < 1 ? 1 : max_nodes, max_edges);
  return *smem <= (size_t)device_info().smem_optin;
}
static int first_grid(size_t smem, long long B) {
  const DeviceInfo dev = device_info();
  int per_sm = (int)((size_t)(228 * 1024) / (smem + 1024));
  if (per_sm > 2) per_sm = 2;     // __launch_bounds__(NT, 2): the weight / accumulator registers need the room
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)per_sm * dev.sm_count;
  if (grid > B) grid = B;
  return (int)(grid < 1 ? 1 : grid);
}

// Returns CGNN_OK when launched (grid in *grid_out: the caller merges `partials`), -1 when the shape is not covered.
int launch_first_fwd(int kind, const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                     int64_t num_graphs, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z, float* agg_out,
                     double* partials, int* grid_out, size_t workspace_bytes, cudaStream_t stream) {
  size_t smem = 0;
  if (!first_shape_ok(csr, kind, d_in, H, max_nodes, max_edges, &smem)) return -1;
  if ((((uintptr_t)z) & 15u) != 0) return -1;
  FirstArgs a{};
  a.t_in = t_in; a.act_in = make_act(act); a.W = W; a.bias = bias;
  a.blob = csr->agg_in; a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.max_nodes = max_nodes < 1 ? 1 : max_nodes; a.max_edges = max_edges;
  a.z = z; a.agg_out = agg_out; a.stats_partials = partials;
  int grid = first_grid(smem, num_graphs);
  if (partials) {
    const size_t rec = (size_t)(1 + 2 * H) * sizeof(double);
    if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
    if (grid < 1) return -1;
  }
  *grid_out = grid;
#define CGNN_FF(S_, QH_, KX_)                                                                                   \
  {                                                                                                        \
    auto kfn = k_first_fwd<S_, QH_, (S_ ? 256 : 512), KX_>;                                                                       \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, (unsigned)grid, (S_ ? 256 : 512), smem, stream, a);                                   \
  }
#define CGNN_FF_H(S_, KX_) { if (H == 32) CGNN_FF(S_, 8, KX_) else if (H == 64) CGNN_FF(S_, 16, KX_) else if (H == 128) CGNN_FF(S_, 32, KX_) else CGNN_FF(S_, 64, KX_) }
  if (d_in <= 5) { if (kind == AGG_SAGE) CGNN_FF_H(1, 5) else CGNN_FF_H(0, 5) }
  else { if (kind == AGG_SAGE) CGNN_FF_H(1, 8) else CGNN_FF_H(0, 8) }
#undef CGNN_FF_H
#undef CGNN_FF
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

// dW [H x K2] and dbias [H] of a narrow layer whose input needs no gradient; partial records [H*K2 + H] per CTA.
int launch_first_bwd(int kind, const float* du, const float* demb, const float* z, const cgnn_act_t* act_out,
                     const cgnn_bn_bwd_t* bn, const float* t_in, const float* agg, const cgnn_act_t* act_in, const cgnn_csr_t* csr,
                     int64_t num_graphs, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* partials,
                     int* grid_out, size_t partial_bytes, cudaStream_t stream) {
  size_t smem = 0;
  if (!first_shape_ok(csr, kind, d_in, H, max_nodes, max_edges, &smem)) return -1;
  if (kind == AGG_SAGE && !agg) return -1;
  if (((((uintptr_t)z) | ((uintptr_t)du) | ((uintptr_t)demb)) & 15u) != 0) return -1;
  FirstArgs a{};
  a.t_in = t_in; a.act_in = make_act(act_in);
  a.blob = csr->agg_in; a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.max_nodes = max_nodes < 1 ? 1 : max_nodes; a.max_edges = max_edges;
  a.du = du; a.demb = demb; a.zin = z; a.act_out = make_act(act_out); a.agg_in = agg; a.bn = make_bn_bwd(bn);
  const int K2 = kind == AGG_SAGE ? 2 * d_in : d_in;
  a.partials = partials; a.part_stride = H * K2 + H;
  int grid = first_grid(smem, num_graphs);
  const size_t rec = (size_t)a.part_stride * sizeof(float);
  if ((size_t)grid * rec > partial_bytes) grid = (int)(partial_bytes / rec);
  if (grid < 1) return -1;
  *grid_out = grid;
#define CGNN_FB(S_, QH_, KX_)                                                                                   \
  {                                                                                                        \
    auto kfn = k_first_bwd<S_, QH_, 256, KX_>;                                                                       \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, (unsigned)grid, 256, smem, stream, a);                                                \
  }
#define CGNN_FB_H(S_, KX_) { if (H == 32) CGNN_FB(S_, 8, KX_) else if (H == 64) CGNN_FB(S_, 16, KX_) else if (H == 128) CGNN_FB(S_, 32, KX_) else CGNN_FB(S_, 64, KX_) }
  if (d_in <= 5) { if (kind == AGG_SAGE) CGNN_FB_H(1, 5) else CGNN_FB_H(0, 5) }
  else { if (kind == AGG_SAGE) CGNN_FB_H(1, 8) else CGNN_FB_H(0, 8) }
#undef CGNN_FB_H
#undef CGNN_FB
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

#endif  // CGNN_EMU
}  // namespace cgnn
