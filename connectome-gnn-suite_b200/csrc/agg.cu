// agg.cu - the gather half of the tensor-core generation of layer kernels.
//
//   k_build_agg      CSR arrays -> packed per-subject aggregation blobs (agg.cuh), once per batch and model family
//   k_gather<MODE>   one subject tile [n, C] in shared memory (two CTAs per SM), one warp per output row:
//     GATHER_SAGE_FWD  agg_i = sum_{e: dst=i} w_e u_src / (w_sum_i + 1e-8), u = act(t_in)     (reference models.py:146-149)
//     GATHER_GCN_FWD   a_i   = sum_{e: dst=i} w^_e u_src + dinv_i^2 u_i, u = act(t_in)  (wide layers, models.py:94-114)
//     GATHER_GCN_BWD   dP_j  = sum_{e: src=j} w^_e dz_dst + dinv_j^2 dz_j, dz from z / upstream / BatchNorm backward
//                      on load, plus dbias = column sums of dz                        (autograd of models.py:112-114)
//     GATHER_SAGE_BWD  du_j  = d_u_j + sum_{e: src=j} w_e d_agg_dst / (w_sum_dst + 1e-8), plus the BatchNorm
//                      backward sums of the layer below                               (autograd of models.py:146-149)
// The dense contractions around them live in gemm_tc.cu.
#include "agg.cuh"
#include "tile.cuh"
#include "rowtile.cuh"

namespace cgnn {

// ------------------------------------------------------------------------------------------------------------
// blob builder: one CTA per subject, one thread per row
// ------------------------------------------------------------------------------------------------------------
struct BuildAggArgs {
  const int32_t* in_rowptr; const int32_t* in_col; const float* in_w; const float* in_wn;
  const int32_t* out_rowptr; const int32_t* out_col; const float* out_w; const float* out_wn;
  const float* dinv; const float* wsum; const int32_t* meta;
  int kind, max_nodes, skip_edge_cap;
  int32_t* agg_in; int32_t* agg_out; int32_t* row_graph;
};

__global__ void __launch_bounds__(256) k_build_agg(BuildAggArgs p) {
  CGNN_SMEM_DECL;
  __shared__ int s_tot[2][8];
  int* s_pos = reinterpret_cast<int*>(cgnn_smem);   // [2][max_nodes] padded record counts -> exclusive positions
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long g = blockIdx.x;
  const int4 m = reinterpret_cast<const int4*>(p.meta)[g];
  const long long nb = m.x, eb = m.z;
  const int n = m.y;
  if (n > p.max_nodes) return;
  if (p.skip_edge_cap >= 0 && m.w <= p.skip_edge_cap && n <= 65535) return;   // the collate kernel already emitted this one
  const int self = p.kind == AGG_GCN ? 1 : 0;
  for (int dir = 0; dir < 2; ++dir) {
    const int32_t* rp = dir == 0 ? p.in_rowptr : p.out_rowptr;
    // exclusive scan of the padded row lengths: chunked per thread, warp scan, cross-warp carry
    const int per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
    const int lo = min(tid * per, n), hi = min(lo + per, n);
    int sum = 0;
    for (int i = lo; i < hi; ++i) {
      const int c = (rp[nb + i + 1] - rp[nb + i] + self + 1) & ~1;
      s_pos[dir * p.max_nodes + i] = c;
      sum += c;
    }
    int inc = sum;
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += v;
    }
    if (lane == 31) s_tot[dir][warp] = inc;
    __syncthreads();
    int carry = 0;
    for (int w = 0; w < warp; ++w) carry += s_tot[dir][w];
    int run = carry + inc - sum;
    for (int i = lo; i < hi; ++i) { const int c = s_pos[dir * p.max_nodes + i]; s_pos[dir * p.max_nodes + i] = run; run += c; }
  }
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) p.row_graph[nb + i] = (int32_t)g;
  for (int dir = 0; dir < 2; ++dir) {
    const int32_t* rp = dir == 0 ? p.in_rowptr : p.out_rowptr;
    const int32_t* col = dir == 0 ? p.in_col : p.out_col;
    const float* wv = p.kind == AGG_GCN ? (dir == 0 ? p.in_wn : p.out_wn) : (dir == 0 ? p.in_w : p.out_w);
    int32_t* blob = (dir == 0 ? p.agg_in : p.agg_out) + agg_base_words(nb, eb, g);
    int4* desc = reinterpret_cast<int4*>(blob);
    int2* rec = reinterpret_cast<int2*>(blob + 4 * (long long)n);
    for (int i = tid; i < n; i += blockDim.x) {
      const int e0 = rp[nb + i], e1 = rp[nb + i + 1];
      int pos = s_pos[dir * p.max_nodes + i];
      const int begin = pos;
      for (int e = e0; e < e1; ++e) {
        const int nbr = (int)(col[e] - nb);
        float w = wv[e];
        if (p.kind == AGG_SAGE && dir == 1) w = w / (p.wsum[nb + nbr] + 1e-8f);   // adjoint of the weighted mean
        rec[pos++] = make_int2(dir == 0 ? agg_rec_x(nbr) : nbr, __float_as_int(w));
      }
      const int self_x = dir == 0 ? agg_rec_x(i) : i;
      if (self) { const float d = p.dinv[nb + i]; rec[pos++] = make_int2(self_x, __float_as_int(__fmul_rn(d, d))); }
      if (pos & 1) rec[pos++] = make_int2(self_x, 0);
      const float aux = p.kind == AGG_SAGE ? p.wsum[nb + i] : p.dinv[nb + i];
      desc[i] = make_int4(begin, pos, __float_as_int(aux), i);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// gather kernels
// ------------------------------------------------------------------------------------------------------------
#ifndef CGNN_EMU
// One CTA works on one 4*LPR-channel slab of one subject at a time (two CTAs per SM for the 32-channel slabs of a
// 360-node subject): the subject's blob arrives by cp.async while the threads transform their channel quad of the
// tile on the way into shared memory; then 32 / LPR rows per warp are gathered with float4 lanes from shared memory.
template <int MODE, int LPR, bool VEC>
__global__ void __launch_bounds__(kThreads, 2) k_gather(GatherArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  constexpr int RP = kThreads / LPR;    // tile rows per load pass
  constexpr int RPW = 32 / LPR;         // rows per warp in the gather
  float4* s_tile = reinterpret_cast<float4*>(cgnn_smem);                       // [max_nodes][LPR]
  int32_t* s_blob = reinterpret_cast<int32_t*>(s_tile + (size_t)p.max_nodes * LPR);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int cl = tid % LPR, rl = tid / LPR;
  const int C = p.C, nslab = p.nslab;
  const int slab = blockIdx.x % nslab;
  const int c0 = slab * 4 * LPR + 4 * cl;
  const bool live_quad = c0 < C;

  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act, c0, C);
  const rt::RowKey rk = rt::row_key(p.act);
  rt::BnQuad bq;
  if (MODE == GATHER_GCN_BWD) rt::bn_quad_init(bq, p.bn, c0, C);
  float pmean[4] = {0.f, 0.f, 0.f, 0.f}, prstd[4] = {0.f, 0.f, 0.f, 0.f};
  if (MODE == GATHER_SAGE_BWD && p.want_prev) rt::bn_stats_quad(pmean, prstd, p.prev_mean, p.prev_rstd, c0, C, true);
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};   // GCN_BWD: s1 = dbias; SAGE_BWD: sums of the layer below

  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  const long long gstep = gridDim.x / nslab;
  int4 m_next = make_int4(0, 0, 0, 0);
  if ((long long)(blockIdx.x / nslab) < p.B) m_next = meta[blockIdx.x / nslab];
  for (long long g = blockIdx.x / nslab; g < p.B; g += gstep) {
    const int4 m = m_next;                       // loaded one unit ahead: no exposed latency at the top of a unit
    if (g + gstep < p.B) m_next = meta[g + gstep];
    const long long nb = m.x, eb = m.z;
    const int n = min(m.y, p.max_nodes), me = min(m.w, p.max_edges);
    // ---- the subject's blob: one asynchronous burst ------------------------------------------------------------
    {
      const int32_t* gb = p.blob + agg_base_words(nb, eb, g);
      const int n16 = (agg_copy_words(n, me) + 3) >> 2;
      for (int i = tid; i < n16; i += kThreads) cp_async_16(s_blob + 4 * i, gb + 4 * i);
      cp_async_commit();
    }
    // ---- load phase: this thread's channel quad of rows rl, rl + RP, ... transformed on the way in --------------
    float4 pooled = make_float4(0.f, 0.f, 0.f, 0.f);
    if (MODE == GATHER_GCN_BWD && !p.du && live_quad) pooled = rt::pooled_quad<VEC>(p.demb, g, C, c0, n);
    // UL rows per thread are loaded before any is processed: one exposed memory latency per batch of UL
    constexpr int UL = MODE == GATHER_GCN_BWD ? 2 : 6;
    for (int r = rl; r < n; r += UL * RP) {
      float4 a[UL], b[MODE == GATHER_GCN_BWD ? UL : 1];
#pragma unroll
      for (int u = 0; u < UL; ++u) {
        const int rr = r + u * RP;
        a[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (MODE == GATHER_GCN_BWD) b[u] = pooled;
        if (rr < n && live_quad) {
          a[u] = rt::ld_quad<VEC>(p.src, nb + rr, C, c0);
          if (MODE == GATHER_GCN_BWD && p.du) b[u] = rt::ld_quad<VEC>(p.du, nb + rr, C, c0);
        }
      }
#pragma unroll
      for (int u = 0; u < UL; ++u) {
        const int rr = r + u * RP;
        if (rr < n) {
          float4 o = a[u];
          if (MODE == GATHER_SAGE_FWD || MODE == GATHER_GCN_FWD) o = rt::act_fwd4(p.act, cq, a[u], rk, (uint32_t)(nb + rr));
          if (MODE == GATHER_GCN_BWD) {
            o = rt::dz4<false>(p.act, cq, p.bn, bq, a[u], b[MODE == GATHER_GCN_BWD ? u : 0], rk, (uint32_t)(nb + rr));
            if (!VEC) o = rt::mask_quad(o, c0, C);
            s1[0] += o.x; s1[1] += o.y; s1[2] += o.z; s1[3] += o.w;
          }
          if (!VEC) o = rt::mask_quad(o, c0, C);
          s_tile[rr * LPR + cl] = o;
          if (MODE == GATHER_SAGE_FWD && p.out_u && live_quad) rt::st_quad<VEC>(p.out_u, nb + rr, C, c0, o);
        }
      }
    }
    cp_async_wait<0>();
    __syncthreads();
    // ---- gather phase --------------------------------------------------------------------------------------------
    const int4* s_desc = reinterpret_cast<const int4*>(s_blob);
    const int4* s_rec2 = reinterpret_cast<const int4*>(s_blob + 4 * n);
    for (int i0 = warp * RPW; i0 < n; i0 += kWarps * RPW) {
      float4 acc;
      float aux;
      int row;
      float4 dpre = make_float4(0.f, 0.f, 0.f, 0.f), rpre = dpre;
      if (MODE == GATHER_SAGE_BWD) {   // the row's direct gradient and stored input: loads fly during the gather
        const int rowp = i0 + (tid & 31) / LPR;
        if (rowp < n && live_quad) {
          dpre = rt::ld_quad<VEC>(p.direct, nb + rowp, C, c0);
          if (p.want_prev) rpre = rt::ld_quad<VEC>(p.t_raw, nb + rowp, C, c0);
        }
      }
      constexpr bool kPre = MODE == GATHER_SAGE_FWD || MODE == GATHER_GCN_FWD;   // by-destination blob
      const bool valid = agg_gather_group<LPR, LPR, kPre>(s_desc, s_rec2, s_tile, i0, n, acc, aux, row);
      if (!valid || !live_quad) continue;
      const long long grow = nb + row;
      if (MODE == GATHER_SAGE_FWD) {
        const float inv = fast_rcp(aux + 1e-8f);   // weighted mean (models.py:149); ~1 ulp off the exact quotient
        acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
      }
      if (MODE == GATHER_SAGE_BWD) {
        const float4 d = dpre;
        acc.x += d.x; acc.y += d.y; acc.z += d.z; acc.w += d.w;
        if (p.want_prev) {
          const float4 raw = rpre;
          const float4 dyp = rt::act_bwd4(p.act, cq, raw, acc, rk, (uint32_t)grow);
          const float rv[4] = {raw.x, raw.y, raw.z, raw.w}, dv[4] = {dyp.x, dyp.y, dyp.z, dyp.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c0 + j < C) bn_sums_add(s1[j], s2[j], dv[j], rv[j], pmean[j], prstd[j]);
        }
      }
      rt::st_quad<VEC>(p.out, grow, C, c0, acc);
    }
    __syncthreads();   // tile and blob are rewritten by the next subject
  }

  // ---- per-CTA partial records (zero outside this CTA's slab) ---------------------------------------------------------
  const bool want = (MODE == GATHER_GCN_BWD && p.partials) || (MODE == GATHER_SAGE_BWD && p.partials && p.want_prev);
  if (want) {
    float* red = reinterpret_cast<float*>(s_tile);   // [kThreads][8]
    *reinterpret_cast<float4*>(red + 8 * tid) = make_float4(s1[0], s1[1], s1[2], s1[3]);
    *reinterpret_cast<float4*>(red + 8 * tid + 4) = make_float4(s2[0], s2[1], s2[2], s2[3]);
    __syncthreads();
    const int nrec = MODE == GATHER_GCN_BWD ? 1 : 2;
    for (int idx = tid; idx < nrec * C; idx += kThreads) {
      const int which = idx / C, c = idx - which * C;
      const float s = c / (4 * LPR) == slab ? quad_sum(red, 8, 4 * which, kThreads, LPR, (c % (4 * LPR)) >> 2, c & 3) : 0.0f;
      p.partials[(size_t)blockIdx.x * p.part_stride + idx] = s;
    }
  }
  (void)RP;
}

// ---- host side -------------------------------------------------------------------------------------------------
static bool gather_shape(int C, int max_nodes, int max_edges, int* lpr, int* nslab, size_t* smem) {
  if (C <= 0 || C > 256) return false;
  int L, S;
  if (C <= 8) { L = 2; S = 1; }
  else if (C <= 32) { L = 8; S = 1; }
  else if (C % 32 == 0) { L = 8; S = C / 32; }
  else return false;
  if (max_nodes < 1) max_nodes = 1;
  size_t bytes = (size_t)max_nodes * L * 16 + (size_t)agg_smem_words(max_nodes, max_edges) * 4;
  if (bytes < (size_t)kThreads * 8 * 4) bytes = (size_t)kThreads * 8 * 4;
  *lpr = L; *nslab = S; *smem = bytes;
  return bytes <= (size_t)device_info().smem_optin;
}
bool gather_supported(int C, int max_nodes, int max_edges) {
  int l, s; size_t b;
  return gather_shape(C, max_nodes, max_edges, &l, &s, &b);
}

// Launches one gather kernel; returns the grid through *grid_out (the caller reduces `partials` over it).
int launch_gather(int mode, GatherArgs& a, int* grid_out, cudaStream_t stream) {
  const DeviceInfo dev = device_info();
  int LPR = 0, nslab = 0;
  size_t smem = 0;
  if (a.max_nodes < 1) a.max_nodes = 1;
  if (!gather_shape(a.C, a.max_nodes, a.max_edges, &LPR, &nslab, &smem)) return CGNN_ERR_INVALID_ARG;
  a.nslab = nslab;
  const int C = a.C;
  auto al16 = [](const void* p) { return p == nullptr || (((uintptr_t)p) & 15u) == 0; };
  const int vec = (C % 4 == 0) && al16(a.src) && al16(a.du) && al16(a.demb) && al16(a.direct) && al16(a.t_raw) && al16(a.out);
  int per_sm = (int)((size_t)(228 * 1024) / (smem + 1024));
  if (per_sm > 2) per_sm = 2;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)per_sm * dev.sm_count;
  grid -= grid % nslab;
  if (grid > a.B * nslab) grid = a.B * nslab;
  if (grid < nslab) grid = nslab;
  *grid_out = (int)grid;
#define CGNN_GATHER(MODE_, LPR_, VEC_)                                                                   \
  {                                                                                                      \
    auto kfn = k_gather<MODE_, LPR_, VEC_>;                                                              \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, (unsigned)grid, kThreads, smem, stream, a);                                         \
  }
#define CGNN_GATHER_L(MODE_)                                                                             \
  {                                                                                                      \
    if (LPR == 2) { if (vec) CGNN_GATHER(MODE_, 2, true) else CGNN_GATHER(MODE_, 2, false) }             \
    else { if (vec) CGNN_GATHER(MODE_, 8, true) else CGNN_GATHER(MODE_, 8, false) }                      \
  }
  if (mode == GATHER_SAGE_FWD) CGNN_GATHER_L(GATHER_SAGE_FWD)
  else if (mode == GATHER_GCN_BWD) CGNN_GATHER_L(GATHER_GCN_BWD)
  else if (mode == GATHER_GCN_FWD) CGNN_GATHER_L(GATHER_GCN_FWD)
  else CGNN_GATHER_L(GATHER_SAGE_BWD)
#undef CGNN_GATHER_L
#undef CGNN_GATHER
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

#endif  // CGNN_EMU

int launch_build_agg(const cgnn_csr_t* csr, int32_t kind, int64_t num_graphs, int32_t max_nodes, int32_t* agg_in, int32_t* agg_out,
                     int32_t* row_graph, int skip_edge_cap, cudaStream_t stream) {
  BuildAggArgs a;
  a.in_rowptr = csr->in_rowptr; a.in_col = csr->in_col; a.in_w = csr->in_w; a.in_wn = csr->in_wn;
  a.out_rowptr = csr->out_rowptr; a.out_col = csr->out_col; a.out_w = csr->out_w; a.out_wn = csr->out_wn;
  a.dinv = csr->dinv; a.wsum = csr->wsum; a.meta = csr->graph_meta;
  a.kind = kind; a.max_nodes = max_nodes < 1 ? 1 : max_nodes; a.skip_edge_cap = skip_edge_cap;
  a.agg_in = agg_in; a.agg_out = agg_out; a.row_graph = row_graph;
  const size_t smem = (size_t)2 * a.max_nodes * sizeof(int) + 16;
  const DeviceInfo dev = device_info();
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  auto kfn = k_build_agg;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  CGNN_LAUNCH(kfn, (unsigned)num_graphs, 256, smem, stream, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

}  // namespace cgnn

using namespace cgnn;

extern "C" {

size_t cgnn_agg_words(int64_t rows, int64_t edges, int64_t num_graphs) {
  if (rows < 0 || edges < 0 || num_graphs < 0) return 0;
  return agg_total_words(rows, edges, num_graphs);
}

int cgnn_build_agg(const cgnn_csr_t* csr, int32_t kind, int64_t num_graphs, int64_t rows, int64_t edges,
                   int32_t max_nodes, int32_t* agg_in, int32_t* agg_out, int32_t* row_graph, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!csr || (kind != AGG_GCN && kind != AGG_SAGE) || num_graphs < 0 || rows < 0 || edges < 0 || max_nodes < 0)
    return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) return CGNN_OK;
  if (!agg_in || !agg_out || !row_graph || !csr->in_rowptr || !csr->in_col || !csr->in_w || !csr->in_wn ||
      !csr->out_rowptr || !csr->out_col || !csr->out_w || !csr->out_wn || !csr->dinv || !csr->wsum || !csr->graph_meta)
    return CGNN_ERR_INVALID_ARG;
  return launch_build_agg(csr, kind, num_graphs, max_nodes, agg_in, agg_out, row_graph, -1, stream);
}

}  // extern "C"
