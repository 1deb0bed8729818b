// sage.cu - K2 / K7: GraphSAGE layer forward and backward, one persistent CTA per subject graph.
//
// Forward (reference models.py:136-152, fused with the previous layer's models.py:260-261):
//   u = dropout(bn(t_in))                               on load (identity for the first layer)
//   agg_i = (sum_{e: dst=i} w_e u_src(e)) / (wsum_i + 1e-8)          COO order
//   z = relu([u || agg] W^T + b)                        + Welford statistics for BatchNorm
// Backward: kernel A (row-local: dq, dW, db, d[u||agg] = dq W) and kernel B (transposed
//   neighbour aggregation of the agg-gradient + previous layer's BatchNorm backward sums).
#include "tile.cuh"
#include "agg.cuh"

namespace cgnn {

// Weighted-mean neighbourhood rows for a chunk: s_cat[r] = [u_i || agg_i], i = r0 + r.
template <int CC>
__device__ __forceinline__ void sage_cat_rows(const float* s_u, int K4, float* s_cat, int ldc, int r0, int rows,
                                              int n, long long nb, const RowCsr& rc, const float* wsum_g) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < kChunkRows; r += kWarps) {
    float acc[CC];
#pragma unroll
    for (int j = 0; j < CC; ++j) acc[j] = 0.0f;
    float denom = 1.0f;
    if (r < rows) {
      gather_row<CC, true>(rc, r0 + r, nb, n, s_u, K4, K4, acc);
      denom = __fadd_rn(wsum_g[r0 + r], 1e-8f);
    }
#pragma unroll
    for (int j = 0; j < CC; ++j) {
      const int ch = lane + 32 * j;
      if (ch < K4) {
        s_cat[r * ldc + ch] = r < rows ? s_u[(r0 + r) * K4 + ch] : 0.0f;
        s_cat[r * ldc + K4 + ch] = r < rows ? acc[j] / denom : 0.0f;
      }
    }
  }
}

// Whole-subject input tile of K % 4 == 0 channels, copied raw into s_u: the previous layer's BatchNorm/dropout in place.
__device__ __forceinline__ void sage_transform_tile(float* s_u, int n, int K, const Act& act, const float* s_scale, const float* s_shift,
                                                    long long nb) {
  const bool affine = act.scale != nullptr;
  for (int idx = threadIdx.x; idx < n * K; idx += blockDim.x) {
    const int r = idx / K, c = idx - r * K;
    const uint32_t rh = act.drop ? drop_row_hash(act, act.row_base + nb + r) : 0u;
    s_u[idx] = act_fwd(act, affine, s_u[idx], s_scale[c], s_shift[c], rh, c);
  }
}

struct SageFwdArgs {
  const float* t_in; Act act; const float* W; const float* bias;
  const int32_t* in_rowptr; const int32_t* in_col; const float* in_w; const float* wsum;
  const int32_t* meta; long long B;
  int K, H, K4, H4, ldc, max_nodes, max_edges, csr_smem;
  float* z; double* partials; float* agg_out;
  int o_wt, o_scale, o_shift, o_bias, o_u, o_cat, o_out, o_st, o_csr;
};

template <int CC>
__global__ void __launch_bounds__(kThreads) k_sage_fwd(SageFwdArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  float* s_wt = sm + p.o_wt;        // [2*K4][H4]
  float* s_scale = sm + p.o_scale;
  float* s_shift = sm + p.o_shift;
  float* s_bias = sm + p.o_bias;
  float* s_u = sm + p.o_u;          // [max_nodes][K4]
  float* s_cat = sm + p.o_cat;      // [kChunkRows][ldc]
  float* s_out = sm + p.o_out;      // [kChunkRows][H4]
  float* s_cnt = sm + p.o_st;
  float* s_mean = s_cnt + kWarps;
  float* s_m2 = s_mean + kWarps * p.H4;
  float* s_csr = sm + p.o_csr;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = p.K, H = p.H, K4 = p.K4, H4 = p.H4, ldc = p.ldc;
  const bool affine = p.act.scale != nullptr;

  for (int idx = tid; idx < 2 * K4 * H4; idx += kThreads) {
    const int kk = idx / H4, h = idx - kk * H4;
    const int half = kk >= K4, k = kk - half * K4;
    s_wt[idx] = (k < K && h < H) ? p.W[h * 2 * K + half * K + k] : 0.0f;
  }
  stage_affine(p.act, K, K4, s_scale, s_shift);
  for (int h = tid; h < H4; h += kThreads) s_bias[h] = (h < H && p.bias) ? p.bias[h] : 0.0f;
  __syncthreads();

  WarpStats<CC> st;
  st.init();
  const int tiles_x = H4 >> 2;
  const int ntiles = (kChunkRows >> 2) * tiles_x;
  const int4* meta = reinterpret_cast<const int4*>(p.meta);

  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    int4 cur = meta[g];
    if (cur.y > p.max_nodes) cur.y = p.max_nodes;
    const long long nb = cur.x;
    const int n = cur.y, eb = cur.z, m = cur.w;
    const bool csr_here = p.csr_smem && m <= p.max_edges;
    // whole input tile + CSR in one async burst
    if (K == K4) cp_async_words(s_u, p.t_in + nb * K, n * K);
    if (csr_here) stage_csr_async(s_csr, p.max_nodes, p.max_edges, p.in_rowptr, p.in_col, p.in_w, p.wsum, nb, n, eb, m);
    cp_async_commit();
    if (K != K4) {   // narrow first layer: rows are not 16-byte multiples, stage with plain loads
      for (int idx = tid; idx < n * K4; idx += kThreads) {
        const int r = idx / K4, c = idx - r * K4;
        float v = 0.0f;
        if (c < K) {
          const uint32_t rh = p.act.drop ? drop_row_hash(p.act, p.act.row_base + nb + r) : 0u;
          v = act_fwd(p.act, affine, p.t_in[(nb + r) * K + c], s_scale[c], s_shift[c], rh, c);
        }
        s_u[idx] = v;
      }
    }
    cp_async_wait<0>();
    __syncthreads();
    if (K == K4) {
      sage_transform_tile(s_u, n, K, p.act, s_scale, s_shift, nb);
      __syncthreads();
    }
    const float* wsum_g = p.wsum + nb;
    RowCsr rc{p.in_rowptr + nb, p.in_col, p.in_w};
    if (csr_here) rc = staged_csr(s_csr, p.max_nodes, p.max_edges, eb, &wsum_g);

    for (int r0 = 0; r0 < n; r0 += kChunkRows) {
      const int rows = min(kChunkRows, n - r0);
      sage_cat_rows<CC>(s_u, K4, s_cat, ldc, r0, rows, n, nb, rc, wsum_g);
      __syncthreads();
      if (p.agg_out) {   // the aggregated neighbourhood, kept for backward
        for (int r = warp; r < rows; r += kWarps) {
#pragma unroll
          for (int j = 0; j < CC; ++j) {
            const int ch = lane + 32 * j;
            if (ch < K) p.agg_out[(nb + r0 + r) * K + ch] = s_cat[r * ldc + K4 + ch];
          }
        }
      }
      for (int t = tid; t < ntiles; t += kThreads) {
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        if (4 * ty >= rows) continue;
        float acc[4][4] = {};
        mma_4x4(s_cat + 4 * ty * ldc, ldc, s_wt + 4 * tx, H4, 2 * K4, acc);
        const float4 b = *reinterpret_cast<const float4*>(s_bias + 4 * tx);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<float4*>(s_out + (4 * ty + i) * H4 + 4 * tx) =
              make_float4(fmaxf(acc[i][0] + b.x, 0.f), fmaxf(acc[i][1] + b.y, 0.f), fmaxf(acc[i][2] + b.z, 0.f),
                          fmaxf(acc[i][3] + b.w, 0.f));
      }
      __syncthreads();
      for (int r = warp; r < rows; r += kWarps) {
        float inv;
        st.begin_row(inv);
#pragma unroll
        for (int j = 0; j < CC; ++j) {
          const int ch = lane + 32 * j;
          if (ch < H) {
            const float v = s_out[r * H4 + ch];
            p.z[(nb + r0 + r) * H + ch] = v;
            st.w[j].push(v, inv);
          }
        }
      }
    }
    __syncthreads();  // s_u / s_out / staged CSR are rewritten by the next subject
  }

  if (p.partials) {
    st.deposit(s_cnt, s_mean, s_m2, H4, H4);
    __syncthreads();
    cta_write_stats(s_cnt, s_mean, s_m2, H4, H, p.partials + (size_t)blockIdx.x * (1 + 2 * H));
  }
}

// ------------------------------------------------------------------------------------------
struct SageBwdArgs {
  const float* du; const float* demb; const float* z; Act act_out; BnBwdDev bn;
  const float* t_in; Act act_in; const float* W;
  const int32_t* in_rowptr; const int32_t* in_col; const float* in_w; const float* wsum;
  const int32_t* meta; long long B;
  int K, H, K4, H4, ldc, ldq, max_nodes, max_edges, csr_smem, vec_h, need_du;
  float* direct; float* nbr;  // scratch [rows, K] each
  float* partials; int part_stride, o_pdw, o_pdb;
  int o_w, o_co, o_ci, o_u, o_cat, o_dq, o_red, o_csr;
};

// dq of one element: dropout backward, BatchNorm backward, ReLU mask of the layer's own output.
__device__ __forceinline__ float sage_dq(const SageBwdArgs& p, const float* s_co, int H4, bool aff_out, float t, float up,
                                         uint32_t rh, int c) {
  const float dz = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, t, up, rh, c);
  return t > 0.0f ? dz : 0.0f;
}

template <int CC, int MAXT>
__global__ void __launch_bounds__(kThreads) k_sage_bwd_a(SageBwdArgs p) {
  act_salt(p.act_out); act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  float* s_w = sm + p.o_w;      // [H4][2*K4] natural layout
  float* s_co = sm + p.o_co;    // [DZ_ROWS][H4]
  float* s_ci = sm + p.o_ci;    // [2][K4] scale, shift of act_in
  float* s_u = sm + p.o_u;      // [max_nodes][K4]
  float* s_cat = sm + p.o_cat;  // [kChunkRows][ldc]
  float* s_dq = sm + p.o_dq;    // [kChunkRows][ldq]
  float* s_red = sm + p.o_red;
  float* s_csr = sm + p.o_csr;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = p.K, H = p.H, K4 = p.K4, H4 = p.H4, ldc = p.ldc, ldq = p.ldq, K8 = 2 * p.K4;
  const bool aff_out = p.act_out.scale != nullptr, aff_in = p.act_in.scale != nullptr;

  for (int idx = tid; idx < H4 * K8; idx += kThreads) {
    const int h = idx / K8, kk = idx - h * K8;
    const int half = kk >= K4, k = kk - half * K4;
    s_w[idx] = (h < H && k < K) ? p.W[h * 2 * K + half * K + k] : 0.0f;
  }
  stage_dz_consts(p.act_out, p.bn, H, H4, s_co);
  stage_affine(p.act_in, K, K4, s_ci, s_ci + K4);
  __syncthreads();

  const int tk = K8 >> 2;
  const int ntiles_w = (H4 >> 2) * tk;
  const int ntiles_u = (kChunkRows >> 2) * tk;

  float acc_w[MAXT][4][4];
#pragma unroll
  for (int it = 0; it < MAXT; ++it)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc_w[it][i][j] = 0.0f;
  float acc_db[CC];
#pragma unroll
  for (int j = 0; j < CC; ++j) acc_db[j] = 0.0f;
  const int4* meta = reinterpret_cast<const int4*>(p.meta);

  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    int4 cur = meta[g];
    if (cur.y > p.max_nodes) cur.y = p.max_nodes;
    const long long nb = cur.x;
    const int n = cur.y, eb = cur.z, m = cur.w;
    const bool csr_here = p.csr_smem && m <= p.max_edges;
    const float inv_n = pool_bwd_scale(n);
    if (K == K4) cp_async_words(s_u, p.t_in + nb * K, n * K);
    if (csr_here) stage_csr_async(s_csr, p.max_nodes, p.max_edges, p.in_rowptr, p.in_col, p.in_w, p.wsum, nb, n, eb, m);
    cp_async_commit();
    if (K != K4) {
      for (int idx = tid; idx < n * K4; idx += kThreads) {
        const int r = idx / K4, c = idx - r * K4;
        float v = 0.0f;
        if (c < K) {
          const uint32_t rh = p.act_in.drop ? drop_row_hash(p.act_in, p.act_in.row_base + nb + r) : 0u;
          v = act_fwd(p.act_in, aff_in, p.t_in[(nb + r) * K + c], s_ci[c], s_ci[K4 + c], rh, c);
        }
        s_u[idx] = v;
      }
    }
    cp_async_wait<0>();
    __syncthreads();
    if (K == K4) {
      sage_transform_tile(s_u, n, K, p.act_in, s_ci, s_ci + K4, nb);
      __syncthreads();
    }
    const float* wsum_g = p.wsum + nb;
    RowCsr rc{p.in_rowptr + nb, p.in_col, p.in_w};
    if (csr_here) rc = staged_csr(s_csr, p.max_nodes, p.max_edges, eb, &wsum_g);

    for (int r0 = 0; r0 < n; r0 += kChunkRows) {
      const int rows = min(kChunkRows, n - r0);
      // (b) dq = relu'(z) * bn_bwd(dropout_bwd(du)): issue the global loads first, they fly during (a)
      if (p.vec_h) {
        const int q4 = H4 >> 2;
        const int total = rows * q4;
        for (int base = tid; base < kChunkRows * q4; base += 4 * kThreads) {
          float4 zv[4], uv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int idx = base + u * kThreads;
            if (idx < total) {
              const int r = idx / q4, c = (idx - r * q4) << 2;
              zv[u] = *reinterpret_cast<const float4*>(p.z + (nb + r0 + r) * H + c);
              if (p.du) uv[u] = *reinterpret_cast<const float4*>(p.du + (nb + r0 + r) * H + c);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int idx = base + u * kThreads;
            if (idx < kChunkRows * q4) {
              const int r = idx / q4, c = (idx - r * q4) << 2;
              float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
              if (idx < total) {
                if (!p.du) {
                  const float4 e = *reinterpret_cast<const float4*>(p.demb + g * H + c);
                  uv[u] = make_float4(e.x * inv_n, e.y * inv_n, e.z * inv_n, e.w * inv_n);
                }
                const uint32_t rh = p.act_out.drop ? drop_row_hash(p.act_out, p.act_out.row_base + nb + r0 + r) : 0u;
                o.x = sage_dq(p, s_co, H4, aff_out, zv[u].x, uv[u].x, rh, c);
                o.y = sage_dq(p, s_co, H4, aff_out, zv[u].y, uv[u].y, rh, c + 1);
                o.z = sage_dq(p, s_co, H4, aff_out, zv[u].z, uv[u].z, rh, c + 2);
                o.w = sage_dq(p, s_co, H4, aff_out, zv[u].w, uv[u].w, rh, c + 3);
              }
              *reinterpret_cast<float4*>(s_dq + r * ldq + c) = o;
            }
          }
        }
      } else {
        for (int idx = tid; idx < kChunkRows * H4; idx += kThreads) {
          const int r = idx / H4, c = idx - r * H4;
          float dq = 0.0f;
          if (r < rows && c < H) {
            const long long grow = nb + r0 + r;
            const float t = p.z[grow * H + c];
            const float up = p.du ? p.du[grow * H + c] : p.demb[g * H + c] * inv_n;
            const uint32_t rh = p.act_out.drop ? drop_row_hash(p.act_out, p.act_out.row_base + grow) : 0u;
            dq = sage_dq(p, s_co, H4, aff_out, t, up, rh, c);
          }
          s_dq[r * ldq + c] = dq;
        }
      }
      // (a) [u || agg] rows
      sage_cat_rows<CC>(s_u, K4, s_cat, ldc, r0, rows, n, nb, rc, wsum_g);
      __syncthreads();
      for (int r = warp; r < rows; r += kWarps) {
#pragma unroll
        for (int j = 0; j < CC; ++j) {
          const int ch = lane + 32 * j;
          if (ch < H4) acc_db[j] += s_dq[r * ldq + ch];
        }
      }
      // (c) dW += dq^T [u || agg]
#pragma unroll
      for (int it = 0; it < MAXT; ++it) {
        const int t = tid + it * kThreads;
        if (t < ntiles_w) {
          const int th = t / tk, tq = t - th * tk;
          outer_4x4(s_dq + 4 * th, ldq, s_cat + 4 * tq, ldc, rows, acc_w[it]);
        }
      }
      // (d) d[u || agg] = dq W : direct half and (already mean-normalised) neighbour half
      if (p.need_du) {
        for (int t = tid; t < ntiles_u; t += kThreads) {
          const int ty = t / tk, tx = t - ty * tk;
          if (4 * ty >= rows) continue;
          float acc[4][4] = {};
          mma_4x4(s_dq + 4 * ty * ldq, ldq, s_w + 4 * tx, K8, H4, acc);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = 4 * ty + i;
            if (r >= rows) continue;
            const long long grow = nb + r0 + r;
            const bool is_nbr = 4 * tx >= K4;
            const float sc = is_nbr ? 1.0f / __fadd_rn(wsum_g[r0 + r], 1e-8f) : 1.0f;
            float* dst = is_nbr ? p.nbr : p.direct;
            const int kb = 4 * tx - (is_nbr ? K4 : 0);
#pragma unroll
            for (int q = 0; q < 4; ++q)
              if (kb + q < K) dst[grow * K + kb + q] = acc[i][q] * sc;
          }
        }
      }
      __syncthreads();
    }
  }

  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
#pragma unroll
  for (int it = 0; it < MAXT; ++it) {
    const int t = tid + it * kThreads;
    if (t < ntiles_w) {
      const int th = t / tk, tq = t - th * tk;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(part + p.o_pdw + (4 * th + i) * K8 + 4 * tq) =
            make_float4(acc_w[it][i][0], acc_w[it][i][1], acc_w[it][i][2], acc_w[it][i][3]);
    }
  }
#pragma unroll
  for (int j = 0; j < CC; ++j) {
    const int ch = lane + 32 * j;
    if (ch < H4) s_red[warp * H4 + ch] = acc_db[j];
  }
  __syncthreads();
  for (int c = tid; c < H4; c += kThreads) part[p.o_pdb + c] = warp_rows_sum(s_red, H4, c);
}

struct SageBwdBArgs {
  const float* direct; const float* nbr; const float* t_in; Act act_in;
  const int32_t* out_rowptr; const int32_t* out_col; const float* out_w;
  const float* prev_mean; const float* prev_rstd; int want_prev;
  const int32_t* meta; long long B;
  int K, K4, max_nodes, max_edges, csr_smem;
  float* du_in; float* partials;  // [grid][2*K4]
  int o_g, o_ci, o_red, o_csr;
};

// du_in[j] = direct[j] + sum_{e: src=j} w_e * nbr[dst(e)]   (nbr already divided by wsum+1e-8)
template <int CC>
__global__ void __launch_bounds__(kThreads) k_sage_bwd_b(SageBwdBArgs p) {
  act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  float* s_g = sm + p.o_g;      // [max_nodes][K4]
  float* s_ci = sm + p.o_ci;    // [4][K4] scale, shift, mean, rstd
  float* s_red = sm + p.o_red;  // [kWarps][2*K4]
  float* s_csr = sm + p.o_csr;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = p.K, K4 = p.K4;
  const bool aff_in = p.act_in.scale != nullptr;

  stage_affine(p.act_in, K, K4, s_ci, s_ci + K4);
  for (int c = tid; c < K4; c += kThreads) {
    const bool ok = c < K && p.want_prev;
    s_ci[2 * K4 + c] = ok ? p.prev_mean[c] : 0.0f;
    s_ci[3 * K4 + c] = ok ? p.prev_rstd[c] : 0.0f;
  }
  __syncthreads();

  float ps1[CC], ps2[CC];
#pragma unroll
  for (int j = 0; j < CC; ++j) { ps1[j] = 0.0f; ps2[j] = 0.0f; }
  const int4* meta = reinterpret_cast<const int4*>(p.meta);

  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    int4 cur = meta[g];
    if (cur.y > p.max_nodes) cur.y = p.max_nodes;
    const long long nb = cur.x;
    const int n = cur.y, eb = cur.z, m = cur.w;
    const bool csr_here = p.csr_smem && m <= p.max_edges;
    if (K == K4) cp_async_words(s_g, p.nbr + nb * K, n * K);
    if (csr_here) stage_csr_async(s_csr, p.max_nodes, p.max_edges, p.out_rowptr, p.out_col, p.out_w, nullptr, nb, n, eb, m);
    cp_async_commit();
    if (K != K4) {
      for (int idx = tid; idx < n * K4; idx += kThreads) {
        const int i = idx / K4, c = idx - i * K4;
        s_g[idx] = c < K ? p.nbr[(nb + i) * K + c] : 0.0f;
      }
    }
    cp_async_wait<0>();
    __syncthreads();
    const float* unused = nullptr;
    RowCsr rc{p.out_rowptr + nb, p.out_col, p.out_w};
    if (csr_here) rc = staged_csr(s_csr, p.max_nodes, p.max_edges, eb, &unused);
    for (int jr = warp; jr < n; jr += kWarps) {
      const long long grow = nb + jr;
      float acc[CC], t0[CC];
#pragma unroll
      for (int j = 0; j < CC; ++j) {
        const int ch = lane + 32 * j;
        acc[j] = ch < K ? p.direct[grow * K + ch] : 0.0f;
        t0[j] = (p.want_prev && ch < K) ? p.t_in[grow * K + ch] : 0.0f;
      }
      gather_row<CC, false>(rc, jr, nb, n, s_g, K4, K4, acc);
      const uint32_t rh = (p.want_prev && p.act_in.drop) ? drop_row_hash(p.act_in, p.act_in.row_base + grow) : 0u;
#pragma unroll
      for (int j = 0; j < CC; ++j) {
        const int ch = lane + 32 * j;
        if (ch < K) {
          p.du_in[grow * K + ch] = acc[j];
          if (p.want_prev) {
            const float dyp = act_bwd(p.act_in, aff_in, t0[j], s_ci[ch], s_ci[K4 + ch], rh, ch, acc[j]);
            bn_sums_add(ps1[j], ps2[j], dyp, t0[j], s_ci[2 * K4 + ch], s_ci[3 * K4 + ch]);
          }
        }
      }
    }
    __syncthreads();
  }

  if (p.want_prev) {
#pragma unroll
    for (int j = 0; j < CC; ++j) {
      const int ch = lane + 32 * j;
      if (ch < K4) { s_red[warp * 2 * K4 + ch] = ps1[j]; s_red[warp * 2 * K4 + K4 + ch] = ps2[j]; }
    }
    __syncthreads();
    float* part = p.partials + (size_t)blockIdx.x * 2 * K4;
    for (int c = tid; c < 2 * K4; c += kThreads) part[c] = warp_rows_sum(s_red, 2 * K4, c);
  }
}

}  // namespace cgnn

using namespace cgnn;

static bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }
static int imax(int a, int b) { return a > b ? a : b; }

extern "C" {

int cgnn_sage_layer_fwd(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias,
                        const cgnn_csr_t* csr, const int64_t* ptr, int64_t num_graphs, int64_t rows,
                        int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z, double* bn_stats,
                        float* agg, void* workspace, size_t workspace_bytes, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || rows < 0 || d_in <= 0 || H <= 0 || max_nodes < 0 || max_edges < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) {
    if (bn_stats) cudaMemsetAsync(bn_stats, 0, (size_t)(1 + 2 * H) * sizeof(double), stream);
    return CGNN_OK;
  }
  // full CSR arrays, or a lean batch (graph_meta + this family's blobs; the tensor-core kernels read nothing else)
  const bool arrays_fwd = csr && csr->in_rowptr && csr->in_col && csr->in_w && csr->wsum;
  const bool lean = csr && !csr->in_col && csr->agg_in && csr->agg_kind == AGG_SAGE;
  if (!t_in || !W || !csr || !csr->graph_meta || !(arrays_fwd || lean) || !ptr || !z) return CGNN_ERR_INVALID_ARG;
  if (d_in % 4 == 0 && !aligned16(t_in)) return CGNN_ERR_INVALID_ARG;
  if (bn_stats && (!workspace || workspace_bytes < (size_t)(1 + 2 * H) * sizeof(double))) return CGNN_ERR_WORKSPACE;
#ifndef CGNN_EMU
  // Narrow first layer: gather + projection in one kernel, no tensor cores.
  if (tensor_cores_enabled() && agg && d_in <= 8) {
    int g0 = 0;
    const int rc0 = launch_first_fwd(AGG_SAGE, t_in, act, W, bias, csr, num_graphs, d_in, H, max_nodes, max_edges, z, agg,
                                     bn_stats ? (double*)workspace : nullptr, &g0, workspace_bytes, stream);
    if (rc0 == CGNN_OK) return bn_stats ? launch_stats_merge((const double*)workspace, g0, H, bn_stats, stream) : CGNN_OK;
    if (rc0 > 0) return rc0;
  }
  // Wide layers (H = d_in = 256): gather + K-looped contraction (wide_tc.cu).
  if (tensor_cores_enabled() && wide_shape(d_in, H)) {
    int gw = 0;
    const int rcw = launch_sage_fwd_wide(t_in, act, agg, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, z,
                                         bn_stats ? 1 : 0, &gw, workspace, workspace_bytes, stream);
    if (rcw == CGNN_OK) return bn_stats ? launch_stats_merge((const double*)workspace, gw, H, bn_stats, stream) : CGNN_OK;
    if (rcw > 0) return rcw;
  }
  // Tensor-core generation: gather kernel (weighted mean of the neighbours) + tcgen05 contraction.
  if (tensor_cores_enabled() && agg && csr->agg_in && csr->agg_kind == AGG_SAGE && aligned16(agg) &&
      gather_supported(d_in, max_nodes, max_edges) &&
      sage_fwd_gemm_supported(t_in, agg, z, rows, d_in, H, bn_stats != nullptr, workspace_bytes)) {
    GatherArgs ga{};
    ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_in;
    ga.C = d_in; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
    ga.src = t_in; ga.act = make_act(act); ga.out = agg;
    int g1 = 0, g2 = 0;
    int rc = launch_gather(GATHER_SAGE_FWD, ga, &g1, stream);
    if (rc != CGNN_OK) return rc;
    rc = launch_sage_fwd_gemm(t_in, act, agg, W, bias, rows, d_in, H, z, bn_stats ? (double*)workspace : nullptr, &g2,
                              workspace_bytes, stream);
    if (rc != CGNN_OK) return rc;
    return bn_stats ? launch_stats_merge((const double*)workspace, g2, H, bn_stats, stream) : CGNN_OK;
  }
#endif
  if (!arrays_fwd) return CGNN_ERR_NEED_CSR;       // the generic kernel walks the CSR arrays
  const DeviceInfo dev = device_info();
  SageFwdArgs a;
  a.t_in = t_in; a.act = make_act(act); a.W = W; a.bias = bias;
  a.in_rowptr = csr->in_rowptr; a.in_col = csr->in_col; a.in_w = csr->in_w; a.wsum = csr->wsum;
  a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.K4 = round_up(d_in, 4); a.H4 = round_up(H, 4); a.ldc = 2 * a.K4 + 4;
  a.max_nodes = max_nodes < 1 ? 1 : max_nodes;
  a.max_edges = max_edges;
  a.z = z; a.agg_out = agg;
  if (a.H4 > 256 || a.K4 > 256) return CGNN_ERR_TILE_TOO_LARGE;
  int off = 0;
  a.o_wt = off; off += 2 * a.K4 * a.H4;
  a.o_scale = off; off += a.K4;
  a.o_shift = off; off += a.K4;
  a.o_bias = off; off += a.H4;
  a.o_u = off; off += a.max_nodes * a.K4;
  a.o_cat = off; off += kChunkRows * a.ldc;
  a.o_out = off; off += kChunkRows * a.H4;
  a.o_st = off; off += round_up(kWarps + 2 * kWarps * a.H4, 4);
  {
    const int csr_w = cgnn::csr_words(a.max_nodes, a.max_edges);
    a.csr_smem = ((size_t)(off + csr_w) * sizeof(float) <= (size_t)dev.smem_optin) ? 1 : 0;
    a.o_csr = off;
    if (a.csr_smem) off += csr_w;
  }
  const size_t smem = (size_t)off * sizeof(float);
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  int grid = persistent_grid(num_graphs, smem, dev, kThreads);
  const size_t rec = (size_t)(1 + 2 * H) * sizeof(double);
  a.partials = nullptr;
  if (bn_stats) {
    if (!workspace || workspace_bytes < rec) return CGNN_ERR_WORKSPACE;
    if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
    a.partials = (double*)workspace;
  }
  const int cc = imax(pick_hc(a.H4), pick_hc(a.K4));
#define CGNN_SAGE_FWD(CC_)                                                                       \
  {                                                                                              \
    auto kfn = k_sage_fwd<CC_>;                                                                  \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);                                           \
  }
  if (cc == 1) CGNN_SAGE_FWD(1) else if (cc == 2) CGNN_SAGE_FWD(2) else if (cc == 4) CGNN_SAGE_FWD(4) else CGNN_SAGE_FWD(8)
#undef CGNN_SAGE_FWD
  CGNN_CHECK_LAUNCH();
  if (bn_stats) return launch_stats_merge(a.partials, grid, H, bn_stats, stream);
  return CGNN_OK;
}

int cgnn_sage_layer_bwd(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out,
                        const cgnn_bn_bwd_t* bn, const float* t_in, const float* agg, const cgnn_act_t* act_in, const float* W,
                        const cgnn_csr_t* csr, const int64_t* ptr, int64_t num_graphs, int64_t rows,
                        int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* dW, float* dbias,
                        float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64, float* scratch,
                        void* workspace, size_t workspace_bytes, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  (void)agg;
  if (max_edges < 0) return CGNN_ERR_INVALID_ARG;
  if (!dW || !dbias || num_graphs < 0 || rows < 0 || d_in <= 0 || H <= 0 || max_nodes < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) {
    cudaMemsetAsync(dW, 0, (size_t)H * 2 * d_in * sizeof(float), stream);
    cudaMemsetAsync(dbias, 0, (size_t)H * sizeof(float), stream);
    if (prev_sums) cudaMemsetAsync(prev_sums, 0, (size_t)2 * d_in * sizeof(float), stream);
    if (prev_sums64) cudaMemsetAsync(prev_sums64, 0, (size_t)2 * d_in * sizeof(double), stream);
    return CGNN_OK;
  }
  if ((du == nullptr) == (demb == nullptr)) return CGNN_ERR_INVALID_ARG;
  const bool arrays_bwd = csr && csr->in_rowptr && csr->in_col && csr->in_w && csr->wsum &&
                          (!du_in || (csr->out_rowptr && csr->out_col && csr->out_w));
  const bool lean = csr && !csr->in_col && csr->agg_in && csr->agg_kind == AGG_SAGE;
  if (!z || !t_in || !W || !csr || !csr->graph_meta || !(arrays_bwd || lean) || !ptr || !workspace) return CGNN_ERR_INVALID_ARG;
  if (d_in % 4 == 0 && (!aligned16(t_in) || (scratch && !aligned16(scratch)))) return CGNN_ERR_INVALID_ARG;
  if (du_in && !scratch) return CGNN_ERR_INVALID_ARG;
  if (prev_sums && (!du_in || !prev_mean || !prev_rstd)) return CGNN_ERR_INVALID_ARG;
  if (bn && (!bn->scale || !bn->mean || !bn->rstd || (bn->train && (!bn->s1 || !bn->s2)))) return CGNN_ERR_INVALID_ARG;
#ifndef CGNN_EMU
  // Narrow first layer whose input needs no gradient: dW = dz^T [u || agg], dbias in one pass, no tensor cores.
  if (tensor_cores_enabled() && !du_in && agg && d_in <= 8) {
    int g0 = 0;
    const int rc0 = launch_first_bwd(AGG_SAGE, du, demb, z, act_out, bn, t_in, agg, act_in, csr, num_graphs, d_in, H, max_nodes,
                                     max_edges, (float*)workspace, &g0, workspace_bytes, stream);
    if (rc0 > 0) return rc0;
    if (rc0 == CGNN_OK) {
      const int stride = H * 2 * d_in + H;
      ReduceQueue rq(stream);
      rq.add((const float*)workspace, g0, stride, H, 2 * d_in, 2 * d_in, dW);
      rq.add((const float*)workspace + H * 2 * d_in, g0, stride, 1, H, H, dbias);
      return rq.flush();
    }
  }
  // Wide layers (H = d_in = 256): dz pass, K-looped contractions, transposed gather (wide_tc.cu; scratch = 3 x [rows, 256]).
  if (tensor_cores_enabled() && wide_shape(d_in, H)) {
    const int rcw = launch_sage_bwd_wide(du, demb, z, act_out, bn, t_in, agg, act_in, W, csr, num_graphs, rows, d_in, H, max_nodes,
                                         max_edges, dW, dbias, du_in, prev_mean, prev_rstd, prev_sums, prev_sums64, scratch, workspace,
                                         workspace_bytes, stream);
    if (rcw >= 0) return rcw;
  }
  // Tensor-core generation: tcgen05 contractions (dz on load, [d_u || d_agg], dW, dbias) + transposed gather kernel.
  // The gather runs second: its coverage is settled before the contractions launch.
  if (tensor_cores_enabled() && agg && csr->agg_out && csr->row_graph && csr->agg_kind == AGG_SAGE &&
      (!du_in || (aligned16(scratch) && gather_supported(d_in, max_nodes, max_edges)))) {
    const int part_stride = H * 2 * d_in + H;
    const size_t region_a = (size_t)160 * part_stride * sizeof(float);   // partial records of <= 160 CTAs
    if (workspace_bytes > region_a + (size_t)2 * 160 * 2 * d_in * sizeof(float)) {
      int g1 = 0, g2 = 0;
      float* direct = du_in ? scratch : nullptr;
      float* nbr = du_in ? scratch + (size_t)rows * d_in : nullptr;
      int rc = launch_sage_bwd_gemm(du, demb, csr->row_graph, csr->graph_meta, z, act_out, bn, t_in, agg, act_in, W, rows, d_in, H,
                                    direct, nbr, (float*)workspace, part_stride, H * 2 * d_in, &g1, region_a, stream);
      if (rc > 0) return rc;
      if (rc == CGNN_OK) {
        ReduceQueue rq(stream);
        rq.add((const float*)workspace, g1, part_stride, H, 2 * d_in, 2 * d_in, dW);
        rq.add((const float*)workspace + H * 2 * d_in, g1, part_stride, 1, H, H, dbias);
        if (!du_in) return rq.flush();
        GatherArgs ga{};
        ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_out;
        ga.C = d_in; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
        ga.src = nbr; ga.act = make_act(act_in); ga.direct = direct; ga.t_raw = t_in;
        ga.prev_mean = prev_mean; ga.prev_rstd = prev_rstd; ga.want_prev = prev_sums ? 1 : 0;
        ga.out = du_in;
        ga.partials = (float*)((char*)workspace + region_a); ga.part_stride = 2 * d_in;
        rc = launch_gather(GATHER_SAGE_BWD, ga, &g2, stream);
        if (rc != CGNN_OK) return rc;
        if (prev_sums) rq.add(ga.partials, g2, 2 * d_in, 2, d_in, d_in, prev_sums, 0, prev_sums64);     // all three after the gather: one launch
        return rq.flush();
      }
    }
  }
#endif
  if (!arrays_bwd) return CGNN_ERR_NEED_CSR;       // the generic kernels walk the CSR arrays
  const DeviceInfo dev = device_info();
  SageBwdArgs a;
  a.du = du; a.demb = demb; a.z = z; a.act_out = make_act(act_out); a.bn = make_bn_bwd(bn);
  a.t_in = t_in; a.act_in = make_act(act_in); a.W = W;
  a.in_rowptr = csr->in_rowptr; a.in_col = csr->in_col; a.in_w = csr->in_w; a.wsum = csr->wsum;
  a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.K4 = round_up(d_in, 4); a.H4 = round_up(H, 4);
  a.ldc = 2 * a.K4 + 4; a.ldq = a.H4 + 4;
  a.max_nodes = max_nodes < 1 ? 1 : max_nodes;
  a.max_edges = max_edges;
  a.vec_h = (H % 4 == 0) && aligned16(z) && (!du || aligned16(du)) && (!demb || aligned16(demb));
  a.need_du = du_in ? 1 : 0;
  a.direct = scratch; a.nbr = scratch ? scratch + (size_t)rows * d_in : nullptr;
  const int ntiles_w = (a.H4 / 4) * (2 * a.K4 / 4);
  if (a.H4 > 128 || a.K4 > 128 || ntiles_w > 4 * kThreads) return CGNN_ERR_TILE_TOO_LARGE;
  int off = 0;
  a.o_w = off; off += a.H4 * 2 * a.K4;
  a.o_co = off; off += DZ_ROWS * a.H4;
  a.o_ci = off; off += 2 * a.K4;
  a.o_u = off; off += a.max_nodes * a.K4;
  a.o_cat = off; off += kChunkRows * a.ldc;
  a.o_dq = off; off += kChunkRows * a.ldq;
  a.o_red = off; off += kWarps * a.H4;
  const int csr_w = cgnn::csr_words(a.max_nodes, a.max_edges);
  a.csr_smem = ((size_t)(off + csr_w) * sizeof(float) <= (size_t)dev.smem_optin) ? 1 : 0;
  a.o_csr = off;
  if (a.csr_smem) off += csr_w;
  const size_t smem = (size_t)off * sizeof(float);
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  a.o_pdw = 0; a.o_pdb = a.H4 * 2 * a.K4;
  a.part_stride = a.o_pdb + a.H4;
  int grid = persistent_grid(num_graphs, smem, dev, kThreads);
  const size_t rec = (size_t)a.part_stride * sizeof(float);
  if (workspace_bytes < rec) return CGNN_ERR_WORKSPACE;
  if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
  a.partials = (float*)workspace;
  const int cc = imax(pick_hc(a.H4), pick_hc(a.K4));
  const int maxt = ntiles_w <= kThreads ? 1 : (ntiles_w <= 2 * kThreads ? 2 : 4);
#define CGNN_SAGE_BWD(CC_, MT_)                                                                  \
  {                                                                                              \
    auto kfn = k_sage_bwd_a<CC_, MT_>;                                                           \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);                                           \
  }
  if (cc == 1) { if (maxt == 1) CGNN_SAGE_BWD(1, 1) else if (maxt == 2) CGNN_SAGE_BWD(1, 2) else CGNN_SAGE_BWD(1, 4) }
  else if (cc == 2) { if (maxt == 1) CGNN_SAGE_BWD(2, 1) else if (maxt == 2) CGNN_SAGE_BWD(2, 2) else CGNN_SAGE_BWD(2, 4) }
  else { if (maxt == 1) CGNN_SAGE_BWD(4, 1) else if (maxt == 2) CGNN_SAGE_BWD(4, 2) else CGNN_SAGE_BWD(4, 4) }
#undef CGNN_SAGE_BWD
  CGNN_CHECK_LAUNCH();
  // dW = [dW_self | dW_neigh]: the two halves sit K4 apart in the padded partial, d_in apart in dW
  int rc = CGNN_OK;
  {
    ReduceQueue rq(stream);
    rq.add(a.partials + a.o_pdw, grid, a.part_stride, H, d_in, 2 * a.K4, dW, 2 * d_in);
    rq.add(a.partials + a.o_pdw + a.K4, grid, a.part_stride, H, d_in, 2 * a.K4, dW + d_in, 2 * d_in);
    rq.add(a.partials + a.o_pdb, grid, a.part_stride, 1, H, a.H4, dbias);
    rc = rq.flush();
    if (rc) return rc;
  }
  if (!du_in) return CGNN_OK;

  // kernel B: transposed neighbour aggregation
  SageBwdBArgs b;
  b.direct = a.direct; b.nbr = a.nbr; b.t_in = t_in; b.act_in = a.act_in;
  b.out_rowptr = csr->out_rowptr; b.out_col = csr->out_col; b.out_w = csr->out_w;
  b.prev_mean = prev_mean; b.prev_rstd = prev_rstd; b.want_prev = prev_sums ? 1 : 0;
  b.meta = csr->graph_meta; b.B = num_graphs; b.K = d_in; b.K4 = a.K4; b.max_nodes = a.max_nodes;
  b.max_edges = a.max_edges;
  b.du_in = du_in;
  int offb = 0;
  b.o_g = offb; offb += a.max_nodes * a.K4;
  b.o_ci = offb; offb += 4 * a.K4;
  b.o_red = offb; offb += kWarps * 2 * a.K4;
  b.csr_smem = ((size_t)(offb + csr_w) * sizeof(float) <= (size_t)dev.smem_optin) ? 1 : 0;
  b.o_csr = offb;
  if (b.csr_smem) offb += csr_w;
  const size_t smem_b = (size_t)offb * sizeof(float);
  if (smem_b > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  int grid_b = persistent_grid(num_graphs, smem_b, dev, kThreads);
  // partials of kernel B live after kernel A's (the reduce kernels above still read those)
  const size_t used_a = (size_t)grid * rec;
  const size_t rec_b = (size_t)2 * a.K4 * sizeof(float);
  if (used_a + rec_b > workspace_bytes) return CGNN_ERR_WORKSPACE;
  if (used_a + (size_t)grid_b * rec_b > workspace_bytes) grid_b = (int)((workspace_bytes - used_a) / rec_b);
  b.partials = (float*)((char*)workspace + used_a);
  const int ccb = pick_hc(a.K4);
#define CGNN_SAGE_BWDB(CC_)                                                                      \
  {                                                                                              \
    auto kfn = k_sage_bwd_b<CC_>;                                                                \
    if (smem_b > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b); \
    CGNN_LAUNCH(kfn, grid_b, kThreads, smem_b, stream, b);                                       \
  }
  if (ccb == 1) CGNN_SAGE_BWDB(1) else if (ccb == 2) CGNN_SAGE_BWDB(2) else CGNN_SAGE_BWDB(4)
#undef CGNN_SAGE_BWDB
  CGNN_CHECK_LAUNCH();
  if (prev_sums) {
    rc = launch_reduce_partials(b.partials, grid_b, 2 * a.K4, 2, d_in, a.K4, prev_sums, stream, 0, prev_sums64);
    if (rc) return rc;
  }
  return CGNN_OK;
}

}  // extern "C"
