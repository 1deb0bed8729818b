// gcn.cu - K1 / K6: GCN layer forward and backward, one persistent CTA per subject graph.
//
// Forward  (reference models.py:84-114, fused with the *previous* layer's models.py:208-210):
//   u = dropout(relu(bn(t_in)))            on load, never materialised in HBM
//   P = u W^T                              subject tile in shared memory
//   z_i = sum_{e: dst=i} w^_e P_src(e)  +  dinv_i^2 P_i  +  b     (COO order, self-loop last)
//   per-channel Welford statistics of z for this layer's BatchNorm
// Backward (autograd of the same lines): dz tile in shared memory, transposed aggregation over the
//   by-source CSR, dW = dP^T u, du_in = dP W, and the BatchNorm backward sums of the previous
//   layer accumulated on the fly.
#include "tile.cuh"
#include "agg.cuh"

namespace cgnn {

struct GcnFwdArgs {
  const float* t_in; Act act; const float* W; const float* bias;
  const int32_t* in_rowptr; const int32_t* in_col; const float* in_wn; const float* dinv;
  const int32_t* meta; long long B;   // meta[g] = {first row, rows, first edge, edges}
  int K, H, K4, H4, ldx, max_nodes, max_edges, csr_smem;
  float* z; double* partials;
  // shared-memory offsets in floats
  int o_wt, o_scale, o_shift, o_bias, o_raw, o_x, o_p, o_st, o_csr;
};

// Pipeline per CTA (persistent over subjects g = blockIdx.x, +gridDim.x, ...):
//   cp.async double buffer of raw 64-row chunks  ->  BN/ReLU/dropout into the padded GEMM operand
//   ->  4x4 register-tile projection into the subject's P tile  ->  (all chunks done)
//   aggregation over the subject's CSR, staged in shared memory by cp.async while the projection runs.
// The first chunk of the NEXT subject is already in flight during the aggregation.
template <int HC>
__global__ void __launch_bounds__(kThreads) k_gcn_fwd(GcnFwdArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  float* s_wt = sm + p.o_wt;        // [K4][H4]  W transposed, zero padded
  float* s_scale = sm + p.o_scale;  // [K4]
  float* s_shift = sm + p.o_shift;  // [K4]
  float* s_bias = sm + p.o_bias;    // [H4]
  float* s_raw = sm + p.o_raw;      // [2][kChunkRows * K]  raw rows as they sit in HBM
  float* s_x = sm + p.o_x;          // [kChunkRows][ldx]    transformed, padded GEMM operand
  float* s_p = sm + p.o_p;          // [max_nodes][H4]
  float* s_cnt = sm + p.o_st;       // [kWarps]
  float* s_mean = s_cnt + kWarps;   // [kWarps][H4]
  float* s_m2 = s_mean + kWarps * p.H4;
  float* s_csr = sm + p.o_csr;      // staged CSR of the current subject (rp | col | wn | dinv)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = p.K, H = p.H, K4 = p.K4, H4 = p.H4, ldx = p.ldx;
  const int raw_stride = kChunkRows * K;
  const bool affine = p.act.scale != nullptr;

  for (int idx = tid; idx < K4 * H4; idx += kThreads) {
    const int k = idx / H4, h = idx - k * H4;
    s_wt[idx] = (k < K && h < H) ? p.W[h * K + k] : 0.0f;
  }
  stage_affine(p.act, K, K4, s_scale, s_shift);
  for (int h = tid; h < H4; h += kThreads) s_bias[h] = (h < H && p.bias) ? p.bias[h] : 0.0f;

  WarpStats<HC> st;
  st.init();
  const int tiles_x = H4 >> 2;
  const int ntiles = (kChunkRows >> 2) * tiles_x;

  // Subject metadata comes as one 16-byte record, loaded one subject ahead so its latency never shows.
  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  auto load_meta = [&](long long g) -> int4 {
    int4 m = make_int4(0, 0, 0, 0);
    if (g < p.B) { m = meta[g]; if (m.y > p.max_nodes) m.y = p.max_nodes; }   // host contract; never index past the tiles
    return m;
  };
  auto issue_chunk = [&](const int4& m, int r0, int buf) {
    const int rows = min(kChunkRows, m.y - r0);
    if (rows > 0) cp_async_words(s_raw + buf * raw_stride, p.t_in + ((long long)m.x + r0) * K, rows * K);
  };

  long long g = blockIdx.x;
  int4 cur = load_meta(g);
  int buf = 0;
  issue_chunk(cur, 0, 0);
  cp_async_commit();
  __syncthreads();   // constants staged

  while (g < p.B) {
    const long long g_next = g + gridDim.x;
    const int4 nxt = load_meta(g_next);
    const long long nb = cur.x;
    const int n = cur.y, eb = cur.z, m = cur.w;
    const bool csr_here = p.csr_smem && m <= p.max_edges;
    if (n == 0) {   // empty subject: keep the "next chunk is in flight" invariant
      issue_chunk(nxt, 0, buf ^ 1);
      cp_async_commit();
      buf ^= 1;
    }

    // ---- projection, kChunkRows rows at a time, next chunk always in flight ------------------
    for (int r0 = 0; r0 < n; r0 += kChunkRows) {
      const int rows = min(kChunkRows, n - r0);
      if (r0 + kChunkRows < n) issue_chunk(cur, r0 + kChunkRows, buf ^ 1);
      else issue_chunk(nxt, 0, buf ^ 1);
      cp_async_commit();
      if (r0 == 0) {
        // the subject's CSR rides behind the next chunk; needed only by the aggregation
        if (csr_here) stage_csr_async(s_csr, p.max_nodes, p.max_edges, p.in_rowptr, p.in_col, p.in_wn, p.dinv, nb, n, eb, m);
        cp_async_commit();
        cp_async_wait<2>();
      } else {
        cp_async_wait<1>();
      }
      __syncthreads();
      // BN affine + ReLU + dropout of the previous layer, raw chunk -> padded operand
      const float* raw = s_raw + buf * raw_stride;
      for (int idx = tid; idx < kChunkRows * K4; idx += kThreads) {
        const int r = idx / K4, c = idx - r * K4;
        float v = 0.0f;
        if (r < rows && c < K) {
          const uint32_t rh = p.act.drop ? drop_row_hash(p.act, p.act.row_base + nb + r0 + r) : 0u;
          v = act_fwd(p.act, affine, raw[r * K + c], s_scale[c], s_shift[c], rh, c);
        }
        s_x[r * ldx + c] = v;
      }
      __syncthreads();
      for (int t = tid; t < ntiles; t += kThreads) {
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        if (4 * ty >= rows) continue;
        float acc[4][4] = {};
        mma_4x4(s_x + 4 * ty * ldx, ldx, s_wt + 4 * tx, H4, K4, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = r0 + 4 * ty + i;
          if (row < n)
            *reinterpret_cast<float4*>(s_p + row * H4 + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        }
      }
      buf ^= 1;
    }
    if (n <= kChunkRows) cp_async_wait<0>();   // single-chunk subject: its CSR group was the most recent one
    __syncthreads();

    // ---- aggregation: one warp per destination row, lanes over channels -------------------
    const float* dinv_g = p.dinv + nb;
    RowCsr rc{p.in_rowptr + nb, p.in_col, p.in_wn};
    if (csr_here) rc = staged_csr(s_csr, p.max_nodes, p.max_edges, eb, &dinv_g);
    for (int i = warp; i < n; i += kWarps) {
      float acc[HC];
#pragma unroll
      for (int j = 0; j < HC; ++j) acc[j] = 0.0f;
      gather_row<HC, true>(rc, i, nb, n, s_p, H4, H4, acc);
      const float d = dinv_g[i];
      const float wself = __fmul_rn(d, d);
      float inv;
      st.begin_row(inv);
#pragma unroll
      for (int j = 0; j < HC; ++j) {
        const int ch = lane + 32 * j;
        if (ch < H) {
          float v = __fadd_rn(acc[j], __fmul_rn(s_p[i * H4 + ch], wself));
          v = __fadd_rn(v, s_bias[ch]);
          p.z[(nb + i) * H + ch] = v;
          st.w[j].push(v, inv);
        }
      }
    }
    __syncthreads();  // s_p and the staged CSR are rewritten by the next subject
    g = g_next;
    cur = nxt;
  }
  cp_async_wait<0>();

  if (p.partials) {
    st.deposit(s_cnt, s_mean, s_m2, H4, H4);
    __syncthreads();
    cta_write_stats(s_cnt, s_mean, s_m2, H4, H, p.partials + (size_t)blockIdx.x * (1 + 2 * H));
  }
}

// ------------------------------------------------------------------------------------------
struct GcnBwdArgs {
  const float* du; const float* demb; const float* z; Act act_out; BnBwdDev bn;
  const float* t_in; Act act_in; const float* W;
  const int32_t* out_rowptr; const int32_t* out_col; const float* out_wn; const float* dinv;
  const int32_t* meta; long long B;
  int K, H, K4, H4, ldp, ldu, max_nodes, max_edges, csr_smem, vec_h;
  float* du_in; const float* prev_mean; const float* prev_rstd; int want_prev;
  float* partials; int part_stride, o_pdw, o_pdb, o_pprev;
  // shared-memory offsets (floats)
  int o_w, o_co, o_ci, o_dz, o_dp, o_u, o_raw, o_red, o_csr;
};

// Per-channel constant rows of the layer input staged in shared memory.
enum { CI_SCALE = 0, CI_SHIFT, CI_MEAN, CI_RSTD, CI_ROWS };   // x K4

template <int HC, int MAXT>
__global__ void __launch_bounds__(kThreads) k_gcn_bwd(GcnBwdArgs p) {
  act_salt(p.act_out); act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  float* s_w = sm + p.o_w;      // [H4][K4] natural layout, zero padded
  float* s_co = sm + p.o_co;    // [DZ_ROWS][H4]
  float* s_ci = sm + p.o_ci;    // [CI_ROWS][K4]
  float* s_dz = sm + p.o_dz;    // [max_nodes][H4]
  float* s_dp = sm + p.o_dp;    // [kChunkRows][ldp]
  float* s_u = sm + p.o_u;      // [kChunkRows][ldu]   transformed layer input (GEMM operand)
  float* s_raw = sm + p.o_raw;  // [2][kChunkRows*K]   raw layer input as it sits in HBM (cp.async double buffer)
  float* s_red = sm + p.o_red;  // reduction scratch
  float* s_csr = sm + p.o_csr;  // staged by-source CSR of the current subject

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = p.K, H = p.H, K4 = p.K4, H4 = p.H4, ldp = p.ldp, ldu = p.ldu;
  const int raw_stride = kChunkRows * K;
  const bool aff_out = p.act_out.scale != nullptr, aff_in = p.act_in.scale != nullptr;

  for (int idx = tid; idx < H4 * K4; idx += kThreads) {
    const int h = idx / K4, k = idx - h * K4;
    s_w[idx] = (h < H && k < K) ? p.W[h * K + k] : 0.0f;
  }
  stage_dz_consts(p.act_out, p.bn, H, H4, s_co);
  stage_affine(p.act_in, K, K4, s_ci + CI_SCALE * K4, s_ci + CI_SHIFT * K4);
  for (int c = tid; c < K4; c += kThreads) {
    const bool ok = c < K && p.want_prev;
    s_ci[CI_MEAN * K4 + c] = ok ? p.prev_mean[c] : 0.0f;
    s_ci[CI_RSTD * K4 + c] = ok ? p.prev_rstd[c] : 0.0f;
  }

  const int tk = K4 >> 2;                         // channel quads of the input width
  const int ntiles_w = (H4 >> 2) * tk;            // dW register tiles
  const int ntu = (kThreads / tk) * tk;           // threads used for du_in tiles (fixed quad per thread)
  const int ntiles_u = (kChunkRows >> 2) * tk;

  float acc_w[MAXT][4][4];
#pragma unroll
  for (int it = 0; it < MAXT; ++it)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc_w[it][i][j] = 0.0f;
  float acc_db[HC];
#pragma unroll
  for (int j = 0; j < HC; ++j) acc_db[j] = 0.0f;
  float ps1[4] = {0.f, 0.f, 0.f, 0.f}, ps2[4] = {0.f, 0.f, 0.f, 0.f};

  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  auto load_meta = [&](long long g) -> int4 {
    int4 m = make_int4(0, 0, 0, 0);
    if (g < p.B) { m = meta[g]; if (m.y > p.max_nodes) m.y = p.max_nodes; }
    return m;
  };
  auto issue_chunk = [&](const int4& m, int r0, int buf) {
    const int rows = min(kChunkRows, m.y - r0);
    if (rows > 0) cp_async_words(s_raw + buf * raw_stride, p.t_in + ((long long)m.x + r0) * K, rows * K);
  };

  long long g = blockIdx.x;
  int4 cur = load_meta(g);
  int buf = 0;
  issue_chunk(cur, 0, 0);
  cp_async_commit();
  __syncthreads();   // constants staged

  while (g < p.B) {
    const long long g_next = g + gridDim.x;
    const int4 nxt = load_meta(g_next);
    const long long nb = cur.x;
    const int n = cur.y, eb = cur.z, m = cur.w;
    const bool csr_here = p.csr_smem && m <= p.max_edges;
    const float inv_n = pool_bwd_scale(n);
    if (csr_here) stage_csr_async(s_csr, p.max_nodes, p.max_edges, p.out_rowptr, p.out_col, p.out_wn, p.dinv, nb, n, eb, m);
    cp_async_commit();

    // ---- phase 1: dz tile (streams z and the upstream gradient once) -------------------------
    if (p.vec_h) {
      const int q4 = H4 >> 2;
      const int total = n * q4;
      for (int base = tid; base < total; base += 4 * kThreads) {
        float4 zv[4], uv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * kThreads;
          if (idx < total) {
            const int i = idx / q4, c = (idx - i * q4) << 2;
            zv[u] = *reinterpret_cast<const float4*>(p.z + (nb + i) * H + c);
            if (p.du) uv[u] = *reinterpret_cast<const float4*>(p.du + (nb + i) * H + c);
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * kThreads;
          if (idx < total) {
            const int i = idx / q4, c = (idx - i * q4) << 2;
            if (!p.du) {
              const float4 e = *reinterpret_cast<const float4*>(p.demb + g * H + c);
              uv[u] = make_float4(e.x * inv_n, e.y * inv_n, e.z * inv_n, e.w * inv_n);
            }
            const uint32_t rh = p.act_out.drop ? drop_row_hash(p.act_out, p.act_out.row_base + nb + i) : 0u;
            float4 o;
            o.x = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, zv[u].x, uv[u].x, rh, c);
            o.y = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, zv[u].y, uv[u].y, rh, c + 1);
            o.z = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, zv[u].z, uv[u].z, rh, c + 2);
            o.w = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, zv[u].w, uv[u].w, rh, c + 3);
            *reinterpret_cast<float4*>(s_dz + i * H4 + c) = o;
          }
        }
      }
    } else {
      for (int idx = tid; idx < n * H4; idx += kThreads) {
        const int i = idx / H4, c = idx - i * H4;
        float dz = 0.0f;
        if (c < H) {
          const float t = p.z[(nb + i) * H + c];
          const float up = p.du ? p.du[(nb + i) * H + c] : p.demb[g * H + c] * inv_n;
          const uint32_t rh = p.act_out.drop ? drop_row_hash(p.act_out, p.act_out.row_base + nb + i) : 0u;
          dz = staged_dz(p.act_out, p.bn, s_co, H4, aff_out, t, up, rh, c);
        }
        s_dz[idx] = dz;
      }
    }
    if (n == 0) {   // empty subject: keep the "next chunk is in flight" invariant
      issue_chunk(nxt, 0, buf ^ 1);
      cp_async_commit();
      buf ^= 1;
    }

    const float* dinv_g = p.dinv + nb;
    RowCsr rc{p.out_rowptr + nb, p.out_col, p.out_wn};
    if (csr_here) rc = staged_csr(s_csr, p.max_nodes, p.max_edges, eb, &dinv_g);

    // ---- phase 2: row chunks --------------------------------------------------------------
    for (int j0 = 0; j0 < n; j0 += kChunkRows) {
      const int rows = min(kChunkRows, n - j0);
      cp_async_wait<0>();   // this chunk's raw rows and the subject's CSR have landed (this thread's copies)
      __syncthreads();      // ... everyone's; s_dz complete; previous chunk's readers are done
      if (j0 + kChunkRows < n) issue_chunk(cur, j0 + kChunkRows, buf ^ 1);
      else issue_chunk(nxt, 0, buf ^ 1);
      cp_async_commit();
      if (j0 == 0) {   // bias gradient: column sums of dz
        for (int i = warp; i < n; i += kWarps) {
#pragma unroll
          for (int j = 0; j < HC; ++j) {
            const int ch = lane + 32 * j;
            if (ch < H4) acc_db[j] += s_dz[i * H4 + ch];
          }
        }
      }
      // (a) dP = A^T dz for the chunk's source rows (by-source CSR), self-loop included
      for (int r = warp; r < kChunkRows; r += kWarps) {
        float acc[HC];
#pragma unroll
        for (int j = 0; j < HC; ++j) acc[j] = 0.0f;
        if (r < rows) {
          const int jr = j0 + r;
          gather_row<HC, false>(rc, jr, nb, n, s_dz, H4, H4, acc);
          const float d = dinv_g[jr];
          const float wself = d * d;
#pragma unroll
          for (int j = 0; j < HC; ++j) {
            const int ch = lane + 32 * j;
            if (ch < H4) acc[j] = fmaf(s_dz[jr * H4 + ch], wself, acc[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < HC; ++j) {
          const int ch = lane + 32 * j;
          if (ch < H4) s_dp[r * ldp + ch] = acc[j];
        }
      }
      // (b) this layer's input rows: raw chunk -> transformed operand
      const float* raw = s_raw + buf * raw_stride;
      for (int idx = tid; idx < kChunkRows * K4; idx += kThreads) {
        const int r = idx / K4, c = idx - r * K4;
        float v = 0.0f;
        if (r < rows && c < K) {
          const uint32_t rh = p.act_in.drop ? drop_row_hash(p.act_in, p.act_in.row_base + nb + j0 + r) : 0u;
          v = act_fwd(p.act_in, aff_in, raw[r * K + c], s_ci[CI_SCALE * K4 + c], s_ci[CI_SHIFT * K4 + c], rh, c);
        }
        s_u[r * ldu + c] = v;
      }
      __syncthreads();
      // (c) dW += dP^T u
#pragma unroll
      for (int it = 0; it < MAXT; ++it) {
        const int t = tid + it * kThreads;
        if (t < ntiles_w) {
          const int th = t / tk, tq = t - th * tk;
          outer_4x4(s_dp + 4 * th, ldp, s_u + 4 * tq, ldu, rows, acc_w[it]);
        }
      }
      // (d) du_in = dP W, plus the previous layer's BatchNorm backward sums
      if (p.du_in && tid < ntu) {
        const int tx = tid % tk;
        for (int t = tid; t < ntiles_u; t += ntu) {
          const int ty = t / tk;
          if (4 * ty >= rows) continue;
          float acc[4][4] = {};
          mma_4x4(s_dp + 4 * ty * ldp, ldp, s_w + 4 * tx, K4, H4, acc);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = 4 * ty + i;
            if (r >= rows) continue;
            const long long grow = nb + j0 + r;
            const uint32_t rh = (p.want_prev && p.act_in.drop) ? drop_row_hash(p.act_in, p.act_in.row_base + grow) : 0u;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int ch = 4 * tx + q;
              if (ch < K) {
                p.du_in[grow * K + ch] = acc[i][q];
                if (p.want_prev) {
                  const float t0 = raw[r * K + ch];
                  const float dyp = act_bwd(p.act_in, aff_in, t0, s_ci[CI_SCALE * K4 + ch], s_ci[CI_SHIFT * K4 + ch], rh, ch, acc[i][q]);
                  bn_sums_add(ps1[q], ps2[q], dyp, t0, s_ci[CI_MEAN * K4 + ch], s_ci[CI_RSTD * K4 + ch]);
                }
              }
            }
          }
        }
      }
      buf ^= 1;
    }
    __syncthreads();   // s_dz, the staged CSR and the chunk buffers are rewritten by the next subject
    g = g_next;
    cur = nxt;
  }
  cp_async_wait<0>();

  // ---- per-CTA partial record: [dW H4*K4][db H4][prev 2*K4] ----------------------------------
  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
#pragma unroll
  for (int it = 0; it < MAXT; ++it) {
    const int t = tid + it * kThreads;
    if (t < ntiles_w) {
      const int th = t / tk, tq = t - th * tk;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(part + p.o_pdw + (4 * th + i) * K4 + 4 * tq) =
            make_float4(acc_w[it][i][0], acc_w[it][i][1], acc_w[it][i][2], acc_w[it][i][3]);
    }
  }
#pragma unroll
  for (int j = 0; j < HC; ++j) {
    const int ch = lane + 32 * j;
    if (ch < H4) s_red[warp * H4 + ch] = acc_db[j];
  }
  __syncthreads();
  for (int c = tid; c < H4; c += kThreads) part[p.o_pdb + c] = warp_rows_sum(s_red, H4, c);
  __syncthreads();
  if (p.want_prev) {
#pragma unroll
    for (int q = 0; q < 4; ++q) { s_red[tid * 8 + q] = ps1[q]; s_red[tid * 8 + 4 + q] = ps2[q]; }
    __syncthreads();
    for (int c = tid; c < 2 * K4; c += kThreads) {
      const int which = c / K4, ch = c - which * K4;
      part[p.o_pprev + c] = quad_sum(s_red, 8, which * 4, ntu, tk, ch >> 2, ch & 3);
    }
  }
}

}  // namespace cgnn

using namespace cgnn;

static bool csr_in_ok(const cgnn_csr_t* c) { return c && c->in_rowptr && c->in_col && c->in_wn && c->dinv && c->graph_meta; }
static bool csr_out_ok_(const cgnn_csr_t* c) { return c && c->out_rowptr && c->out_col && c->out_wn && c->dinv && c->graph_meta; }
// a lean batch: graph_meta + this family's blobs, no arrays (the tensor-core kernels read nothing else)
static bool csr_lean_gcn(const cgnn_csr_t* c) { return c && c->graph_meta && c->agg_in && c->agg_kind == AGG_GCN && !c->in_col; }
static bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

extern "C" {

int cgnn_gcn_layer_fwd(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias,
                       const cgnn_csr_t* csr, const int64_t* ptr, int64_t num_graphs, int64_t rows,
                       int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z, double* bn_stats,
                       void* workspace, size_t workspace_bytes, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || rows < 0 || d_in <= 0 || H <= 0 || max_nodes < 0 || max_edges < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) {  // a rank may hold no subjects: empty statistics record
    if (bn_stats) cudaMemsetAsync(bn_stats, 0, (size_t)(1 + 2 * H) * sizeof(double), stream);
    return CGNN_OK;
  }
  if (!t_in || !W || !(csr_in_ok(csr) || csr_lean_gcn(csr)) || !ptr || !z) return CGNN_ERR_INVALID_ARG;
  if (bn_stats && (!workspace || workspace_bytes < (size_t)(1 + 2 * H) * sizeof(double))) return CGNN_ERR_WORKSPACE;
  if (tensor_cores_enabled()) {   // warp-specialised hidden layer (TMA + tensor memory); also runs on the simulator
    int ws_grid = 0;
    const int rc = launch_gcn_fwd_ws(t_in, act, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, z,
                                     bn_stats ? (double*)workspace : nullptr, &ws_grid, workspace_bytes, stream);
    if (rc == CGNN_OK) return bn_stats ? launch_stats_merge((const double*)workspace, ws_grid, H, bn_stats, stream) : CGNN_OK;
    if (rc > 0) return rc;
  }
#ifndef CGNN_EMU
  if (tensor_cores_enabled()) {   // tcgen05 / TMEM editions for the shapes they cover
    int tc_grid = 0;
    int rc = launch_first_fwd(AGG_GCN, t_in, act, W, bias, csr, num_graphs, d_in, H, max_nodes, max_edges, z, nullptr,
                              bn_stats ? (double*)workspace : nullptr, &tc_grid, workspace_bytes, stream);
    if (rc == CGNN_OK) return bn_stats ? launch_stats_merge((const double*)workspace, tc_grid, H, bn_stats, stream) : CGNN_OK;
    if (rc > 0) return rc;
    rc = launch_gcn_fwd_wide(t_in, act, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, z, bn_stats ? 1 : 0,
                             &tc_grid, workspace, workspace_bytes, stream);
    if (rc == CGNN_OK) return bn_stats ? launch_stats_merge((const double*)workspace, tc_grid, H, bn_stats, stream) : CGNN_OK;
    if (rc > 0) return rc;
  }
#endif
  if (!csr_in_ok(csr)) return CGNN_ERR_NEED_CSR;     // the generic kernel walks the CSR arrays
  const DeviceInfo dev = device_info();
  GcnFwdArgs a;
  a.t_in = t_in; a.act = make_act(act); a.W = W; a.bias = bias;
  a.in_rowptr = csr->in_rowptr; a.in_col = csr->in_col; a.in_wn = csr->in_wn; a.dinv = csr->dinv;
  a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.K4 = round_up(d_in, 4); a.H4 = round_up(H, 4); a.ldx = a.K4 + 4;
  a.max_nodes = max_nodes < 1 ? 1 : max_nodes;
  a.max_edges = max_edges;
  a.z = z;
  if (a.H4 > 256) return CGNN_ERR_TILE_TOO_LARGE;
  int off = 0;
  a.o_wt = off; off += a.K4 * a.H4;
  a.o_scale = off; off += a.K4;
  a.o_shift = off; off += a.K4;
  a.o_bias = off; off += a.H4;
  a.o_raw = off; off += 2 * round_up(kChunkRows * d_in, 4);
  a.o_x = off; off += kChunkRows * a.ldx;
  a.o_p = off; off += a.max_nodes * a.H4;
  a.o_st = off; off += round_up(kWarps + 2 * kWarps * a.H4, 4);
  // the subject's CSR goes to shared memory when it fits next to the tiles, else rows read it from L2
  const int csr_words = cgnn::csr_words(a.max_nodes, a.max_edges);
  a.csr_smem = ((size_t)(off + csr_words) * sizeof(float) <= (size_t)dev.smem_optin) ? 1 : 0;
  a.o_csr = off;
  if (a.csr_smem) off += csr_words;
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
  const int hc = pick_hc(a.H4);
#define CGNN_GCN_FWD(HC_)                                                                        \
  {                                                                                              \
    auto kfn = k_gcn_fwd<HC_>;                                                                   \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);                                           \
  }
  if (hc == 1) CGNN_GCN_FWD(1) else if (hc == 2) CGNN_GCN_FWD(2) else if (hc == 4) CGNN_GCN_FWD(4) else CGNN_GCN_FWD(8)
#undef CGNN_GCN_FWD
  CGNN_CHECK_LAUNCH();
  if (bn_stats) return launch_stats_merge(a.partials, grid, H, bn_stats, stream);
  return CGNN_OK;
}

int cgnn_gcn_layer_fwd_pool(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                            const int64_t* ptr, int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes,
                            int32_t max_edges, const cgnn_act_t* act_out, float* emb, cgnn_stream_t stream_) {
  (void)ptr;
  if (num_graphs < 0 || rows < 0 || d_in <= 0 || H <= 0 || max_nodes < 0 || max_edges < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) return CGNN_OK;
  if (rows == 0) return CGNN_ERR_UNSUPPORTED;   // subjects without a row: cgnn_pool_fwd writes their embeddings
  if (!t_in || !W || !csr || !csr->graph_meta || !csr->agg_in || !emb) return CGNN_ERR_INVALID_ARG;
  if (!tensor_cores_enabled()) return CGNN_ERR_UNSUPPORTED;
  const int rc = launch_gcn_fwd_ws_pool(t_in, act, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, act_out, emb,
                                        (cudaStream_t)stream_);
  if (rc == CGNN_OK) return CGNN_OK;
  return rc > 0 ? rc : CGNN_ERR_UNSUPPORTED;
}

int cgnn_gcn_layer_bwd(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out,
                       const cgnn_bn_bwd_t* bn, const float* t_in, const cgnn_act_t* act_in, const float* W,
                       const cgnn_csr_t* csr, const int64_t* ptr, int64_t num_graphs, int64_t rows,
                       int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* dW, float* dbias,
                       float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64, float* scratch,
                       void* workspace, size_t workspace_bytes, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (max_edges < 0) return CGNN_ERR_INVALID_ARG;
  if (!dW || !dbias || num_graphs < 0 || rows < 0 || d_in <= 0 || H <= 0 || max_nodes < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) {  // a rank may hold no subjects: zero contributions
    cudaMemsetAsync(dW, 0, (size_t)H * d_in * sizeof(float), stream);
    cudaMemsetAsync(dbias, 0, (size_t)H * sizeof(float), stream);
    if (prev_sums) cudaMemsetAsync(prev_sums, 0, (size_t)2 * d_in * sizeof(float), stream);
    if (prev_sums64) cudaMemsetAsync(prev_sums64, 0, (size_t)2 * d_in * sizeof(double), stream);
    return CGNN_OK;
  }
  if ((du == nullptr) == (demb == nullptr)) return CGNN_ERR_INVALID_ARG;
  if (!z || !t_in || !W || !(csr_out_ok_(csr) || csr_lean_gcn(csr)) || !ptr || !workspace) return CGNN_ERR_INVALID_ARG;
  if (prev_sums && (!du_in || !prev_mean || !prev_rstd)) return CGNN_ERR_INVALID_ARG;
  if (bn && (!bn->scale || !bn->mean || !bn->rstd || (bn->train && (!bn->s1 || !bn->s2)))) return CGNN_ERR_INVALID_ARG;
#ifndef CGNN_EMU
  // Narrow first layer whose input needs no gradient: dW = dz^T (A^ u), dbias in one pass, no tensor cores.
  if (tensor_cores_enabled() && !du_in && d_in <= 8) {
    int g0 = 0;
    const int rc0 = launch_first_bwd(AGG_GCN, du, demb, z, act_out, bn, t_in, nullptr, act_in, csr, num_graphs, d_in, H, max_nodes,
                                     max_edges, (float*)workspace, &g0, workspace_bytes, stream);
    if (rc0 > 0) return rc0;
    if (rc0 == CGNN_OK) {
      const int stride = H * d_in + H;
      ReduceQueue rq(stream);
      rq.add((const float*)workspace, g0, stride, H, d_in, d_in, dW);
      rq.add((const float*)workspace + H * d_in, g0, stride, 1, H, H, dbias);
      return rq.flush();
    }
  }
  // Wide layers (H = d_in = 256): gather + K-looped contractions (wide_tc.cu).
  if (tensor_cores_enabled() && wide_shape(d_in, H)) {
    const int rcw = launch_gcn_bwd_wide(du, demb, z, act_out, bn, t_in, act_in, W, csr, ptr, num_graphs, rows, d_in, H, max_nodes,
                                        max_edges, dW, dbias, du_in, prev_mean, prev_rstd, prev_sums, prev_sums64, scratch, workspace,
                                        workspace_bytes, stream);
    if (rcw >= 0) return rcw;
  }
  // Tensor-core generation: gather kernel (dz on load, dP = A^^T dz, dbias) + tcgen05 contractions (du_in, dW).
  const size_t region_a = (size_t)2 * 160 * 128 * sizeof(float);   // dbias partials of <= 2 CTAs per SM
  const int part_stride = H * d_in + 2 * d_in;
  if (tensor_cores_enabled() && scratch && csr->agg_out && csr->agg_kind == AGG_GCN && aligned16(z) && (!du || aligned16(du)) &&
      (!demb || aligned16(demb)) && workspace_bytes > region_a && gather_supported(H, max_nodes, max_edges) &&
      gcn_bwd_gemm_supported(scratch, t_in, du_in, rows, d_in, H, part_stride, workspace_bytes - region_a)) {
    GatherArgs ga{};
    ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_out;
    ga.C = H; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
    ga.src = z; ga.act = make_act(act_out); ga.du = du; ga.demb = demb; ga.bn = make_bn_bwd(bn);
    ga.out = scratch; ga.partials = (float*)workspace; ga.part_stride = H;
    int g1 = 0, g2 = 0;
    int rc = launch_gather(GATHER_GCN_BWD, ga, &g1, stream);
    if (rc != CGNN_OK) return rc;
    float* parts_b = (float*)((char*)workspace + region_a);
    rc = launch_gcn_bwd_gemm(scratch, t_in, act_in, W, rows, d_in, H, du_in, prev_mean, prev_rstd, prev_sums ? 1 : 0,
                             parts_b, part_stride, H * d_in, &g2, workspace_bytes - region_a, stream);
    if (rc != CGNN_OK) return rc;
    ReduceQueue rq(stream);
    rq.add((const float*)workspace, g1, H, 1, H, H, dbias);
    rq.add(parts_b, g2, part_stride, H, d_in, d_in, dW);
    if (prev_sums) rq.add(parts_b + H * d_in, g2, part_stride, 2, d_in, d_in, prev_sums, 0, prev_sums64);
    return rq.flush();
  }
#endif
  if (!csr_out_ok_(csr)) return CGNN_ERR_NEED_CSR;   // the generic kernel walks the CSR arrays
  const DeviceInfo dev = device_info();
  GcnBwdArgs a;
  a.du = du; a.demb = demb; a.z = z; a.act_out = make_act(act_out); a.bn = make_bn_bwd(bn);
  a.t_in = t_in; a.act_in = make_act(act_in); a.W = W;
  a.out_rowptr = csr->out_rowptr; a.out_col = csr->out_col; a.out_wn = csr->out_wn; a.dinv = csr->dinv;
  a.meta = csr->graph_meta; a.B = num_graphs;
  a.K = d_in; a.H = H; a.K4 = round_up(d_in, 4); a.H4 = round_up(H, 4);
  a.ldp = a.H4 + 4; a.ldu = a.K4 + 4;
  a.max_nodes = max_nodes < 1 ? 1 : max_nodes;
  a.max_edges = max_edges;
  a.vec_h = (H % 4 == 0) && aligned16(z) && (!du || aligned16(du)) && (!demb || aligned16(demb));
  a.du_in = du_in; a.prev_mean = prev_mean; a.prev_rstd = prev_rstd; a.want_prev = prev_sums ? 1 : 0;
  const int ntiles_w = (a.H4 / 4) * (a.K4 / 4);
  if (a.H4 > 128 || ntiles_w > 4 * kThreads) return CGNN_ERR_TILE_TOO_LARGE;
  int off = 0;
  a.o_w = off; off += a.H4 * a.K4;
  a.o_co = off; off += DZ_ROWS * a.H4;
  a.o_ci = off; off += CI_ROWS * a.K4;
  a.o_dz = off; off += a.max_nodes * a.H4;
  a.o_dp = off; off += kChunkRows * a.ldp;
  a.o_u = off; off += kChunkRows * a.ldu;
  a.o_raw = off; off += 2 * kChunkRows * d_in;
  a.o_red = off; off += (kThreads * 8 > kWarps * a.H4 ? kThreads * 8 : kWarps * a.H4);
  const int csr_w = cgnn::csr_words(a.max_nodes, a.max_edges);
  a.csr_smem = ((size_t)(off + csr_w) * sizeof(float) <= (size_t)dev.smem_optin) ? 1 : 0;
  a.o_csr = off;
  if (a.csr_smem) off += csr_w;
  const size_t smem = (size_t)off * sizeof(float);
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  a.o_pdw = 0; a.o_pdb = a.H4 * a.K4; a.o_pprev = a.o_pdb + a.H4;
  a.part_stride = a.o_pprev + 2 * a.K4;
  int grid = persistent_grid(num_graphs > 0 ? num_graphs : 1, smem, dev, kThreads);
  const size_t rec = (size_t)a.part_stride * sizeof(float);
  if (workspace_bytes < rec) return CGNN_ERR_WORKSPACE;
  if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
  a.partials = (float*)workspace;
  const int hc = pick_hc(a.H4);
  const int maxt = ntiles_w <= kThreads ? 1 : (ntiles_w <= 2 * kThreads ? 2 : 4);
#define CGNN_GCN_BWD(HC_, MT_)                                                                   \
  {                                                                                              \
    auto kfn = k_gcn_bwd<HC_, MT_>;                                                              \
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);                                           \
  }
  if (hc == 1) { if (maxt == 1) CGNN_GCN_BWD(1, 1) else if (maxt == 2) CGNN_GCN_BWD(1, 2) else CGNN_GCN_BWD(1, 4) }
  else if (hc == 2) { if (maxt == 1) CGNN_GCN_BWD(2, 1) else if (maxt == 2) CGNN_GCN_BWD(2, 2) else CGNN_GCN_BWD(2, 4) }
  else { if (maxt == 1) CGNN_GCN_BWD(4, 1) else if (maxt == 2) CGNN_GCN_BWD(4, 2) else CGNN_GCN_BWD(4, 4) }
#undef CGNN_GCN_BWD
  CGNN_CHECK_LAUNCH();
  ReduceQueue rq(stream);
  rq.add(a.partials + a.o_pdw, grid, a.part_stride, H, d_in, a.K4, dW);
  rq.add(a.partials + a.o_pdb, grid, a.part_stride, 1, H, a.H4, dbias);
  if (prev_sums) rq.add(a.partials + a.o_pprev, grid, a.part_stride, 2, d_in, a.K4, prev_sums, 0, prev_sums64);
  return rq.flush();
}

}  // extern "C"
