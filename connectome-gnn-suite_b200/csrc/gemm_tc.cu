// gemm_tc.cu - the dense half of the tensor-core generation of layer kernels (sm_100a only).
//
// Row-tile streaming kernels: TR rows of the batch at a time, operands split into TF32 hi/lo parts and written as
// swizzled canonical tiles, products issued by one thread as tcgen05.mma kind::tf32 (three terms: lo*hi, hi*lo,
// hi*hi; fp32 accumulators in tensor memory), results read back with tcgen05.ld.  The subject structure is gone
// at this point - the gathers around these contractions live in agg.cu.
//
//   k_sage_fwd_gemm   z = relu([u || agg] W^T + b), BatchNorm partial statistics        (reference models.py:151-152)
//   k_gcn_bwd_gemm    du_in = dP W,  dW += dP^T u,  BatchNorm-backward sums of the layer below
//                                                                            (autograd of reference models.py:111)
//   k_sage_bwd_gemm   dz from z / upstream / BatchNorm backward on load,  [d_u || d_agg] = dz W,
//                     dW += dz^T [u || agg],  dbias                  (autograd of reference models.py:151-152)
//
// X B products (contraction over channels) read K-major 128B-swizzled tiles, X^T Y products (contraction over the
// rows of the tile) read MN-major SWIZZLE_128B_BASE32B tiles - the only MN-major layout for tf32; see tc05.cuh.
// Every thread owns a fixed channel quad of the tile (rowtile.cuh), so the per-channel constants sit in registers.
#include "agg.cuh"
#include "rowtile.cuh"
#include "tile.cuh"

namespace cgnn {
#ifndef CGNN_EMU

static_assert(kThreads == 512, "the drain / staging maps below assume 16 warps");
constexpr int kRows = 128;

__device__ __forceinline__ float f4_get(const float4& v, int j) { return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w)); }

// W[n][k] (row stride ldw, zero beyond n_valid / k_valid) -> hi/lo K-major operand of `rows` rows, KP padded channels
__device__ __forceinline__ void stage_weight_kmajor(const float* __restrict__ W, int ldw, int n_valid, int k_valid, int rows,
                                                    int KP, unsigned char* hi, unsigned char* lo, int nthreads = kThreads) {
  const int Q = KP >> 2;
  for (int idx = threadIdx.x; idx < rows * Q; idx += nthreads) {
    const int n = idx / Q, q = idx - n * Q;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n < n_valid) v = rt::ld_quad<false>(W, n, ldw, 4 * q);
    v = rt::mask_quad(v, 4 * q, k_valid);
    float4 h, l;
    tc::split4(v, h, l);
    const uint32_t off = rt::kmajor_quad_offset(n, q, rows);
    rt::sts4(hi + off, h);
    rt::sts4(lo + off, l);
  }
}
// the transposed view: operand row n = column n of W, contraction index k = row of W:  element (n, k) = W[k][n]
__device__ __forceinline__ void stage_weight_transposed(const float* __restrict__ W, int ldw, int n_valid, int k_valid, int rows,
                                                        int KP, unsigned char* hi, unsigned char* lo) {
  const int Q = KP >> 2;
  for (int idx = threadIdx.x; idx < rows * Q; idx += kThreads) {
    const int n = idx / Q, q = idx - n * Q, k = 4 * q;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n < n_valid) {
      if (k + 0 < k_valid) v.x = W[(size_t)(k + 0) * ldw + n];
      if (k + 1 < k_valid) v.y = W[(size_t)(k + 1) * ldw + n];
      if (k + 2 < k_valid) v.z = W[(size_t)(k + 2) * ldw + n];
      if (k + 3 < k_valid) v.w = W[(size_t)(k + 3) * ldw + n];
    }
    float4 h, l;
    tc::split4(v, h, l);
    const uint32_t off = rt::kmajor_quad_offset(n, q, rows);
    rt::sts4(hi + off, h);
    rt::sts4(lo + off, l);
  }
}

// ================================================================================================================
// GraphSAGE forward contraction
// ================================================================================================================
struct SageFwdGemmArgs {
  const float* t_in; Act act; const float* agg; const float* W; const float* bias;
  long long rows; int C, H;
  float* z; double* partials;
  uint32_t tmem_cols; int o_stage;
};

// KB = padded K / 32 (K = 2C), HB = H / 32.  WIDE: C = 16 KB is a multiple of 32 - the u and agg halves are two quad
// maps with 16-byte loads; otherwise one element-wise map over the padded K (first layer, C = 5).
template <int KB, int HB, bool WIDE, int NT>
__global__ void __launch_bounds__(NT, 1) k_sage_fwd_gemm(SageFwdGemmArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  constexpr int KP = 32 * KB, H = 32 * HB, TR = kRows;
  constexpr int A_HALF = KB * TR * 128, B_HALF = KB * H * 128;
  constexpr int QC = WIDE ? KP / 8 : KP / 4;           // quads per row of one loaded tensor (wide) / of the padded K
  using MC = rt::QuadMap<QC, TR, NT>;
  constexpr int QH = H / 4;
  using MH = rt::QuadMap<QH, TR, NT>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  unsigned char* a_hi = base;
  unsigned char* a_lo = a_hi + A_HALF;
  unsigned char* b_hi = a_lo + A_HALF;
  unsigned char* b_lo = b_hi + B_HALF;
  float* s_scale = reinterpret_cast<float*>(b_lo + B_HALF);   // [KP] (element-wise path)
  float* s_shift = s_scale + KP;
  float4* stage = reinterpret_cast<float4*>(base + p.o_stage);   // [TR][H] swizzled; aliases the A operand when wide
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = p.C, K = 2 * C;
  const bool affine = p.act.scale != nullptr;

  if (warp == 0) tc::tmem_alloc(&tmem_base_s, p.tmem_cols);
  if (tid == 0) { tc::mbar_init(&mbar, 1); tc::fence_mbar_init(); }
  stage_weight_kmajor(p.W, K, H, K, H, KP, b_hi, b_lo, NT);
  if (!WIDE) {
    for (int c = tid; c < KP; c += NT) { s_scale[c] = (c < C && p.act.scale) ? p.act.scale[c] : (c < C ? 1.0f : 0.0f); s_shift[c] = (c < C && p.act.scale) ? p.act.shift[c] : 0.0f; }
    for (int i = tid; i < 2 * A_HALF / 16; i += NT) reinterpret_cast<float4*>(a_hi)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // this thread's input quad(s) and output quad
  const int qc = tid % QC, rc = tid / QC;
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act, 4 * qc, C);
  const rt::RowKey rk = rt::row_key(p.act);
  const uint32_t koff_u = rt::kmajor_quad_offset(rc, qc, TR);
  const uint32_t koff_a = WIDE ? rt::kmajor_quad_offset(rc, qc + QC, TR) : 0u;
  const int qh = tid % QH, rh = tid / QH;
  float bias4[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) bias4[j] = p.bias ? p.bias[4 * qh + j] : 0.0f;
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  const uint32_t a_hi_u = tc::smem_u32(a_hi), a_lo_u = tc::smem_u32(a_lo), b_hi_u = tc::smem_u32(b_hi), b_lo_u = tc::smem_u32(b_lo);
  const uint32_t idesc = tc::idesc_tf32(TR, H);
  const int ksteps = WIDE ? KP / 8 : (K + 7) / 8;
  const rt::OperandDescs od = rt::kmajor_descs(a_hi_u, a_lo_u, b_hi_u, b_lo_u);

  const long long ntiles = (p.rows + TR - 1) / TR;
  float4 pu[MC::NQ], pa[WIDE ? MC::NQ : 1];
  auto load_tile = [&](long long t) {
    const long long r0 = t * TR;
#pragma unroll
    for (int i = 0; i < MC::NQ; ++i) {
      const long long row = r0 + rc + i * MC::RS;
      float4 u = make_float4(0.f, 0.f, 0.f, 0.f), a = u;
      if (t < ntiles && row < p.rows) {
        if constexpr (WIDE) {
          u = rt::ld_quad<true>(p.t_in, row, C, 4 * qc);
          a = rt::ld_quad<true>(p.agg, row, C, 4 * qc);
        } else if (4 * qc < K) {
          float e[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int kk = 4 * qc + j;
            e[j] = kk < C ? p.t_in[row * C + kk] : (kk < K ? p.agg[row * C + (kk - C)] : 0.0f);
          }
          u = make_float4(e[0], e[1], e[2], e[3]);
        }
      }
      pu[i] = u;
      if constexpr (WIDE) pa[i] = a;
    }
  };

  const bool want_stats = p.partials != nullptr;
  QuadWelford wf;
  wf.init();

  // accumulators of the tile starting at row r0 (TMEM buffer b) -> bias + ReLU -> z, BatchNorm statistics
  auto epilogue = [&](long long r0, uint32_t b) {
    rt::drain_rows_to_staging<H, NT>(taddr + b * (uint32_t)H, stage, warp, lane);
    tc::fence_before_sync();
    __syncthreads();
#pragma unroll
    for (int i = 0; i < MH::NQ; ++i) {
      const int r = rh + i * MH::RS;
      if (r0 + r < p.rows) {
        float4 v = stage[rt::stage_index(r, qh, QH)];
        v.x = fmaxf(v.x + bias4[0], 0.0f);
        v.y = fmaxf(v.y + bias4[1], 0.0f);
        v.z = fmaxf(v.z + bias4[2], 0.0f);
        v.w = fmaxf(v.w + bias4[3], 0.0f);
        *reinterpret_cast<float4*>(p.z + (r0 + r) * H + 4 * qh) = v;
        if (want_stats) wf.push(v);   // BatchNorm batch statistics: training only
      }
    }
  };

  long long t = blockIdx.x;
  load_tile(t);
  uint32_t phase = 0, buf = 0;
  bool have_prev = false;
  long long prev_r0 = 0;
  for (; t < ntiles; t += gridDim.x) {
    const long long r0 = t * TR;
    // (1) previous layer's BatchNorm / dropout on the u half, hi/lo split, swizzled operand stores
#pragma unroll
    for (int i = 0; i < MC::NQ; ++i) {
      const long long row = r0 + rc + i * MC::RS;
      const bool live = row < p.rows;
      float4 h, l;
      if constexpr (WIDE) {
        const float4 u = live ? rt::act_fwd4(p.act, cq, pu[i], rk, (uint32_t)row) : make_float4(0.f, 0.f, 0.f, 0.f);
        tc::split4(u, h, l);
        rt::sts4(a_hi + koff_u + i * MC::RS * rt::kRowBytes, h);
        rt::sts4(a_lo + koff_u + i * MC::RS * rt::kRowBytes, l);
        tc::split4(pa[i], h, l);
        rt::sts4(a_hi + koff_a + i * MC::RS * rt::kRowBytes, h);
        rt::sts4(a_lo + koff_a + i * MC::RS * rt::kRowBytes, l);
      } else if (4 * qc < K) {
        float e[4] = {pu[i].x, pu[i].y, pu[i].z, pu[i].w};
        const uint32_t rhash = (live && p.act.drop) ? drop_row_hash(p.act, p.act.row_base + row) : 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int kk = 4 * qc + j;
          if (live && kk < C) e[j] = act_fwd(p.act, affine, e[j], s_scale[kk], s_shift[kk], rhash, kk);
        }
        tc::split4(make_float4(e[0], e[1], e[2], e[3]), h, l);
        rt::sts4(a_hi + koff_u + i * MC::RS * rt::kRowBytes, h);
        rt::sts4(a_lo + koff_u + i * MC::RS * rt::kRowBytes, l);
      }
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tid == 0) {
      rt::issue_kmajor_x3<KP / 8, TR, H>(taddr + buf * (uint32_t)H, od, ksteps, idesc, false);
      tc::mma_commit(&mbar);
    }
    load_tile(t + gridDim.x);          // next tile's loads fly during the MMA and the epilogue
    if (have_prev) epilogue(prev_r0, buf ^ 1u);   // the previous tile's accumulators leave while this tile multiplies
    tc::mbar_wait(&mbar, phase);       // the operand tile may be rewritten once this tile's MMAs have read it
    phase ^= 1;
    have_prev = true;
    prev_r0 = r0;
    buf ^= 1u;
  }
  if (have_prev) {
    tc::fence_after_sync();
    epilogue(prev_r0, buf ^ 1u);
  }
  __syncthreads();

  if (p.partials) {
    float* rec = reinterpret_cast<float*>(base);   // [NT][9] over the operand tile (every MMA has completed)
    wf.deposit(rec + tid * 9);
    __syncthreads();
    cta_write_quad_stats(rec, NT, QH, H, tid, p.partials + (size_t)blockIdx.x * (1 + 2 * H));
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, p.tmem_cols);
}


// Launch shape of one contraction: KB blocks of 32 contraction channels, WIDE operand rows (16-byte aligned, a multiple of
// 32 channels), dynamic shared memory and grid.
struct GemmShape {
  int KB; bool wide; size_t smem; long long grid;
  int o_stage;   // k_sage_fwd_gemm: the epilogue staging area
};

bool sage_fwd_gemm_supported(const float* t_in, const float* agg, const float* z, int64_t rows, int32_t C, int32_t H,
                             bool want_stats, size_t workspace_bytes, GemmShape* s) {
  GemmShape unused;
  if (!s) s = &unused;
  if (H != 32 && H != 64 && H != 128) return false;
  if (C <= 0 || 2 * C > 128) return false;
  s->wide = (C % 32 == 0) && ((((uintptr_t)t_in) | ((uintptr_t)agg)) & 15u) == 0;
  s->KB = (2 * C + 31) / 32;
  if (s->KB == 3 || (!s->wide && s->KB > 2)) return false;
  if ((((uintptr_t)z) & 15u) != 0) return false;
  const DeviceInfo dev = device_info();
  const int KP = 32 * s->KB;
  const size_t a_bytes = (size_t)2 * s->KB * kRows * 128, b_bytes = (size_t)2 * s->KB * H * 128;
  const size_t c_bytes = (size_t)2 * KP * 4;
  size_t stage_bytes = (size_t)kRows * H * 4;
  size_t total = a_bytes + b_bytes + c_bytes;
  s->o_stage = (int)((total + 15) & ~(size_t)15);     // never aliases the operand: the epilogue of tile t-1 runs
  total = s->o_stage + stage_bytes;                     // while the MMAs of tile t read it
  s->smem = total + 1024;
  if (s->smem > (size_t)dev.smem_optin) return false;
  const long long ntiles = (rows + kRows - 1) / kRows;
  s->grid = dev.sm_count;
  if (s->grid > ntiles) s->grid = ntiles;
  if (want_stats) {
    const size_t rec = (size_t)(1 + 2 * H) * sizeof(double);
    if ((size_t)s->grid * rec > workspace_bytes) s->grid = (long long)(workspace_bytes / rec);
  }
  return s->grid >= 1;
}

int launch_sage_fwd_gemm(const float* t_in, const cgnn_act_t* act, const float* agg, const float* W, const float* bias,
                         int64_t rows, int32_t C, int32_t H, float* z, double* partials, int* grid_out,
                         size_t workspace_bytes, cudaStream_t stream) {
  GemmShape s;
  if (!sage_fwd_gemm_supported(t_in, agg, z, rows, C, H, partials != nullptr, workspace_bytes, &s)) return CGNN_ERR_INVALID_ARG;
  const int KB = s.KB, HB = H / 32;
  const bool wide = s.wide; const size_t smem = s.smem; const long long grid = s.grid;
  SageFwdGemmArgs a;
  a.t_in = t_in; a.act = make_act(act); a.agg = agg; a.W = W; a.bias = bias;
  a.rows = rows; a.C = C; a.H = H;
  a.z = z; a.partials = partials;
  a.tmem_cols = 32;
  while (a.tmem_cols < (uint32_t)(2 * H)) a.tmem_cols <<= 1;   // two accumulator buffers
  a.o_stage = s.o_stage;
  *grid_out = (int)grid;
#define CGNN_SF(KB_, HB_, W_, NT_)                                                                    \
  {                                                                                                   \
    auto kfn = k_sage_fwd_gemm<KB_, HB_, W_, NT_>;                                                    \
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                \
    CGNN_LAUNCH(kfn, (unsigned)grid, NT_, smem, stream, a);                                           \
  }
#define CGNN_SF_H(KB_, W_) { if (HB == 1) CGNN_SF(KB_, 1, W_, 512) else if (HB == 2) CGNN_SF(KB_, 2, W_, 512) else CGNN_SF(KB_, 4, W_, 512) }
  // (1024-thread CTAs were measured: no faster than 512 - the kernel is not occupancy-bound)
  if (wide) { if (KB == 2) CGNN_SF_H(2, true) else CGNN_SF_H(4, true) }
  else { if (KB == 1) CGNN_SF_H(1, false) else CGNN_SF_H(2, false) }
#undef CGNN_SF_H
#undef CGNN_SF
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

// ================================================================================================================
// GCN backward contractions
// ================================================================================================================
struct GcnBwdGemmArgs {
  const float* dP; const float* t_in; Act act_in; const float* W;
  long long rows; int H, Kin;
  float* du_in; const float* prev_mean; const float* prev_rstd; int want_prev;
  float* partials; int part_stride, o_pprev;   // per CTA: [dW H x Kin][prev 2 x Kin]
  uint32_t tmem_cols;
};

// HB = H / 32, KB = padded Kin / 32.  WIDE: Kin is a multiple of 32 and t_in / du_in are 16-byte aligned.
template <int HB, int KB, bool WIDE>
__global__ void __launch_bounds__(kThreads, 1) k_gcn_bwd_gemm(GcnBwdGemmArgs p) {
  act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  constexpr int H = 32 * HB, KP = 32 * KB, TR = kRows;
  constexpr int Q1 = H / 4, Q2 = KP / 4;
  using M1 = rt::QuadMap<Q1, TR>;     // dP quads
  using M2 = rt::QuadMap<Q2, TR>;     // layer-input / du_in quads
  constexpr int A1_HALF = HB * TR * 128, A2_HALF = KB * TR * 128, B1_HALF = HB * KP * 128;
  // M of the dW product: always 128 (an M = 64 instruction costs the same tensor-pipe time); for H < 128 the upper
  // MN groups of the A view run into the neighbouring operand tiles and fill accumulator rows that are never read.
  constexpr int MM = 128;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar, mbar_dw;   // du_in MMAs / dW MMAs of a tile complete
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  unsigned char* a1k_hi = base;                 // dP [128 rows][H], K-major (for du_in = dP W)
  unsigned char* a1k_lo = a1k_hi + A1_HALF;
  unsigned char* a1_hi = a1k_lo + A1_HALF;      // dP again, MN-major (for dW = dP^T u)
  unsigned char* a1_lo = a1_hi + A1_HALF;
  unsigned char* a2_hi = a1_lo + A1_HALF;       // u  [128 rows][KP], MN-major
  unsigned char* a2_lo = a2_hi + A2_HALF;
  unsigned char* b1_hi = a2_lo + A2_HALF;       // W^T [KP rows (input channel)][H]
  unsigned char* b1_lo = b1_hi + B1_HALF;
  float* s_ci = reinterpret_cast<float*>(b1_lo + B1_HALF);    // [2][KP] scale, shift of act_in (element-wise path)
  float4* stage = reinterpret_cast<float4*>(base);             // [128][KP] swizzled / end-of-kernel scratch; aliases a1k
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Kin = p.Kin;
  const bool aff_in = p.act_in.scale != nullptr;

  if (warp == 0) tc::tmem_alloc(&tmem_base_s, p.tmem_cols);
  if (tid == 0) { tc::mbar_init(&mbar, 1); tc::mbar_init(&mbar_dw, 1); tc::fence_mbar_init(); }
  stage_weight_transposed(p.W, Kin, Kin, H, KP, H, b1_hi, b1_lo);   // operand row n = input channel, k = h: W[h][n]
  stage_affine(p.act_in, Kin, KP, s_ci, s_ci + KP);
  if (!WIDE) {   // padded channels of the u operand stay zero
    for (int i = tid; i < 2 * A2_HALF / 16; i += kThreads) reinterpret_cast<float4*>(a2_hi)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int q1 = tid % Q1, r1 = tid / Q1;
  const int q2 = tid % Q2, r2 = tid / Q2;
  const int c2 = 4 * q2;
  const uint32_t koff1 = rt::kmajor_quad_offset(r1, q1, TR), moff1 = rt::mnmajor_quad_offset(r1, q1, TR);
  const uint32_t moff2 = rt::mnmajor_quad_offset(r2, q2, TR);
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act_in, c2, Kin);
  const rt::RowKey rk = rt::row_key(p.act_in);
  float pmean[4], prstd[4];
  rt::bn_stats_quad(pmean, prstd, p.prev_mean, p.prev_rstd, c2, Kin, p.want_prev);
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  const uint32_t a1h = tc::smem_u32(a1_hi), a1l = tc::smem_u32(a1_lo), a2h = tc::smem_u32(a2_hi), a2l = tc::smem_u32(a2_lo);
  const uint32_t a1kh = tc::smem_u32(a1k_hi), a1kl = tc::smem_u32(a1k_lo);
  const uint32_t b1h = tc::smem_u32(b1_hi), b1l = tc::smem_u32(b1_lo);
  const uint32_t id1 = tc::idesc_tf32(TR, KP), id2 = tc::idesc_tf32(MM, KP, 1, 1);
  const rt::OperandDescs od1 = rt::kmajor_descs(a1kh, a1kl, b1h, b1l), od2 = rt::mnmajor_descs(a1h, a1l, a2h, a2l, TR);

  const long long ntiles = (p.rows + TR - 1) / TR;
  float4 dpn[M1::NQ], tin[M2::NQ], tcur[M2::NQ];
  auto load_tile = [&](long long t) {
    const long long r0 = t * TR;
#pragma unroll
    for (int i = 0; i < M1::NQ; ++i) {
      const long long row = r0 + r1 + i * M1::RS;
      dpn[i] = (t < ntiles && row < p.rows) ? rt::ld_quad<true>(p.dP, row, H, 4 * q1) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < M2::NQ; ++i) {
      const long long row = r0 + r2 + i * M2::RS;
      tin[i] = (t < ntiles && row < p.rows && c2 < Kin) ? rt::ld_quad<WIDE>(p.t_in, row, Kin, c2) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };

  float ps1[4] = {0.f, 0.f, 0.f, 0.f}, ps2[4] = {0.f, 0.f, 0.f, 0.f};
  long long t = blockIdx.x;
  load_tile(t);
  uint32_t phase = 0;
  bool first = true;
  for (; t < ntiles; t += gridDim.x) {
    const long long r0 = t * TR;
    // (1) operands: dP as is (both layouts), u = BatchNorm / ReLU / dropout of the stored layer input
#pragma unroll
    for (int i = 0; i < M1::NQ; ++i) {
      float4 h, l;
      tc::split4(dpn[i], h, l);
      if (p.du_in) {
        rt::sts4(a1k_hi + koff1 + i * M1::RS * rt::kRowBytes, h);
        rt::sts4(a1k_lo + koff1 + i * M1::RS * rt::kRowBytes, l);
      }
      rt::sts4(a1_hi + moff1 + i * M1::RS * rt::kRowBytes, h);
      rt::sts4(a1_lo + moff1 + i * M1::RS * rt::kRowBytes, l);
    }
    if (WIDE || c2 < Kin) {
#pragma unroll
      for (int i = 0; i < M2::NQ; ++i) {
        const long long row = r0 + r2 + i * M2::RS;
        tcur[i] = tin[i];
        float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < p.rows) u = rt::mask_quad(rt::act_fwd4(p.act_in, cq, tin[i], rk, (uint32_t)row), c2, Kin);
        float4 h, l;
        tc::split4(u, h, l);
        rt::sts4(a2_hi + moff2 + i * M2::RS * rt::kRowBytes, h);
        rt::sts4(a2_lo + moff2 + i * M2::RS * rt::kRowBytes, l);
      }
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tid == 0) {
      // two commits: the du_in product (a third of the tensor work) is waited for first, its epilogue - staged over the
      // K-major dP operand only that product reads - then runs while the dW product is still multiplying
      if (p.du_in) {
        rt::issue_kmajor_x3<H / 8, TR, KP>(taddr, od1, H / 8, id1, false);   // du_in tile = dP W
        tc::mma_commit(&mbar);
      }
      // dW += dP^T u : M = H (MN-major view of the dP tile), N = KP (MN-major view of the u tile), K = 128 rows
      rt::issue_mnmajor_x3<TR>(taddr + (uint32_t)KP, od2, id2, !first);
      tc::mma_commit(&mbar_dw);
    }
    first = false;
    load_tile(t + gridDim.x);
    if (p.du_in) {
      tc::mbar_wait(&mbar, phase);
      tc::fence_after_sync();
      rt::drain_rows_to_staging<KP>(taddr, stage, warp, lane);
      tc::fence_before_sync();
      __syncthreads();
      // (2) coalesced du_in store + BatchNorm-backward sums of the layer below (fixed channel quad per thread)
      if (WIDE || c2 < Kin) {
#pragma unroll
        for (int i = 0; i < M2::NQ; ++i) {
          const int r = r2 + i * M2::RS;
          const long long row = r0 + r;
          if (row < p.rows) {
            const float4 d = stage[rt::stage_index(r, q2, Q2)];
            rt::st_quad<WIDE>(p.du_in, row, Kin, c2, d);
            if (p.want_prev) {
              const float4 dyp = rt::act_bwd4(p.act_in, cq, tcur[i], d, rk, (uint32_t)row);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (WIDE || c2 + j < Kin) {
                  const float xh = (f4_get(tcur[i], j) - pmean[j]) * prstd[j];
                  ps1[j] += f4_get(dyp, j);
                  ps2[j] = fmaf(f4_get(dyp, j), xh, ps2[j]);
                }
              }
            }
          }
        }
      }
    }
    tc::mbar_wait(&mbar_dw, phase);   // the MN-major operands may be rewritten once the dW product has read them
    phase ^= 1;
    tc::fence_after_sync();
    __syncthreads();   // operand tiles / staging are rewritten by the next tile
  }
  (void)aff_in;

  // ---- per-CTA partial record ---------------------------------------------------------------------------------
  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
  {
    constexpr int CW = KP / 4;
    const int q = warp & 3, cg = warp >> 2;
    float v[CW];
    tc::tmem_ld<CW>(taddr + ((uint32_t)(32 * q) << 16) + (uint32_t)(KP + cg * CW), v);
    tc::tmem_ld_wait();
    const int h = 32 * q + lane;
    if (h < H) {
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        const int c = cg * CW + j;
        if (c < Kin) part[(size_t)h * Kin + c] = v[j];
      }
    }
  }
  if (p.want_prev) {
    float* red = reinterpret_cast<float*>(stage);   // [kThreads][8]
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[tid * 8 + j] = ps1[j]; red[tid * 8 + 4 + j] = ps2[j]; }
    __syncthreads();
    for (int c = tid; c < 2 * Kin; c += kThreads) {
      const int which = c / Kin, ch = c - which * Kin;
      part[p.o_pprev + c] = quad_sum(red, 8, which * 4, kThreads, Q2, ch >> 2, ch & 3);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, p.tmem_cols);
}

bool gcn_bwd_gemm_supported(const float* dP, const float* t_in, const float* du_in, int64_t rows, int32_t d_in, int32_t H,
                            int part_stride, size_t partial_bytes, GemmShape* s) {
  GemmShape unused;
  if (!s) s = &unused;
  if (H != 32 && H != 64 && H != 128) return false;
  if (d_in <= 0 || d_in > 128) return false;
  const int HB = H / 32, KB = (d_in + 31) / 32;
  if (KB == 3) return false;
  if ((((uintptr_t)dP) & 15u) != 0) return false;
  s->KB = KB;
  s->wide = (d_in % 32 == 0) && ((((uintptr_t)t_in) & 15u) == 0) && (!du_in || (((uintptr_t)du_in) & 15u) == 0);
  if (!s->wide && KB > 2) return false;
  if (du_in && 32 * KB > 2 * H) return false;   // the du_in staging must stay inside the K-major dP operand (see the two commits)
  const DeviceInfo dev = device_info();
  const int KP = 32 * KB;
  size_t total = (size_t)4 * HB * kRows * 128 + (size_t)2 * KB * kRows * 128 + (size_t)2 * HB * KP * 128 + (size_t)2 * KP * 4;
  const size_t a_view = (size_t)3 * HB * kRows * 128 + (size_t)4 * kRows * 128;   // the M = 128 view of the MN-major dP lo tile ends here
  if (total < a_view) total = a_view;
  if (total < (size_t)kRows * KP * 4) total = (size_t)kRows * KP * 4;
  s->smem = total + 1024;
  if (s->smem > (size_t)dev.smem_optin) return false;
  const long long ntiles = (rows + kRows - 1) / kRows;
  s->grid = dev.sm_count;
  if (s->grid > ntiles) s->grid = ntiles;
  const size_t rec = (size_t)part_stride * sizeof(float);
  if ((size_t)s->grid * rec > partial_bytes) s->grid = (long long)(partial_bytes / rec);
  return s->grid >= 1;
}

// Launches k_gcn_bwd_gemm (grid in *grid_out; the caller reduces the partial records).
int launch_gcn_bwd_gemm(const float* dP, const float* t_in, const cgnn_act_t* act_in, const float* W, int64_t rows,
                        int32_t d_in, int32_t H, float* du_in, const float* prev_mean, const float* prev_rstd, int want_prev,
                        float* partials, int part_stride, int o_pprev, int* grid_out, size_t partial_bytes,
                        cudaStream_t stream) {
  GemmShape s;
  if (!gcn_bwd_gemm_supported(dP, t_in, du_in, rows, d_in, H, part_stride, partial_bytes, &s)) return CGNN_ERR_INVALID_ARG;
  const int KB = s.KB, HB = H / 32;
  const bool wide = s.wide; const size_t smem = s.smem; const long long grid = s.grid;
  GcnBwdGemmArgs a;
  a.dP = dP; a.t_in = t_in; a.act_in = make_act(act_in); a.W = W;
  a.rows = rows; a.H = H; a.Kin = d_in;
  a.du_in = du_in; a.prev_mean = prev_mean; a.prev_rstd = prev_rstd; a.want_prev = want_prev;
  a.partials = partials; a.part_stride = part_stride; a.o_pprev = o_pprev;
  a.tmem_cols = 32;
  while (a.tmem_cols < (uint32_t)(2 * 32 * KB)) a.tmem_cols <<= 1;
  *grid_out = (int)grid;
#define CGNN_GB(HB_, KB_, W_)                                                                         \
  {                                                                                                   \
    auto kfn = k_gcn_bwd_gemm<HB_, KB_, W_>;                                                          \
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                \
    CGNN_LAUNCH(kfn, (unsigned)grid, kThreads, smem, stream, a);                                      \
  }
#define CGNN_GB_K(HB_)                                                                                \
  {                                                                                                   \
    if (wide) { if (KB == 1) CGNN_GB(HB_, 1, true) else if (KB == 2) CGNN_GB(HB_, 2, true) else CGNN_GB(HB_, 4, true) } \
    else { if (KB == 1) CGNN_GB(HB_, 1, false) else CGNN_GB(HB_, 2, false) }                          \
  }
  if (HB == 1) CGNN_GB_K(1) else if (HB == 2) CGNN_GB_K(2) else CGNN_GB_K(4)
#undef CGNN_GB_K
#undef CGNN_GB
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

// ================================================================================================================
// GraphSAGE backward contractions (64-row tiles)
// ================================================================================================================
struct SageBwdGemmArgs {
  const float* du; const float* demb; const int32_t* row_graph; const int32_t* meta;   // upstream: per row, or pooled per subject
  const float* z; Act act_out; BnBwdDev bn;
  const float* t_in; const float* agg; Act act_in; const float* W;
  long long rows; int H, C;
  float* direct; float* nbr;          // d_u, d_agg [rows, C] (NULL: the layer input needs no gradient)
  float* partials; int part_stride, o_pdb;   // per CTA: [dW H x 2C][dbias H]
  uint32_t tmem_cols;
};

// HB = H / 32; CB = padded 2C / 32 (2C = 32 CB when WIDE).  Output channels j of [d_u || d_agg] and of dW^T sit on the
// TMEM lanes (M = 128, rows of W^T beyond 2C are zero), tile rows / h on the columns: the d_u / d_agg rows leave
// tensor memory as 128-byte coalesced stores without a staging pass.
template <int HB, int CB, bool WIDE>
__global__ void __launch_bounds__(kThreads, 1) k_sage_bwd_gemm(SageBwdGemmArgs p) {
  act_salt(p.act_out); act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  constexpr int H = 32 * HB, TR = 64, MP = 128;
  constexpr int QH = H / 4;
  using MHq = rt::QuadMap<QH, TR>;                      // z / du / dz quads
  constexpr int QC = WIDE ? (32 * CB) / 8 : (32 * CB) / 4;   // quads per row of t_in and of agg (wide) / of the padded 2C
  using MCq = rt::QuadMap<QC, TR>;
  constexpr int DZ_HALF = HB * TR * 128;                // dz tile, either layout
  constexpr int UA_HALF = 4 * TR * 128;                 // [u || agg] MN-major, always 4 channel groups (zero padded)
  constexpr int WK_HALF = HB * MP * 128;                // W^T rows j (padded to 128), K-major over h
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  unsigned char* dzk_hi = base;
  unsigned char* dzk_lo = dzk_hi + DZ_HALF;
  unsigned char* dzm_hi = dzk_lo + DZ_HALF;
  unsigned char* dzm_lo = dzm_hi + DZ_HALF;
  unsigned char* ua_hi = dzm_lo + DZ_HALF;
  unsigned char* ua_lo = ua_hi + UA_HALF;
  unsigned char* wk_hi = ua_lo + UA_HALF;
  unsigned char* wk_lo = wk_hi + WK_HALF;
  float* s_ci = reinterpret_cast<float*>(wk_lo + WK_HALF);   // [2][32 CB] scale, shift of act_in (element-wise path)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = p.C, K2 = 2 * C;
  const bool aff_in = p.act_in.scale != nullptr;
  const bool need_du = p.direct != nullptr;

  if (warp == 0) tc::tmem_alloc(&tmem_base_s, p.tmem_cols);
  if (tid == 0) { tc::mbar_init(&mbar, 1); tc::fence_mbar_init(); }
  // operand row j = column j of W [H][2C], contraction index = h
  stage_weight_transposed(p.W, K2, K2, H, MP, H, wk_hi, wk_lo);
  stage_affine(p.act_in, C, 32 * CB, s_ci, s_ci + 32 * CB);
  for (int i = tid; i < 2 * UA_HALF / 16; i += kThreads) reinterpret_cast<float4*>(ua_hi)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int qh = tid % QH, rh = tid / QH;
  const int qc = tid % QC, rc = tid / QC;
  rt::ChanQuad cq_out, cq_in;
  rt::chan_quad_init(cq_out, p.act_out, 4 * qh, H);
  rt::chan_quad_init(cq_in, p.act_in, 4 * qc, C);
  const rt::RowKey rk_out = rt::row_key(p.act_out), rk_in = rt::row_key(p.act_in);
  rt::BnQuad bq;
  rt::bn_quad_init(bq, p.bn, 4 * qh, H);
  const uint32_t koff_z = rt::kmajor_quad_offset(rh, qh, TR), moff_z = rt::mnmajor_quad_offset(rh, qh, TR);
  const uint32_t moff_u = rt::mnmajor_quad_offset(rc, qc, TR);
  const uint32_t moff_a = WIDE ? rt::mnmajor_quad_offset(rc, qc + QC, TR) : 0u;
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  const uint32_t dzkh = tc::smem_u32(dzk_hi), dzkl = tc::smem_u32(dzk_lo), dzmh = tc::smem_u32(dzm_hi), dzml = tc::smem_u32(dzm_lo);
  const uint32_t uah = tc::smem_u32(ua_hi), ual = tc::smem_u32(ua_lo), wkh = tc::smem_u32(wk_hi), wkl = tc::smem_u32(wk_lo);
  const uint32_t id1 = tc::idesc_tf32(MP, TR), id2 = tc::idesc_tf32(MP, H, 1, 1);
  const uint32_t t_du = taddr, t_dw = taddr + (uint32_t)(2 * TR);   // two [d_u || d_agg] buffers, one dW accumulator
  const rt::OperandDescs od1 = rt::kmajor_descs(wkh, wkl, dzkh, dzkl), od2 = rt::mnmajor_descs(uah, ual, dzmh, dzml, TR);

  const long long ntiles = (p.rows + TR - 1) / TR;
  float4 zq[MHq::NQ], uq[MHq::NQ], tq[MCq::NQ], aq[WIDE ? MCq::NQ : 1];
  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  // pooled upstream (top layer): the subject of a row is needed before its pooled gradient can be addressed - that
  // index is loaded one tile further ahead than the data, so no load in load_tile waits for another
  int rg[MHq::NQ];
  auto load_rg = [&](long long t) {
#pragma unroll
    for (int i = 0; i < MHq::NQ; ++i) {
      const long long row = t * TR + rh + i * MHq::RS;
      rg[i] = (!p.du && t < ntiles && row < p.rows) ? p.row_graph[row] : 0;
    }
  };
  auto load_tile = [&](long long t) {
    const long long r0 = t * TR;
#pragma unroll
    for (int i = 0; i < MHq::NQ; ++i) {
      const long long row = r0 + rh + i * MHq::RS;
      float4 zv = make_float4(0.f, 0.f, 0.f, 0.f), uv = zv;
      if (t < ntiles && row < p.rows) {
        zv = rt::ld_quad<true>(p.z, row, H, 4 * qh);
        if (p.du) uv = rt::ld_quad<true>(p.du, row, H, 4 * qh);
        else uv = rt::pooled_quad<true>(p.demb, rg[i], H, 4 * qh, meta[rg[i]].y);
      }
      zq[i] = zv; uq[i] = uv;
    }
#pragma unroll
    for (int i = 0; i < MCq::NQ; ++i) {
      const long long row = r0 + rc + i * MCq::RS;
      float4 tv = make_float4(0.f, 0.f, 0.f, 0.f), av = tv;
      if (t < ntiles && row < p.rows) {
        if constexpr (WIDE) {
          tv = rt::ld_quad<true>(p.t_in, row, C, 4 * qc);
          av = rt::ld_quad<true>(p.agg, row, C, 4 * qc);
        } else if (4 * qc < K2) {
          float e[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int kk = 4 * qc + j;
            e[j] = kk < C ? p.t_in[row * C + kk] : (kk < K2 ? p.agg[row * C + (kk - C)] : 0.0f);
          }
          tv = make_float4(e[0], e[1], e[2], e[3]);
        }
      }
      tq[i] = tv;
      if constexpr (WIDE) aq[i] = av;
    }
    load_rg(t + gridDim.x);
  };

  // [d_u || d_agg] rows of the tile at r0 (accumulator buffer b): lane = output channel j, 16 tile rows per warp -
  // every store instruction writes 32 consecutive channels of one row
  auto store_du = [&](long long r0, uint32_t b) {
    const int lq = warp & 3, cg = warp >> 2;
    float v[16];
    tc::tmem_ld<16>(t_du + b * (uint32_t)TR + ((uint32_t)(32 * lq) << 16) + (uint32_t)(16 * cg), v);
    tc::tmem_ld_wait();
    const int j = 32 * lq + lane;
    if (j < K2) {
      float* dst = (j < C ? p.direct + j : p.nbr + (j - C)) + (r0 + 16 * cg) * C;
#pragma unroll
      for (int rr = 0; rr < 16; ++rr)
        if (r0 + 16 * cg + rr < p.rows) dst[(long long)rr * C] = v[rr];
    }
  };

  float colsum[4] = {0.f, 0.f, 0.f, 0.f};
  long long t = blockIdx.x;
  load_rg(t);
  load_tile(t);
  uint32_t phase = 0, buf = 0;
  bool first = true, have_prev = false;
  long long prev_r0 = 0;
  for (; t < ntiles; t += gridDim.x) {
    const long long r0 = t * TR;
    // (1) dz = relu'(z) * BatchNorm backward of the dropout backward of the upstream gradient; both operand layouts
#pragma unroll
    for (int i = 0; i < MHq::NQ; ++i) {
      const long long row = r0 + rh + i * MHq::RS;
      float4 dz = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < p.rows) {
        dz = rt::dz4<true>(p.act_out, cq_out, p.bn, bq, zq[i], uq[i], rk_out, (uint32_t)row);
        colsum[0] += dz.x; colsum[1] += dz.y; colsum[2] += dz.z; colsum[3] += dz.w;
      }
      float4 h, l;
      tc::split4(dz, h, l);
      if (need_du) {
        rt::sts4(dzk_hi + koff_z + i * MHq::RS * rt::kRowBytes, h);
        rt::sts4(dzk_lo + koff_z + i * MHq::RS * rt::kRowBytes, l);
      }
      rt::sts4(dzm_hi + moff_z + i * MHq::RS * rt::kRowBytes, h);
      rt::sts4(dzm_lo + moff_z + i * MHq::RS * rt::kRowBytes, l);
    }
    //     [u || agg] with the previous layer's BatchNorm / dropout on the u half
#pragma unroll
    for (int i = 0; i < MCq::NQ; ++i) {
      const long long row = r0 + rc + i * MCq::RS;
      const bool live = row < p.rows;
      float4 h, l;
      if constexpr (WIDE) {
        const float4 u = live ? rt::act_fwd4(p.act_in, cq_in, tq[i], rk_in, (uint32_t)row) : make_float4(0.f, 0.f, 0.f, 0.f);
        tc::split4(u, h, l);
        rt::sts4(ua_hi + moff_u + i * MCq::RS * rt::kRowBytes, h);
        rt::sts4(ua_lo + moff_u + i * MCq::RS * rt::kRowBytes, l);
        tc::split4(aq[i], h, l);
        rt::sts4(ua_hi + moff_a + i * MCq::RS * rt::kRowBytes, h);
        rt::sts4(ua_lo + moff_a + i * MCq::RS * rt::kRowBytes, l);
      } else if (4 * qc < K2) {
        float e[4] = {tq[i].x, tq[i].y, tq[i].z, tq[i].w};
        const uint32_t rhash = (live && p.act_in.drop) ? drop_row_hash(p.act_in, p.act_in.row_base + row) : 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int kk = 4 * qc + j;
          if (live && kk < C) e[j] = act_fwd(p.act_in, aff_in, e[j], s_ci[kk], s_ci[32 * CB + kk], rhash, kk);
        }
        tc::split4(make_float4(e[0], e[1], e[2], e[3]), h, l);
        rt::sts4(ua_hi + moff_u + i * MCq::RS * rt::kRowBytes, h);
        rt::sts4(ua_lo + moff_u + i * MCq::RS * rt::kRowBytes, l);
      }
    }
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tid == 0) {
      // [d_u || d_agg]^T tile = W^T dz^T : M = 128 (j), N = 64 tile rows, K = H
      if (need_du) rt::issue_kmajor_x3<H / 8, MP, TR>(t_du + buf * (uint32_t)TR, od1, H / 8, id1, false);
      // dW^T += [u || agg]^T dz : M = 128 (j), N = H, K = 64 tile rows
      rt::issue_mnmajor_x3<TR>(t_dw, od2, id2, !first);
      tc::mma_commit(&mbar);
    }
    first = false;
    load_tile(t + gridDim.x);
    if (need_du && have_prev) store_du(prev_r0, buf ^ 1u);   // the previous tile's rows leave while this tile multiplies
    tc::mbar_wait(&mbar, phase);                              // operand tiles may be rewritten after this
    phase ^= 1;
    have_prev = true;
    prev_r0 = r0;
    buf ^= 1u;
  }
  tc::fence_after_sync();
  if (need_du && have_prev) store_du(prev_r0, buf ^ 1u);
  tc::fence_before_sync();
  __syncthreads();

  // ---- per-CTA partial record: dW [H][2C] from the transposed accumulator, dbias from the column sums --------------
  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
  {
    constexpr int CW = H / 4;
    const int lq = warp & 3, cg = warp >> 2;
    float v[CW];
    tc::tmem_ld<CW>(t_dw + ((uint32_t)(32 * lq) << 16) + (uint32_t)(cg * CW), v);
    tc::tmem_ld_wait();
    const int j = 32 * lq + lane;
    if (j < K2) {
#pragma unroll
      for (int hh = 0; hh < CW; ++hh) part[(size_t)(cg * CW + hh) * K2 + j] = first ? 0.0f : v[hh];
    }
  }
  {
    float* red = reinterpret_cast<float*>(base);   // [kThreads][4]; the operand tiles are dead
    __syncthreads();
    *reinterpret_cast<float4*>(red + 4 * tid) = make_float4(colsum[0], colsum[1], colsum[2], colsum[3]);
    __syncthreads();
    for (int c = tid; c < H; c += kThreads) part[p.o_pdb + c] = quad_sum(red, 4, 0, kThreads, QH, c >> 2, c & 3);
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, p.tmem_cols);
}

// Returns CGNN_OK when launched (grid in *grid_out; the caller reduces the partial records [dW H x 2C][dbias H]),
// -1 when the shape is not covered.
int launch_sage_bwd_gemm(const float* du, const float* demb, const int32_t* row_graph, const int32_t* meta, const float* z,
                         const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn, const float* t_in, const float* agg,
                         const cgnn_act_t* act_in, const float* W, int64_t rows, int32_t C, int32_t H, float* direct,
                         float* nbr, float* partials, int part_stride, int o_pdb, int* grid_out, size_t partial_bytes,
                         cudaStream_t stream) {
  if (H != 32 && H != 64 && H != 128) return -1;
  if (C <= 0 || 2 * C > 128) return -1;
  const int HB = H / 32, CB = (2 * C + 31) / 32;
  if (CB == 3) return -1;
  const bool wide = (C % 32 == 0) && ((((uintptr_t)t_in) | ((uintptr_t)agg)) & 15u) == 0;
  if (!wide && CB > 2) return -1;
  if (((((uintptr_t)z) | ((uintptr_t)du) | ((uintptr_t)demb)) & 15u) != 0) return -1;
  if (!du && (!row_graph || !meta)) return -1;
  const DeviceInfo dev = device_info();
  SageBwdGemmArgs a;
  a.du = du; a.demb = demb; a.row_graph = row_graph; a.meta = meta;
  a.z = z; a.act_out = make_act(act_out); a.bn = make_bn_bwd(bn);
  a.t_in = t_in; a.agg = agg; a.act_in = make_act(act_in); a.W = W;
  a.rows = rows; a.H = H; a.C = C;
  a.direct = direct; a.nbr = nbr;
  a.partials = partials; a.part_stride = part_stride; a.o_pdb = o_pdb;
  a.tmem_cols = 32;
  while (a.tmem_cols < (uint32_t)(2 * 64 + H)) a.tmem_cols <<= 1;
  const size_t total = (size_t)4 * HB * 64 * 128 + (size_t)2 * 4 * 64 * 128 + (size_t)2 * HB * 128 * 128 + (size_t)2 * 32 * CB * 4;
  const size_t smem = total + 1024;
  if (smem > (size_t)dev.smem_optin) return -1;
  const long long ntiles = (rows + 63) / 64;
  long long grid = dev.sm_count;
  if (grid > ntiles) grid = ntiles;
  const size_t rec = (size_t)part_stride * sizeof(float);
  if ((size_t)grid * rec > partial_bytes) grid = (long long)(partial_bytes / rec);
  if (grid < 1) return -1;
  *grid_out = (int)grid;
#define CGNN_SB(HB_, CB_, W_)                                                                         \
  {                                                                                                   \
    auto kfn = k_sage_bwd_gemm<HB_, CB_, W_>;                                                         \
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                \
    CGNN_LAUNCH(kfn, (unsigned)grid, kThreads, smem, stream, a);                                      \
  }
#define CGNN_SB_C(HB_)                                                                                \
  {                                                                                                   \
    if (wide) { if (CB == 2) CGNN_SB(HB_, 2, true) else CGNN_SB(HB_, 4, true) }                       \
    else { if (CB == 1) CGNN_SB(HB_, 1, false) else CGNN_SB(HB_, 2, false) }                          \
  }
  if (HB == 1) CGNN_SB_C(1) else if (HB == 2) CGNN_SB_C(2) else CGNN_SB_C(4)
#undef CGNN_SB_C
#undef CGNN_SB
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

#endif  // CGNN_EMU
}  // namespace cgnn
