// wide_tc.cu - GCN layers of width 256 (BASELINE configs[4]: 360-node subjects, hidden 256) on tcgen05 (sm_100a only).
//
// At H = 256 neither a whole subject tile (360 x 256 fp32 = 360 KB) nor the hi/lo operands of a 256 x 256 weight
// (512 KB) fit the 227 KB of shared memory, so the layer is gather + K-looped contraction:
//
//   forward    k_gather<GCN_FWD>  a = A^ act(t_in)   (32-channel slabs, agg.cu; written into z)
//              k_wide_xw          z = a W^T + b, BatchNorm partial statistics            (reference models.py:111-114)
//                                 IN PLACE: a row tile's input rows are consumed before its output rows are written,
//                                 both have 256 channels, so the aggregate never needs a buffer of its own
//   backward   k_gather<GCN_BWD>  dz on load, dP = A^^T dz, dbias                        (agg.cu)
//              k_wide_xw          du_in = dP W                                           (autograd of models.py:111)
//              k_wide_xty         dW = dP^T act(t_in), accumulated in tensor memory over all of a CTA's rows; the
//                                 BatchNorm-backward sums of the layer below ride along (t_in is in registers there)
//
// k_wide_xw streams the weight, pre-split into TF32 hi/lo parts and laid out as swizzled K-major blocks by
// k_wide_prep_w (512 KB, L2 resident), one 32-channel block per pipeline stage; the accumulator of a 128-row tile is
// 256 TMEM columns, two of them alternate so the epilogue of tile t-1 is spread over the first K blocks of tile t.
#include "agg.cuh"
#include "rowtile.cuh"
#include "tile.cuh"

#include <type_traits>

namespace cgnn {
#ifndef CGNN_EMU
namespace {

constexpr int WN = 256;                                  // output channels of k_wide_xw / both widths of k_wide_xty
constexpr int WTR = 128;                                 // rows per tile
constexpr int W_A_HALF = WTR * 128;                      // one 32-channel block of 128 rows (hi or lo): 16 KB
constexpr int W_B_HALF = WN * 128;                       // one 32-channel block of the 256 weight rows: 32 KB
constexpr int W_STAGE = 2 * W_A_HALF + 2 * W_B_HALF;     // 96 KB
constexpr int W_SLAB = 64;                               // epilogue: columns per pass
constexpr int W_STAGING = WTR * W_SLAB * 4;              // 32 KB
constexpr int W_PASSES = WN / W_SLAB;
constexpr size_t W_XW_SMEM = (size_t)2 * W_STAGE + W_STAGING + 1024;

constexpr int XR = 16;                                   // k_wide_xty: contraction rows per pipeline stage
constexpr int X_HALF = (WN / 32) * XR * 128;             // 256 channels x 16 rows (hi or lo): 16 KB
constexpr int X_STAGE = 4 * X_HALF;                      // dP hi/lo + u hi/lo: 64 KB
constexpr int X_STAGES = 3;
constexpr size_t W_XTY_SMEM = (size_t)X_STAGES * X_STAGE + 1024;

// ---- weight image --------------------------------------------------------------------------------------------------
// B[n][k] (n < 256 operand rows, k < K contraction index) = W[n][k] or, transposed, W[k][n]; image = K/32 blocks of
// {hi [256 rows x 128 B], lo [256 rows x 128 B]}, each a K-major 128B-swizzled canonical tile.
__global__ void __launch_bounds__(256) k_wide_prep_w(const float* __restrict__ W, int ldw, int K, int transposed,
                                                     unsigned char* __restrict__ img) {
  const int Q = K >> 2;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < WN * Q; idx += gridDim.x * blockDim.x) {
    int n, q;
    if (transposed) { q = idx / WN; n = idx - q * WN; }   // consecutive threads read consecutive floats of a W row
    else { n = idx / Q; q = idx - n * Q; }
    float4 v;
    if (transposed) {
      v.x = W[(size_t)(4 * q + 0) * ldw + n];
      v.y = W[(size_t)(4 * q + 1) * ldw + n];
      v.z = W[(size_t)(4 * q + 2) * ldw + n];
      v.w = W[(size_t)(4 * q + 3) * ldw + n];
    } else {
      v = *reinterpret_cast<const float4*>(W + (size_t)n * ldw + 4 * q);
    }
    float4 h, l;
    tc::split4(v, h, l);
    const size_t off = (size_t)(q >> 3) * (2 * W_B_HALF) + rt::kmajor_quad_offset(n, q & 7, WN);
    *reinterpret_cast<float4*>(img + off) = h;
    *reinterpret_cast<float4*>(img + off + W_B_HALF) = l;
  }
}

// ---- out = A B^T (+ bias), 128-row tiles, K streamed in 32-channel blocks ----------------------------------------------
struct WideXwArgs {
  const float* A; long long rows; int K;
  const float* A2; int KB1, lda;     // K blocks >= KB1 come from A2 (GraphSAGE: [u || agg]); both have row stride lda
  int relu;                          // epilogue: max(. + bias, 0)
  const unsigned char* Bimg; const float* bias; float* out; double* partials;
};

__global__ void __launch_bounds__(kThreads, 1) k_wide_xw(WideXwArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar[2];
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  float4* staging = reinterpret_cast<float4*>(base + 2 * W_STAGE);   // [128][64] swizzled
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (warp == 0) tc::tmem_alloc(&tmem_base_s, 512);
  if (tid == 0) { tc::mbar_init(&mbar[0], 1); tc::mbar_init(&mbar[1], 1); tc::fence_mbar_init(); }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  const uint32_t idesc = tc::idesc_tf32(WTR, WN);
  // descriptors of stage 0; stage s adds s * W_STAGE to the 14-bit start-address field (>> 4)
  const uint32_t a0 = tc::smem_u32(base);
  const rt::OperandDescs od0 = rt::kmajor_descs(a0, a0 + W_A_HALF, a0 + 2 * W_A_HALF, a0 + 2 * W_A_HALF + W_B_HALF);
  const int KB = p.K >> 5;
  const long long ntiles = (p.rows + WTR - 1) / WTR;

  // operand map: quad qa of rows ra, ra + 64 of the block;  epilogue map: quad qs of rows rs + 32 i of a 64-column slab
  const int qa = tid & 7, ra = tid >> 3;
  const uint32_t koff = rt::kmajor_quad_offset(ra, qa, WTR);
  const int qs = tid & 15, rs = tid >> 4;
  float bias4[W_PASSES][4];
#pragma unroll
  for (int J = 0; J < W_PASSES; ++J)
#pragma unroll
    for (int j = 0; j < 4; ++j) bias4[J][j] = p.bias ? p.bias[J * W_SLAB + 4 * qs + j] : 0.0f;
  const bool want_stats = p.partials != nullptr;
  QuadWelford wf[W_PASSES];
#pragma unroll
  for (int J = 0; J < W_PASSES; ++J) wf[J].init();

  float4 pa[2];
  auto load_a = [&](long long tt, int kk) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const long long row = tt * WTR + ra + 64 * i;
      const bool second = kk >= p.KB1;
      pa[i] = (tt < ntiles && row < p.rows)
                  ? rt::ld_quad<true>(second ? p.A2 : p.A, row, p.lda, 32 * (second ? kk - p.KB1 : kk) + 4 * qa)
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto copy_b = [&](int kk, uint32_t s) {
    const unsigned char* src = p.Bimg + (size_t)kk * (2 * W_B_HALF);
    unsigned char* dst = base + s * W_STAGE + 2 * W_A_HALF;
    for (int i = tid; i < 2 * W_B_HALF / 16; i += kThreads) cp_async_16(dst + 16 * i, src + 16 * i);
    cp_async_commit();
  };

  // epilogue of a finished tile, one 64-column slab per call
  bool pending = false;
  long long pend_r0 = 0;
  uint32_t pend_buf = 0;
  int pend_pass = 0;
  auto epi = [&](auto JC) {
    constexpr int J = decltype(JC)::value;
    const int lq = warp & 3, cg = warp >> 2, row = 32 * lq + lane;
    float v[16];
    tc::tmem_ld<16>(taddr + ((uint32_t)(32 * lq) << 16) + pend_buf * (uint32_t)WN + (uint32_t)(J * W_SLAB + cg * 16), v);
    tc::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 4; ++j)
      staging[rt::stage_index(row, 4 * cg + j, W_SLAB / 4)] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    tc::fence_before_sync();
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rs + 32 * i;
      if (pend_r0 + r < p.rows) {
        float4 x = staging[rt::stage_index(r, qs, W_SLAB / 4)];
        x.x += bias4[J][0]; x.y += bias4[J][1]; x.z += bias4[J][2]; x.w += bias4[J][3];
        if (p.relu) { x.x = fmaxf(x.x, 0.0f); x.y = fmaxf(x.y, 0.0f); x.z = fmaxf(x.z, 0.0f); x.w = fmaxf(x.w, 0.0f); }
        *reinterpret_cast<float4*>(p.out + (pend_r0 + r) * WN + J * W_SLAB + 4 * qs) = x;
        if (want_stats) wf[J].push(x);
      }
    }
  };
  auto epi_next = [&]() {
    switch (pend_pass) {
      case 0: epi(std::integral_constant<int, 0>{}); break;
      case 1: epi(std::integral_constant<int, 1>{}); break;
      case 2: epi(std::integral_constant<int, 2>{}); break;
      default: epi(std::integral_constant<int, 3>{}); break;
    }
    if (++pend_pass == W_PASSES) pending = false;
  };

  long long t = blockIdx.x;
  int kb = 0;
  if (t < ntiles) { load_a(t, 0); copy_b(0, 0); }
  uint32_t gc = 0, tb = 0;      // blocks issued so far (stage = gc & 1), TMEM buffer of the current tile
  while (t < ntiles) {
    const uint32_t s = gc & 1u;
    unsigned char* a_hi = base + s * W_STAGE;
    unsigned char* a_lo = a_hi + W_A_HALF;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float4 h, l;
      tc::split4(pa[i], h, l);
      rt::sts4(a_hi + koff + i * 64 * rt::kRowBytes, h);
      rt::sts4(a_lo + koff + i * 64 * rt::kRowBytes, l);
    }
    long long tn = t;
    int kn = kb + 1;
    if (kn == KB) { kn = 0; tn = t + gridDim.x; }
    load_a(tn, kn);                       // next block's rows fly during the barrier and the MMA issue
    cp_async_wait<0>();                   // this block's weight slice has landed (this thread's copies)
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tid == 0) {
      const uint64_t ds = (uint64_t)((s * (uint32_t)W_STAGE) >> 4);
      const rt::OperandDescs od{od0.a_hi + ds, od0.a_lo + ds, od0.b_hi + ds, od0.b_lo + ds};
      rt::issue_kmajor_x3<4, WTR, WN>(taddr + tb * (uint32_t)WN, od, 4, idesc, kb > 0);
      tc::mma_commit(&mbar[s]);
    }
    if (gc >= 1u) tc::mbar_wait(&mbar[s ^ 1u], ((gc - 1u) >> 1) & 1u);   // the other stage's MMAs have read it
    if (tn < ntiles) copy_b(kn, s ^ 1u);
    if (pending) { tc::fence_after_sync(); epi_next(); }
    ++gc;
    if (kn == 0) {                        // every block of this tile is issued: its accumulators become pending
      while (pending) { __syncthreads(); epi_next(); }   // K < 128: passes of the previous tile that found no slot
      pending = true; pend_r0 = t * WTR; pend_buf = tb; pend_pass = 0;
      tb ^= 1u;
    }
    t = tn;
    kb = kn;
  }
  if (gc >= 1u) tc::mbar_wait(&mbar[(gc - 1u) & 1u], ((gc - 1u) >> 1) & 1u);
  tc::fence_after_sync();
  while (pending) { __syncthreads(); epi_next(); }
  __syncthreads();

  if (p.partials) {
    float* rec = reinterpret_cast<float*>(base);   // [W_PASSES][kThreads][9] over stage 0 (every MMA has completed)
#pragma unroll
    for (int J = 0; J < W_PASSES; ++J) wf[J].deposit(rec + ((size_t)J * kThreads + tid) * 9);
    __syncthreads();
    cta_write_quad_stats(rec, kThreads, W_SLAB / 4, WN, tid, p.partials + (size_t)blockIdx.x * (1 + 2 * WN));
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, 512);
}

// ---- partial dW[h][k] = sum_r dP[r][h] act(t_in)[r][k] over this CTA's rows --------------------------------------------
struct WideXtyArgs {
  const float* dP; const float* t_in; Act act_in; long long rows; float* partials;
  // optional: BatchNorm-backward sums of the layer below from du_in (the layer input is in registers here anyway)
  const float* du_in; const float* prev_mean; const float* prev_rstd; float* prev_partials;   // per CTA [2][256]
};

__global__ void __launch_bounds__(kThreads, 1) k_wide_xty(WideXtyArgs p) {
  act_salt(p.act_in);   // device-side dropout salt (CUDA-graph replays)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar[X_STAGES];
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (warp == 0) tc::tmem_alloc(&tmem_base_s, 512);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < X_STAGES; ++s) tc::mbar_init(&mbar[s], 1);
    tc::fence_mbar_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  // M = 128 output rows (channels of dP) per instruction: two halves of the MN-major dP view, 4 MN groups apart
  const uint32_t idesc = tc::idesc_tf32(128, WN, 1, 1);
  // descriptors of stage 0 (stage s adds s * X_STAGE >> 4 to the start-address field); the second half of the dP
  // channels starts 4 MN groups (4 * XR * 128 bytes) further
  const uint32_t a0 = tc::smem_u32(base);
  const rt::OperandDescs od0 = rt::mnmajor_descs(a0, a0 + X_HALF, a0 + 2 * X_HALF, a0 + 3 * X_HALF, XR);
  constexpr uint64_t kHalfStep = (uint64_t)((4 * XR * 128) >> 4);
  // thread = quad q of rows r, r + 8 of a 16-row chunk (both tensors)
  const int q = tid & 63, r = tid >> 6;
  const uint32_t moff = rt::mnmajor_quad_offset(r, q, XR);
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act_in, 4 * q, WN);
  const rt::RowKey rk = rt::row_key(p.act_in);

  const bool want_prev = p.prev_partials != nullptr;
  float pmean[4], prstd[4], ps1[4] = {0.f, 0.f, 0.f, 0.f}, ps2[4] = {0.f, 0.f, 0.f, 0.f};
  rt::bn_stats_quad(pmean, prstd, p.prev_mean, p.prev_rstd, 4 * q, WN, want_prev);

  const long long nchunks = (p.rows + XR - 1) / XR;
  float4 dp[2], tu[2], dd[2];
  auto load_chunk = [&](long long c) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const long long row = c * XR + r + 8 * i;
      const bool live = c < nchunks && row < p.rows;
      dp[i] = live ? rt::ld_quad<true>(p.dP, row, WN, 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
      tu[i] = live ? rt::ld_quad<true>(p.t_in, row, WN, 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
      dd[i] = (live && want_prev) ? rt::ld_quad<true>(p.du_in, row, WN, 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  long long c = blockIdx.x;
  load_chunk(c);
  uint32_t s = 0, use = 0, issued = 0;     // stage, how often it has been used before, chunks issued
  uint32_t last_s = 0, last_par = 0;
  for (; c < nchunks; c += gridDim.x) {
    if (use >= 1u) tc::mbar_wait(&mbar[s], (use - 1u) & 1u);   // the MMAs that read this stage three chunks ago
    unsigned char* a_hi = base + s * X_STAGE;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const long long row = c * XR + r + 8 * i;
      float4 h, l;
      tc::split4(dp[i], h, l);
      rt::sts4(a_hi + moff + i * 8 * rt::kRowBytes, h);
      rt::sts4(a_hi + X_HALF + moff + i * 8 * rt::kRowBytes, l);
      float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < p.rows) {
        u = rt::act_fwd4(p.act_in, cq, tu[i], rk, (uint32_t)row);
        if (want_prev) {
          const float4 dy = rt::act_bwd4(p.act_in, cq, tu[i], dd[i], rk, (uint32_t)row);
          const float tv[4] = {tu[i].x, tu[i].y, tu[i].z, tu[i].w}, dv[4] = {dy.x, dy.y, dy.z, dy.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) bn_sums_add(ps1[j], ps2[j], dv[j], tv[j], pmean[j], prstd[j]);
        }
      }
      tc::split4(u, h, l);
      rt::sts4(a_hi + 2 * X_HALF + moff + i * 8 * rt::kRowBytes, h);
      rt::sts4(a_hi + 3 * X_HALF + moff + i * 8 * rt::kRowBytes, l);
    }
    load_chunk(c + gridDim.x);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (tid == 0) {
      const uint64_t ds = (uint64_t)((s * (uint32_t)X_STAGE) >> 4);
      const rt::OperandDescs lo_half{od0.a_hi + ds, od0.a_lo + ds, od0.b_hi + ds, od0.b_lo + ds};
      const rt::OperandDescs hi_half{lo_half.a_hi + kHalfStep, lo_half.a_lo + kHalfStep, lo_half.b_hi, lo_half.b_lo};
      rt::issue_mnmajor_x3<XR>(taddr, lo_half, idesc, issued > 0u);
      rt::issue_mnmajor_x3<XR>(taddr + (uint32_t)WN, hi_half, idesc, issued > 0u);
      tc::mma_commit(&mbar[s]);
    }
    last_s = s; last_par = use & 1u;
    ++issued;
    if (++s == (uint32_t)X_STAGES) { s = 0; ++use; }
  }
  if (issued > 0u) tc::mbar_wait(&mbar[last_s], last_par);
  tc::fence_after_sync();

  float* part = p.partials + (size_t)blockIdx.x * WN * WN;
  {
    const int lq = warp & 3, cg = warp >> 2;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int h = half * 128 + 32 * lq + lane;
#pragma unroll 1
      for (int sub = 0; sub < 2; ++sub) {
        float v[32];
        const int c0 = cg * 64 + sub * 32;
        if (issued > 0u) {
          tc::tmem_ld<32>(taddr + ((uint32_t)(32 * lq) << 16) + (uint32_t)(half * WN + c0), v);
          tc::tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.0f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(part + (size_t)h * WN + c0 + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
    }
  }
  if (want_prev) {
    float* red = reinterpret_cast<float*>(base);   // [kThreads][8] over stage 0 (every MMA has completed)
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[tid * 8 + j] = ps1[j]; red[tid * 8 + 4 + j] = ps2[j]; }
    __syncthreads();
    for (int c2 = tid; c2 < 2 * WN; c2 += kThreads) {
      const int which = c2 / WN, ch = c2 - which * WN;
      p.prev_partials[(size_t)blockIdx.x * 2 * WN + c2] = quad_sum(red, 8, which * 4, kThreads, WN / 4, ch >> 2, ch & 3);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, 512);
}

// ---- dz = relu'(z) * BatchNorm-backward(dropout-backward(upstream)) materialised, plus its column sums (GraphSAGE) ------
struct WideDzArgs {
  const float* z; const float* du; const float* demb; const int32_t* row_graph; const int32_t* meta;
  Act act_out; BnBwdDev bn; long long rows; float* dz; float* partials;   // per CTA [256]
};

__global__ void __launch_bounds__(kThreads, 2) k_wide_dz(WideDzArgs p) {
  act_salt(p.act_out);   // device-side dropout salt (CUDA-graph replays)
  __shared__ float4 s_red[kThreads];
  const int tid = threadIdx.x, q = tid & 63, r = tid >> 6;
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act_out, 4 * q, WN);
  const rt::RowKey rk = rt::row_key(p.act_out);
  rt::BnQuad bq;
  rt::bn_quad_init(bq, p.bn, 4 * q, WN);
  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  float cs[4] = {0.f, 0.f, 0.f, 0.f};
  const long long step = (long long)gridDim.x * 16;
  for (long long row0 = (long long)blockIdx.x * 16 + r; row0 < p.rows; row0 += step) {
    float4 zv[2], uv[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {          // two rows in flight per thread
      const long long row = row0 + 8 * i;
      zv[i] = make_float4(0.f, 0.f, 0.f, 0.f); uv[i] = zv[i];
      if (row < p.rows) {
        zv[i] = rt::ld_quad<true>(p.z, row, WN, 4 * q);
        if (p.du) uv[i] = rt::ld_quad<true>(p.du, row, WN, 4 * q);
        else {
          const int g = p.row_graph[row];
          uv[i] = rt::pooled_quad<true>(p.demb, g, WN, 4 * q, meta[g].y);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const long long row = row0 + 8 * i;
      if (row >= p.rows) continue;
      const float4 dz = rt::dz4<true>(p.act_out, cq, p.bn, bq, zv[i], uv[i], rk, (uint32_t)row);
      cs[0] += dz.x; cs[1] += dz.y; cs[2] += dz.z; cs[3] += dz.w;
      rt::st_quad<true>(p.dz, row, WN, 4 * q, dz);
    }
  }
  s_red[tid] = make_float4(cs[0], cs[1], cs[2], cs[3]);
  __syncthreads();
  if (tid < WN) p.partials[(size_t)blockIdx.x * WN + tid] = quad_sum(reinterpret_cast<const float*>(s_red), 4, 0, kThreads, WN / 4, tid >> 2, tid & 3);
}

bool al16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }

int launch_prep_w(const float* W, int ldw, int K, int transposed, unsigned char* img, cudaStream_t stream) {
  auto kfn = k_wide_prep_w;
  CGNN_LAUNCH(kfn, 64, 256, 0, stream, W, ldw, K, transposed, img);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int launch_wide_xw(const float* A, long long rows, int K, const unsigned char* img, const float* bias, float* out,
                   double* partials, size_t partial_bytes, int* grid_out, cudaStream_t stream, const float* A2 = nullptr,
                   int KB1 = -1, int relu = 0) {
  const DeviceInfo dev = device_info();
  if (W_XW_SMEM > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  WideXwArgs a;
  a.A = A; a.rows = rows; a.K = K; a.Bimg = img; a.bias = bias; a.out = out; a.partials = partials;
  a.A2 = A2; a.KB1 = KB1 < 0 ? K / 32 : KB1; a.lda = A2 ? 32 * a.KB1 : K; a.relu = relu;
  const long long ntiles = (rows + WTR - 1) / WTR;
  long long grid = dev.sm_count;
  if (grid > ntiles) grid = ntiles;
  if (partials) {
    const size_t rec = (size_t)(1 + 2 * WN) * sizeof(double);
    if ((size_t)grid * rec > partial_bytes) grid = (long long)(partial_bytes / rec);
  }
  if (grid < 1) return CGNN_ERR_WORKSPACE;
  *grid_out = (int)grid;
  auto kfn = k_wide_xw;
  cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)W_XW_SMEM);
  CGNN_LAUNCH(kfn, (unsigned)grid, kThreads, W_XW_SMEM, stream, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int launch_wide_xty(const float* dP, const float* t_in, const cgnn_act_t* act_in, long long rows, float* partials,
                    size_t partial_bytes, const float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_partials,
                    size_t prev_bytes, int* grid_out, cudaStream_t stream) {
  const DeviceInfo dev = device_info();
  if (W_XTY_SMEM > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  WideXtyArgs a;
  a.dP = dP; a.t_in = t_in; a.act_in = make_act(act_in); a.rows = rows; a.partials = partials;
  a.du_in = du_in; a.prev_mean = prev_mean; a.prev_rstd = prev_rstd; a.prev_partials = prev_partials;
  const long long nchunks = (rows + XR - 1) / XR;
  long long grid = dev.sm_count;
  if (grid > nchunks) grid = nchunks;
  const size_t rec = (size_t)WN * WN * sizeof(float);
  if ((size_t)grid * rec > partial_bytes) grid = (long long)(partial_bytes / rec);
  if (prev_partials && (size_t)grid * 2 * WN * sizeof(float) > prev_bytes) grid = (long long)(prev_bytes / (2 * WN * sizeof(float)));
  if (grid < 1) return CGNN_ERR_WORKSPACE;
  *grid_out = (int)grid;
  auto kfn = k_wide_xty;
  cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)W_XTY_SMEM);
  CGNN_LAUNCH(kfn, (unsigned)grid, kThreads, W_XTY_SMEM, stream, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

constexpr size_t kImgBytes = (size_t)8 * WN * WN;   // hi + lo images of a 256 x 256 weight

}  // namespace

bool wide_shape(int d_in, int H) { return d_in == WN && H == WN; }

// z = (A^ act(t_in)) W^T + b for H = d_in = 256.  Returns CGNN_OK when launched (the caller merges *grid_out statistics
// records at the start of `workspace`), -1 when the shape is not covered, else an error status.
int launch_gcn_fwd_wide(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                        int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z,
                        int want_stats, int* grid_out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!wide_shape(d_in, H)) return -1;
  if (!csr->agg_in || csr->agg_kind != AGG_GCN || !gather_supported(WN, max_nodes, max_edges)) return -1;
  if (!al16(t_in) || !al16(z) || !al16(W) || !al16(workspace)) return -1;
  const DeviceInfo dev = device_info();
  const size_t stats_bytes = (((size_t)dev.sm_count * (1 + 2 * WN) * sizeof(double)) + 1023) & ~(size_t)1023;
  if (!workspace || workspace_bytes < stats_bytes + kImgBytes) return CGNN_ERR_WORKSPACE;
  unsigned char* img = (unsigned char*)workspace + stats_bytes;
  GatherArgs ga{};
  ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_in;
  ga.C = WN; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
  ga.src = t_in; ga.act = make_act(act); ga.out = z;
  int g0 = 0;
  int rc = launch_gather(GATHER_GCN_FWD, ga, &g0, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_prep_w(W, d_in, d_in, 0, img, stream);
  if (rc != CGNN_OK) return rc;
  return launch_wide_xw(z, rows, d_in, img, bias, z, want_stats ? (double*)workspace : nullptr, stats_bytes, grid_out, stream);
}

// Backward of the same layer; `scratch` = [rows, 256] floats (dP).  Same return convention.
int launch_gcn_bwd_wide(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn,
                        const float* t_in, const cgnn_act_t* act_in, const float* W, const cgnn_csr_t* csr, const int64_t* ptr,
                        int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges,
                        float* dW, float* dbias, float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64,
                        float* scratch, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!wide_shape(d_in, H)) return -1;
  if (!scratch || !csr->agg_out || csr->agg_kind != AGG_GCN || !gather_supported(WN, max_nodes, max_edges)) return -1;
  if (!al16(scratch) || !al16(z) || !al16(t_in) || !al16(W) || !al16(workspace) || (du && !al16(du)) || (demb && !al16(demb)) ||
      (du_in && !al16(du_in)))
    return -1;
  const DeviceInfo dev = device_info();
  const size_t region_a = (((size_t)2 * dev.sm_count * WN * sizeof(float)) + 1023) & ~(size_t)1023;   // dbias partials
  const size_t region_p = (((size_t)dev.sm_count * 2 * WN * sizeof(float)) + 1023) & ~(size_t)1023;      // prev-sum partials
  if (workspace_bytes < region_a + region_p + kImgBytes + (size_t)WN * WN * sizeof(float)) return CGNN_ERR_WORKSPACE;
  float* prev_parts = (float*)((unsigned char*)workspace + region_a);
  unsigned char* img = (unsigned char*)workspace + region_a + region_p;
  float* parts = (float*)(img + kImgBytes);
  const size_t parts_bytes = workspace_bytes - region_a - region_p - kImgBytes;
  const bool fuse_prev = prev_sums != nullptr && du_in != nullptr;

  GatherArgs ga{};
  ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_out;
  ga.C = WN; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
  ga.src = z; ga.act = make_act(act_out); ga.du = du; ga.demb = demb; ga.bn = make_bn_bwd(bn);
  ga.out = scratch; ga.partials = (float*)workspace; ga.part_stride = WN;
  int g1 = 0, g2 = 0, g3 = 0;
  int rc = launch_gather(GATHER_GCN_BWD, ga, &g1, stream);
  if (rc != CGNN_OK) return rc;
  if ((size_t)g1 * WN * sizeof(float) > region_a) return CGNN_ERR_WORKSPACE;
  if (du_in) {
    rc = launch_prep_w(W, d_in, H, 1, img, stream);     // operand row = input channel, contraction over h: W[h][n]
    if (rc != CGNN_OK) return rc;
    rc = launch_wide_xw(scratch, rows, H, img, nullptr, du_in, nullptr, 0, &g2, stream);
    if (rc != CGNN_OK) return rc;
  }
  rc = launch_wide_xty(scratch, t_in, act_in, rows, parts, parts_bytes, fuse_prev ? du_in : nullptr, prev_mean, prev_rstd,
                       fuse_prev ? prev_parts : nullptr, region_p, &g3, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_reduce_partials((const float*)workspace, g1, WN, 1, WN, WN, dbias, stream);
  if (rc) return rc;
  rc = launch_reduce_partials(parts, g3, WN * WN, WN, WN, WN, dW, stream);
  if (rc) return rc;
  if (fuse_prev) rc = launch_reduce_partials(prev_parts, g3, 2 * WN, 2, WN, WN, prev_sums, stream, 0, prev_sums64);
  (void)ptr;
  return rc;
}
// GraphSAGE, H = d_in = 256:  z = relu([u || agg] W^T + b).  The gather writes the weighted mean into `agg` and, from the same
// staged rows, u = act(t_in) into z; the contraction then reads its K = 512 operand from z and agg and writes z in place.
int launch_sage_fwd_wide(const float* t_in, const cgnn_act_t* act, float* agg, const float* W, const float* bias,
                         const cgnn_csr_t* csr, int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes,
                         int32_t max_edges, float* z, int want_stats, int* grid_out, void* workspace, size_t workspace_bytes,
                         cudaStream_t stream) {
  if (!wide_shape(d_in, H)) return -1;
  if (!agg || !csr->agg_in || csr->agg_kind != AGG_SAGE || !gather_supported(WN, max_nodes, max_edges)) return -1;
  if (!al16(t_in) || !al16(z) || !al16(agg) || !al16(W) || !al16(workspace)) return -1;
  const DeviceInfo dev = device_info();
  const size_t stats_bytes = (((size_t)dev.sm_count * (1 + 2 * WN) * sizeof(double)) + 1023) & ~(size_t)1023;
  if (!workspace || workspace_bytes < stats_bytes + 2 * kImgBytes) return CGNN_ERR_WORKSPACE;
  unsigned char* img = (unsigned char*)workspace + stats_bytes;
  GatherArgs ga{};
  ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_in;
  ga.C = WN; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
  ga.src = t_in; ga.act = make_act(act); ga.out = agg; ga.out_u = z;
  int g0 = 0;
  int rc = launch_gather(GATHER_SAGE_FWD, ga, &g0, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_prep_w(W, 2 * d_in, 2 * d_in, 0, img, stream);
  if (rc != CGNN_OK) return rc;
  return launch_wide_xw(z, rows, 2 * d_in, img, bias, z, want_stats ? (double*)workspace : nullptr, stats_bytes, grid_out, stream,
                        agg, d_in / 32, 1);
}

// Backward of the same layer; `scratch` = [3][rows, 256] floats: d_u, d_agg, dz.
int launch_sage_bwd_wide(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn,
                         const float* t_in, const float* agg, const cgnn_act_t* act_in, const float* W, const cgnn_csr_t* csr,
                         int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* dW,
                         float* dbias, float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64, float* scratch,
                         void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!wide_shape(d_in, H)) return -1;
  if (!scratch || !agg || !csr->agg_out || !csr->row_graph || csr->agg_kind != AGG_SAGE || !gather_supported(WN, max_nodes, max_edges))
    return -1;
  if (!al16(scratch) || !al16(z) || !al16(t_in) || !al16(agg) || !al16(W) || !al16(workspace) || (du && !al16(du)) ||
      (demb && !al16(demb)) || (du_in && !al16(du_in)))
    return -1;
  const DeviceInfo dev = device_info();
  const size_t region_a = (((size_t)2 * dev.sm_count * 2 * WN * sizeof(float)) + 1023) & ~(size_t)1023;   // dbias / prev-sum partials
  if (workspace_bytes < region_a + kImgBytes + (size_t)WN * WN * sizeof(float)) return CGNN_ERR_WORKSPACE;
  unsigned char* img = (unsigned char*)workspace + region_a;
  float* parts = (float*)(img + kImgBytes);
  const size_t parts_bytes = workspace_bytes - region_a - kImgBytes;
  float* direct = scratch;
  float* nbr = scratch + (size_t)rows * WN;
  float* dz = scratch + (size_t)2 * rows * WN;

  // (1) dz and dbias
  WideDzArgs a{};
  a.z = z; a.du = du; a.demb = demb; a.row_graph = csr->row_graph; a.meta = csr->graph_meta;
  a.act_out = make_act(act_out); a.bn = make_bn_bwd(bn);
  a.rows = rows; a.dz = dz; a.partials = (float*)workspace;
  long long gdz = 2LL * dev.sm_count;
  if (gdz > (rows + 15) / 16) gdz = (rows + 15) / 16;
  {
    auto kfn = k_wide_dz;
    CGNN_LAUNCH(kfn, (unsigned)gdz, kThreads, 0, stream, a);
    CGNN_CHECK_LAUNCH();
  }
  int rc = launch_reduce_partials((const float*)workspace, (int)gdz, WN, 1, WN, WN, dbias, stream);
  if (rc) return rc;
  // (2) dW = dz^T [u || agg]: two 256 x 256 halves through the same partial buffer
  int g3 = 0;
  rc = launch_wide_xty(dz, t_in, act_in, rows, parts, parts_bytes, nullptr, nullptr, nullptr, nullptr, 0, &g3, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_reduce_partials(parts, g3, WN * WN, WN, WN, WN, dW, stream, 2 * WN);
  if (rc) return rc;
  rc = launch_wide_xty(dz, agg, nullptr, rows, parts, parts_bytes, nullptr, nullptr, nullptr, nullptr, 0, &g3, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_reduce_partials(parts, g3, WN * WN, WN, WN, WN, dW + WN, stream, 2 * WN);
  if (rc) return rc;
  if (!du_in) return CGNN_OK;
  // (3) [d_u || d_agg] = dz W: the two column halves of W as transposed operand images
  int g2 = 0;
  rc = launch_prep_w(W, 2 * d_in, H, 1, img, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_wide_xw(dz, rows, H, img, nullptr, direct, nullptr, 0, &g2, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_prep_w(W + d_in, 2 * d_in, H, 1, img, stream);
  if (rc != CGNN_OK) return rc;
  rc = launch_wide_xw(dz, rows, H, img, nullptr, nbr, nullptr, 0, &g2, stream);
  if (rc != CGNN_OK) return rc;
  // (4) du_in = d_u + A~^T d_agg, BatchNorm-backward sums of the layer below
  GatherArgs ga{};
  ga.meta = csr->graph_meta; ga.B = num_graphs; ga.blob = csr->agg_out;
  ga.C = WN; ga.max_nodes = max_nodes; ga.max_edges = max_edges;
  ga.src = nbr; ga.act = make_act(act_in); ga.direct = direct; ga.t_raw = t_in;
  ga.prev_mean = prev_mean; ga.prev_rstd = prev_rstd; ga.want_prev = prev_sums ? 1 : 0;
  ga.out = du_in;
  ga.partials = (float*)workspace; ga.part_stride = 2 * WN;
  int g4 = 0;
  rc = launch_gather(GATHER_SAGE_BWD, ga, &g4, stream);
  if (rc != CGNN_OK) return rc;
  if ((size_t)g4 * 2 * WN * sizeof(float) > region_a) return CGNN_ERR_WORKSPACE;
  if (prev_sums) return launch_reduce_partials(ga.partials, g4, 2 * WN, 2, WN, WN, prev_sums, stream, 0, prev_sums64);
  return CGNN_OK;
}
#endif  // CGNN_EMU
}  // namespace cgnn
