// tc_project.cu - stand-alone fp32-grade projection on the 5th-generation tensor cores:
//   P[rows, N] = X[rows, K] W[N, K]^T   as 3xTF32 (tcgen05.mma kind::tf32, accumulators in TMEM).
// This is the per-layer H.W contraction of reference models.py:111 / :152 in isolation; the layer kernels
// embed the same sequence.  It doubles as the on-device check of the descriptor / swizzle / TMEM plumbing.
#include "tc05.cuh"

#include <cstdlib>

namespace cgnn {
#ifndef CGNN_EMU

constexpr int kTcRows = 128;   // rows of X per CTA = UMMA M

__global__ void __launch_bounds__(128) k_project_tf32x3(const float* __restrict__ X, const float* __restrict__ W,
                                                        long long rows, int K, int N, float* __restrict__ P,
                                                        uint32_t tmem_cols) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  const int kblocks = K >> 5;
  unsigned char* a_hi = base;
  unsigned char* a_lo = a_hi + kblocks * kTcRows * 128;
  unsigned char* b_hi = a_lo + kblocks * kTcRows * 128;
  unsigned char* b_lo = b_hi + kblocks * N * 128;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long r0 = (long long)blockIdx.x * kTcRows;
  if (warp == 0) tc::tmem_alloc(&tmem_base_s, tmem_cols);
  if (tid == 0) { tc::mbar_init(&mbar, 1); tc::fence_mbar_init(); }

  const int q = K >> 2;
  for (int idx = tid; idx < kTcRows * q; idx += blockDim.x) {
    const int r = idx / q, k = (idx - r * q) << 2;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < rows) v = *reinterpret_cast<const float4*>(X + (r0 + r) * K + k);
    tc::store_split4(a_hi, a_lo, r, k, kTcRows, v);
  }
  for (int idx = tid; idx < N * q; idx += blockDim.x) {
    const int n = idx / q, k = (idx - n * q) << 2;
    tc::store_split4(b_hi, b_lo, n, k, N, *reinterpret_cast<const float4*>(W + (size_t)n * K + k));
  }
  tc::fence_proxy_async();      // generic-proxy smem writes -> visible to the tensor core (async proxy)
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  if (tid == 0) {
    tc::mma_tf32x3(taddr, tc::smem_u32(a_hi), tc::smem_u32(a_lo), tc::smem_u32(b_hi), tc::smem_u32(b_lo), kTcRows, N, K);
    tc::mma_commit(&mbar);
  }
  tc::mbar_wait(&mbar, 0);
  tc::fence_after_sync();
  const long long row = r0 + 32 * warp + lane;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    tc::tmem_ld<32>(taddr + ((uint32_t)(32 * warp) << 16) + (uint32_t)c0, v);
    tc::tmem_ld_wait();
    if (row < rows) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (c0 + j < N)
          *reinterpret_cast<float4*>(P + row * N + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, tmem_cols);
}
// The same product with the A operand in TENSOR MEMORY (experiment for the next generation of row-tile kernels: the
// shared-memory pipe carries the 3 x A reads of every SS-mode K step, profiles/r01d_summary.md).  Thread = row: it
// loads its row, splits it and writes hi / lo straight into its TMEM lane with tcgen05.st - A never touches shared
// memory.  TMEM columns: [0, N) accumulator, [N, N + K) A hi, [N + K, N + 2K) A lo.
__global__ void __launch_bounds__(128) k_project_tf32x3_ts(const float* __restrict__ X, const float* __restrict__ W,
                                                           long long rows, int K, int N, float* __restrict__ P,
                                                           uint32_t tmem_cols) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  const int kblocks = K >> 5;
  unsigned char* b_hi = base;
  unsigned char* b_lo = b_hi + kblocks * N * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long r0 = (long long)blockIdx.x * kTcRows;
  if (warp == 0) tc::tmem_alloc(&tmem_base_s, tmem_cols);
  if (tid == 0) { tc::mbar_init(&mbar, 1); tc::fence_mbar_init(); }
  const int q = K >> 2;
  for (int idx = tid; idx < N * q; idx += blockDim.x) {
    const int n = idx / q, k = (idx - n * q) << 2;
    tc::store_split4(b_hi, b_lo, n, k, N, *reinterpret_cast<const float4*>(W + (size_t)n * K + k));
  }
  tc::fence_proxy_async();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t taddr = tmem_base_s;
  const uint32_t lane_base = taddr + ((uint32_t)(32 * warp) << 16);
  const long long row = r0 + tid;
  for (int k = 0; k < K; k += 8) {
    float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
    if (row < rows) {
      x0 = *reinterpret_cast<const float4*>(X + row * K + k);
      x1 = *reinterpret_cast<const float4*>(X + row * K + k + 4);
    }
    const float v[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
    float h[8], l[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { h[j] = tc::tf32_hi(v[j]); l[j] = v[j] - h[j]; }
    tc::tmem_st<8>(lane_base + (uint32_t)(N + k), h);
    tc::tmem_st<8>(lane_base + (uint32_t)(N + K + k), l);
  }
  tc::tmem_st_wait();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  if (tid == 0) {
    const uint32_t idesc = tc::idesc_tf32(kTcRows, N);
    const uint32_t bh = tc::smem_u32(b_hi), bl = tc::smem_u32(b_lo);
    uint32_t acc = 0;
    for (int k = 0; k < K; k += 8) {
      const uint32_t kb = (uint32_t)(k >> 5), ko = (uint32_t)((k & 31) * 4);
      const uint64_t dh = tc::smem_desc_sw128(bh + kb * (uint32_t)N * 128u + ko), dl = tc::smem_desc_sw128(bl + kb * (uint32_t)N * 128u + ko);
      tc::mma_tf32x3_ts(taddr, taddr + (uint32_t)(N + k), taddr + (uint32_t)(N + K + k), dh, dl, idesc, acc);
      acc = 1;
    }
    tc::mma_commit(&mbar);
  }
  tc::mbar_wait(&mbar, 0);
  tc::fence_after_sync();
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    tc::tmem_ld<32>(lane_base + (uint32_t)c0, v);
    tc::tmem_ld_wait();
    if (row < rows) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (c0 + j < N)
          *reinterpret_cast<float4*>(P + row * N + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(taddr, tmem_cols);
}
#endif
}  // namespace cgnn

extern "C" int cgnn_project_tf32x3(const float* X, const float* W, int64_t rows, int32_t K, int32_t N, float* P,
                                   cgnn_stream_t stream_) {
#ifdef CGNN_EMU
  (void)X; (void)W; (void)rows; (void)K; (void)N; (void)P; (void)stream_;
  return CGNN_ERR_INVALID_ARG;   // tensor cores do not exist in the simulator
#else
  using namespace cgnn;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!X || !W || !P || rows < 0 || K <= 0 || N <= 0) return CGNN_ERR_INVALID_ARG;
  if (K % 32 != 0 || N % 32 != 0 || N > 256 || K > 256) return CGNN_ERR_INVALID_ARG;
  if ((((uintptr_t)X) | ((uintptr_t)W) | ((uintptr_t)P)) & 15u) return CGNN_ERR_INVALID_ARG;
  if (rows == 0) return CGNN_OK;
  const size_t smem = (size_t)(K / 32) * (2 * kTcRows + 2 * N) * 128 + 1024;
  const DeviceInfo dev = device_info();
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  if (N + 2 * K <= 512) {   // A operand in tensor memory whenever its columns fit next to the accumulators (27 - 36 % faster, profiles/r01d_summary.md)
    uint32_t tcols = 32;
    while (tcols < (uint32_t)(N + 2 * K)) tcols <<= 1;
    const size_t smem_ts = (size_t)(K / 32) * (2 * N) * 128 + 1024;
    auto kts = k_project_tf32x3_ts;
    if (smem_ts > 48 * 1024) cudaFuncSetAttribute(kts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ts);
    const unsigned grid_ts = (unsigned)((rows + kTcRows - 1) / kTcRows);
    CGNN_LAUNCH(kts, grid_ts, 128, smem_ts, stream, X, W, (long long)rows, (int)K, (int)N, P, tcols);
    CGNN_CHECK_LAUNCH();
    return CGNN_OK;
  }
  uint32_t cols = 32;
  while (cols < (uint32_t)N) cols <<= 1;
  auto kfn = k_project_tf32x3;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const unsigned grid = (unsigned)((rows + kTcRows - 1) / kTcRows);
  CGNN_LAUNCH(kfn, grid, 128, smem, stream, X, W, (long long)rows, (int)K, (int)N, P, cols);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
#endif
}
