// common.cuh - shared device helpers for the cgnn sm_100a kernels.
//
// The kernels are written against a small portable subset of CUDA so that the very same
// sources can also be compiled by g++ against tests/emu/cuda_emu.h (-DCGNN_EMU) for
// logic tests on GPU-less boxes.  The product build is nvcc -arch sm_100a only.
#pragma once

#include "../../include/cgnn.h"

#ifdef CGNN_EMU
#include "cuda_emu.h"
#define CGNN_SMEM_DECL unsigned char* cgnn_smem = cgnn_emu::g_dyn_smem
#define CGNN_LAUNCH(kernel, grid, block, smem, stream, ...) \
  (cgnn::count_launch(), cgnn_emu::launch(dim3(grid), dim3(block), (smem), [=]() { kernel(__VA_ARGS__); }))
#else
#include <cuda_runtime.h>
#define CGNN_SMEM_DECL extern __shared__ __align__(16) unsigned char cgnn_smem[]
#define CGNN_LAUNCH(kernel, grid, block, smem, stream, ...) \
  (cgnn::count_launch(), kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__))
#endif

#include <stdint.h>

namespace cgnn {

void count_launch();  // bumps the process-wide kernel-launch counter (cgnn_kernel_launches)

constexpr int kThreads = 512;          // threads per CTA of the tile kernels
constexpr int kWarps = kThreads / 32;
constexpr int kChunkRows = 64;         // rows per projection chunk
constexpr unsigned kFull = 0xffffffffu;

// ---- host-side launch helpers --------------------------------------------------------
struct DeviceInfo {
  int sm_count;
  int smem_optin;  // max dynamic shared memory per CTA (bytes)
};
DeviceInfo device_info();
void set_cuda_error(int err);

#define CGNN_CHECK_LAUNCH()                         \
  do {                                              \
    cudaError_t e__ = cudaGetLastError();           \
    if (e__ != cudaSuccess) {                       \
      cgnn::set_cuda_error((int)e__);               \
      return CGNN_ERR_CUDA;                         \
    }                                               \
  } while (0)

static inline __host__ __device__ int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Persistent grid: one CTA per work item up to `resident` CTAs per SM.
static inline int persistent_grid(long long items, size_t smem_bytes, const DeviceInfo& d, int threads) {
  long long per_sm = (228 * 1024) / (long long)(smem_bytes + 1024);
  long long by_threads = 2048 / threads;
  if (per_sm > by_threads) per_sm = by_threads;
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  long long g = per_sm * d.sm_count;
  if (g > items) g = items;
  if (g < 1) g = 1;
  return (int)g;
}

// ---- activation-on-load: BatchNorm affine + ReLU + dropout -----------------------------
// Device-side form of cgnn_act_t with the dropout constants derived once on the host.
struct Act {
  const float* scale;
  const float* shift;
  int relu;
  int drop;           // 1 when p_drop > 0
  uint32_t k0, k1;    // dropout stream key (seed, site)
  uint32_t thresh;    // keep when 16 random bits >= thresh; thresh = round(p * 65536)
  float keep_scale;   // 1 / (1 - p)
  long long row_base;
  const uint32_t* salt;   // optional device words {s0, s1} folded into the stream key at kernel start (act_salt)
};

static inline Act make_act(const cgnn_act_t* a) {
  Act r;
  r.scale = nullptr; r.shift = nullptr; r.relu = 0; r.drop = 0;
  r.k0 = r.k1 = 0; r.thresh = 0; r.keep_scale = 1.0f; r.row_base = 0; r.salt = nullptr;
  if (!a) return r;
  r.scale = a->scale;
  r.shift = a->shift;
  r.relu = a->relu;
  r.row_base = a->row_base;
  if (a->p_drop > 0.0f) {
    r.drop = 1;
    double t = (double)a->p_drop * 65536.0 + 0.5;
    r.thresh = t >= 65535.0 ? 65535u : (uint32_t)t;
    r.keep_scale = 1.0f / (1.0f - a->p_drop);
    r.k0 = (uint32_t)(a->seed & 0xffffffffu) ^ (a->site * 0x9E3779B9u);
    r.k1 = (uint32_t)(a->seed >> 32) + a->site * 0x85EBCA6Bu + 0x27D4EB2Fu;
    r.salt = a->salt;
  }
  return r;
}

// ---- BatchNorm backward: dz = scale * (dy - s1 / count - xhat * s2 / count), xhat = (t - mean) * rstd -----------------
// Device-side form of cgnn_bn_bwd_t (has = 0: no BatchNorm after this layer).
struct BnBwdDev {
  const float* scale; const float* mean; const float* rstd; const float* s1; const float* s2;
  float inv_count; int train, has;
  const double* sums64;     // [2, C] in double, read instead of s1 / s2 when given
};

static inline BnBwdDev make_bn_bwd(const cgnn_bn_bwd_t* bn) {
  BnBwdDev r{};
  if (!bn) return r;
  r.scale = bn->scale; r.mean = bn->mean; r.rstd = bn->rstd; r.s1 = bn->s1; r.s2 = bn->s2; r.sums64 = bn->sums64;
  r.inv_count = bn->count > 0 ? (float)(1.0 / bn->count) : 0.0f;
  r.train = bn->train; r.has = 1;
  return r;
}

// sum / count of channel c: from the double record when there is one
__device__ __forceinline__ float bn_sum_over_count(const float* s, const double* s64, int c, float inv_count) {
  return s64 ? (float)(s64[c] * (double)inv_count) : s[c] * inv_count;
}
// the per-channel coefficients of the BatchNorm backward, channel c of C (c >= C: padding)
struct BnCoef {
  float mean, rstd, bsc, s1n, s2n;   // in the order bn_bwd_dz reads them
};
__device__ __forceinline__ BnCoef bn_bwd_coef(const BnBwdDev& bn, int c, int C) {
  const bool ok = bn.has && c < C;
  BnCoef k;
  k.bsc = ok ? bn.scale[c] : (c < C ? 1.0f : 0.0f);
  k.mean = ok ? bn.mean[c] : 0.0f;
  k.rstd = ok ? bn.rstd[c] : 0.0f;
  k.s1n = (ok && bn.train) ? bn_sum_over_count(bn.s1, bn.sums64, c, bn.inv_count) : 0.0f;
  k.s2n = (ok && bn.train) ? bn_sum_over_count(bn.s2, bn.sums64 ? bn.sums64 + C : nullptr, c, bn.inv_count) : 0.0f;
  return k;
}
// dz of one element in train mode (eval mode: dz = bsc * dy)
__device__ __forceinline__ float bn_bwd_dz(const BnCoef& k, float t, float dy) {
  const float xh = (t - k.mean) * k.rstd;
  return k.bsc * (dy - k.s1n - xh * k.s2n);
}
// one element's share of the BatchNorm-backward sums of the layer below: s1 += dy, s2 += dy * xhat
__device__ __forceinline__ void bn_sums_add(float& s1, float& s2, float dy, float t, float mean, float rstd) {
  const float xh = (t - mean) * rstd;
  s1 += dy;
  s2 = fmaf(dy, xh, s2);
}

// d loss / d row of a mean-pooled subject of n rows = d loss / d embedding * pool_bwd_scale(n)
__device__ __forceinline__ float pool_bwd_scale(int n) { return 1.0f / ((float)n + 1e-8f); }

// Dropout streams of CUDA-graph replays: the host-side seed is baked into a captured launch, so a graphed training step
// keeps two salt words on the device (refreshed by cgnn_step_tick inside the graph) and every kernel folds them into
// its stream key before anything else.  No salt (eager mode): the stream is a function of the host seed alone.
__device__ __forceinline__ void act_salt(Act& a) {
  if (a.drop && a.salt != nullptr) {
    a.k0 ^= a.salt[0];
    a.k1 += a.salt[1];
  }
}

__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
// Dropout stream: one mix per row (cheap, no avalanche of its own), one full-avalanche hash per channel QUAD, from
// which the four 16-bit fields of the quad are cut - the second pair from a multiply / xor-shift of the first word.
__device__ __forceinline__ uint32_t drop_row_hash(const Act& a, long long grow) {
  uint32_t lo = (uint32_t)grow, hi = (uint32_t)((unsigned long long)grow >> 32);
  return (lo * 0x9E3779B1u) ^ a.k0 ^ fmix32(hi + a.k1);
}
__device__ __forceinline__ uint32_t drop_second_word(uint32_t y) {
  uint32_t w = y * 0x9E3779B1u + 0x7F4A7C15u;
  return w ^ (w >> 15);
}
// the stream's key of channel quad `quad` (channels 4 quad .. 4 quad + 3), the same for every row
__device__ __forceinline__ uint32_t drop_quad_key(const Act& a, int quad) { return (uint32_t)quad * 0x632BE5ABu + a.k1; }
// whether the low (half 0) or high (half 1) 16-bit field of a stream word keeps its channel
__device__ __forceinline__ bool drop_field_kept(const Act& a, uint32_t w, int half) { return (half ? (w >> 16) : (w & 0xffffu)) >= a.thresh; }
// keep bits of a channel quad at a row: bit j = channel 4 quad + j kept
__device__ __forceinline__ uint32_t drop_keep4(const Act& a, uint32_t row_hash, uint32_t quad_key) {
  const uint32_t w0 = fmix32(row_hash + quad_key), w1 = drop_second_word(w0);
  return (drop_field_kept(a, w0, 0) ? 1u : 0u) | (drop_field_kept(a, w0, 1) ? 2u : 0u) | (drop_field_kept(a, w1, 0) ? 4u : 0u) |
         (drop_field_kept(a, w1, 1) ? 8u : 0u);
}
__device__ __forceinline__ bool drop_keep(const Act& a, uint32_t row_hash, int c) {
  const uint32_t y = fmix32(row_hash + drop_quad_key(a, c >> 2));
  return drop_field_kept(a, (c & 2) ? drop_second_word(y) : y, c & 1);
}

// u = dropout(relu?(sc * t + sh)).  `affine` is warp-uniform (a.scale != nullptr).
__device__ __forceinline__ float act_fwd(const Act& a, bool affine, float t, float sc, float sh,
                                         uint32_t row_hash, int c) {
  float y = affine ? fmaf(t, sc, sh) : t;
  if (a.relu) y = fmaxf(y, 0.0f);
  if (a.drop) y = drop_keep(a, row_hash, c) ? y * a.keep_scale : 0.0f;
  return y;
}
// d act / d y at this element, times upstream du:   dy = du * keep_scale * [kept] * [y > 0 or no relu]
__device__ __forceinline__ float act_bwd(const Act& a, bool affine, float t, float sc, float sh,
                                         uint32_t row_hash, int c, float du) {
  float y = affine ? fmaf(t, sc, sh) : t;
  bool pass = !(a.relu && !(y > 0.0f));
  if (a.drop) { pass = pass && drop_keep(a, row_hash, c); du *= a.keep_scale; }
  return pass ? du : 0.0f;
}

// ---- asynchronous global->shared copies (LDGSTS) ---------------------------------------------
// Under the simulator these degrade to immediate copies, which is a legal (stronger) ordering.
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem) {
#ifdef CGNN_EMU
  memcpy(smem, gmem, 16);
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
#ifdef CGNN_EMU
  memcpy(smem, gmem, 4);
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() {
#ifndef CGNN_EMU
  asm volatile("cp.async.commit_group;\n" ::: "memory");
#endif
}
// Wait until at most N of the most recently committed groups are still in flight.
template <int N>
__device__ __forceinline__ void cp_async_wait() {
#ifndef CGNN_EMU
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
#endif
}
// Copy `count` 4-byte words global->shared with the whole CTA; 16-byte transfers when both sides allow.
__device__ __forceinline__ void cp_async_words(void* smem, const void* gmem, int count) {
  const bool wide = ((((uintptr_t)smem) | ((uintptr_t)gmem)) & 15u) == 0;
  if (wide) {
    const int n16 = count >> 2;
    for (int i = threadIdx.x; i < n16; i += blockDim.x)
      cp_async_16(reinterpret_cast<char*>(smem) + 16 * i, reinterpret_cast<const char*>(gmem) + 16 * i);
    for (int i = (n16 << 2) + threadIdx.x; i < count; i += blockDim.x)
      cp_async_4(reinterpret_cast<char*>(smem) + 4 * i, reinterpret_cast<const char*>(gmem) + 4 * i);
  } else {
    for (int i = threadIdx.x; i < count; i += blockDim.x)
      cp_async_4(reinterpret_cast<char*>(smem) + 4 * i, reinterpret_cast<const char*>(gmem) + 4 * i);
  }
}

// ---- warp helpers ----------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}

// ---- 4x4 register-tile GEMM micro kernels over shared memory ---------------------------
// acc[i][j] += sum_k A[(r0+i)*lda + k] * B[k*ldb + c0 + j],  k in [0, K4), K4 % 4 == 0.
// A rows and B rows must be 16-byte aligned at k % 4 == 0 / c0 % 4 == 0.
__device__ __forceinline__ void mma_4x4(const float* __restrict__ A, int lda, const float* __restrict__ B,
                                        int ldb, int K4, float (&acc)[4][4]) {
  for (int k = 0; k < K4; k += 4) {
    float4 a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(A + i * lda + k);
#pragma unroll
    for (int q = 0; q < 4; ++q) b[q] = *reinterpret_cast<const float4*>(B + (k + q) * ldb);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float av[4] = {a[i].x, a[i].y, a[i].z, a[i].w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        acc[i][0] = fmaf(av[q], b[q].x, acc[i][0]);
        acc[i][1] = fmaf(av[q], b[q].y, acc[i][1]);
        acc[i][2] = fmaf(av[q], b[q].z, acc[i][2]);
        acc[i][3] = fmaf(av[q], b[q].w, acc[i][3]);
      }
    }
  }
}

// Outer-product accumulate for weight gradients:
// acc[i][j] += sum_r P[r*ldp + h0 + i] * U[r*ldu + k0 + j],  r in [0, rows).
__device__ __forceinline__ void outer_4x4(const float* __restrict__ P, int ldp, const float* __restrict__ U,
                                          int ldu, int rows, float (&acc)[4][4]) {
#pragma unroll 4
  for (int r = 0; r < rows; ++r) {
    const float4 p = *reinterpret_cast<const float4*>(P + r * ldp);
    const float4 u = *reinterpret_cast<const float4*>(U + r * ldu);
    const float pv[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[i][0] = fmaf(pv[i], u.x, acc[i][0]);
      acc[i][1] = fmaf(pv[i], u.y, acc[i][1]);
      acc[i][2] = fmaf(pv[i], u.z, acc[i][2]);
      acc[i][3] = fmaf(pv[i], u.w, acc[i][3]);
    }
  }
}

// 1 / x to ~1 ulp (MUFU.RCP): the Welford updates below only need 1 / count approximately, the exact division
// compiles to a dozen instructions with a slow path.
__device__ __forceinline__ float fast_rcp(float x) {
#ifdef CGNN_EMU
  return 1.0f / x;
#else
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#endif
}

// ---- Welford accumulators for BatchNorm statistics --------------------------------------
struct Welford {
  float mean, m2;
  __device__ __forceinline__ void init() { mean = 0.0f; m2 = 0.0f; }
  // `inv_n` = 1 / (number of samples including this one)
  __device__ __forceinline__ void push(float v, float inv_n) {
    float d = v - mean;
    mean = fmaf(d, inv_n, mean);
    m2 = fmaf(d, v - mean, m2);
  }
};

// Welford state of one thread's channel quad; deposit() leaves the record {count, mean[4], M2[4]} at rec[0..8]
struct QuadWelford {
  int cnt;
  Welford w[4];
  __device__ __forceinline__ void init() {
    cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j].init();
  }
  __device__ __forceinline__ void push(float4 v) {
    cnt += 1;
    const float inv = fast_rcp((float)cnt);
    w[0].push(v.x, inv); w[1].push(v.y, inv); w[2].push(v.z, inv); w[3].push(v.w, inv);
  }
  __device__ __forceinline__ void deposit(float* rec) const {
    rec[0] = (float)cnt;
#pragma unroll
    for (int j = 0; j < 4; ++j) { rec[1 + j] = w[j].mean; rec[5 + j] = w[j].m2; }
  }
};

// Chan's merge of the Welford record {nb, mb, qb} into {n, mean, m2}; empty records are skipped
__device__ __forceinline__ void welford_merge(double& n, double& mean, double& m2, double nb, double mb, double qb) {
  if (nb <= 0.0) return;
  const double nt = n + nb, delta = mb - mean;
  mean += delta * (nb / nt);
  m2 += qb + delta * delta * (n * nb / nt);
  n = nt;
}

// Shared by the layer kernels: merge per-warp Welford records held in shared memory into the
// CTA's record and write it (as doubles) to `out` = {count, mean[C], M2[C]} of this CTA.
//   s_cnt[kWarps], s_mean[kWarps][ldc], s_m2[kWarps][ldc]
__device__ __forceinline__ void cta_write_stats(const float* s_cnt, const float* s_mean, const float* s_m2,
                                                int ldc, int C, double* out) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
      welford_merge(n, mean, m2, (double)s_cnt[w], (double)s_mean[w * ldc + c], (double)s_m2[w * ldc + c]);
    out[1 + c] = mean;
    out[1 + C + c] = m2;
    if (c == 0) out[0] = n;
  }
}

// The same record from per-thread quad records (QuadWelford::deposit): thread th < nt owns channel quad th % Q of each
// pass of 4 Q channels and left pass P's record at rec[9 (P nt + th)].  Channel c is merged over th = q, q + Q, ...
// in that order; thread t of the nt threads writes channels t, t + nt, ...
__device__ __forceinline__ void cta_write_quad_stats(const float* rec, int nt, int Q, int C, int t, double* out) {
  for (int c = t; c < C; c += nt) {
    const float* r = rec + (size_t)(c / (4 * Q)) * nt * 9;
    const int q = (c >> 2) % Q, j = c & 3;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int th = q; th < nt; th += Q) welford_merge(n, mean, m2, (double)r[th * 9], (double)r[th * 9 + 1 + j], (double)r[th * 9 + 5 + j]);
    out[1 + c] = mean;
    out[1 + C + c] = m2;
    if (c == 0) out[0] = n;
  }
}

// Launchers shared across translation units -------------------------------------------------
// out[r*out_ld + c] = sum_g partials[g*stride + r*ld + c] for r < rows, c < cols (fp64 accumulation,
// fixed order): maps a zero-padded [rows, ld] partial onto a dense output (out_ld <= 0 -> cols).
int launch_reduce_partials(const float* partials, int G, int stride, int rows, int cols, int ld,
                           float* out, cudaStream_t stream, int out_ld = 0, double* out64 = nullptr);
// Several of them in one launch: q.add(...) per reduction, then q.flush() (returns the first error).
constexpr int kReduceMaxSegs = 4;
struct ReduceSeg { const float* partials; float* out; double* out64; int G, stride, rows, cols, ld, out_ld, first_block; };
struct ReduceBatch { ReduceSeg seg[kReduceMaxSegs]; int n; };
struct ReduceQueue {
  ReduceBatch b; int blocks; int status; cudaStream_t stream;
  explicit ReduceQueue(cudaStream_t s) : blocks(0), status(0), stream(s) { b.n = 0; }
  // out64 (optional): the same sums unrounded, dense [rows, cols]
  void add(const float* partials, int G, int stride, int rows, int cols, int ld, float* out, int out_ld = 0, double* out64 = nullptr);
  int flush();
};
int launch_stats_merge(const double* parts, int parts_n, int C, double* stats, cudaStream_t stream);

// Process-wide switch (cgnn_set_option): 1 = eligible shapes run on the tcgen05 kernels (default),
// 0 = everything on the generic SIMT kernels (used to cross-check the two on the device).
bool tensor_cores_enabled();

}  // namespace cgnn
