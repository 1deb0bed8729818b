// norm.cu - K3: BatchNorm1d bookkeeping around the layer kernels (reference models.py:191-193,
// 208, 260 -> nn.BatchNorm1d defaults: eps 1e-5, momentum 0.1, affine, running stats) and the
// standalone BatchNorm-backward reduction used for the top layer.
#include "tile.cuh"
#include "rowtile.cuh"

namespace cgnn {

__global__ void __launch_bounds__(256) k_bn_finalize(const double* __restrict__ stats, const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, int C, float eps, float momentum,
                                                     float* running_mean, float* running_var,
                                                     long long* num_batches_tracked, float* __restrict__ scale,
                                                     float* __restrict__ shift, float* __restrict__ mean_out,
                                                     float* __restrict__ rstd_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && num_batches_tracked) num_batches_tracked[0] += 1;
  if (c >= C) return;
  const double n = stats[0];
  const double mean = stats[1 + c];
  const double var_b = n > 0.0 ? stats[1 + C + c] / n : 0.0;            // biased: normalisation
  const double var_u = n > 1.0 ? stats[1 + C + c] / (n - 1.0) : var_b;  // unbiased: running estimate
  const float rstd = (float)(1.0 / sqrt(var_b + (double)eps));
  const float g = gamma ? gamma[c] : 1.0f, b = beta ? beta[c] : 0.0f;
  const float sc = g * rstd;
  scale[c] = sc;
  shift[c] = b - (float)mean * sc;
  mean_out[c] = (float)mean;
  rstd_out[c] = rstd;
  if (running_mean) running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mean;
  if (running_var) running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)var_u;
}

__global__ void __launch_bounds__(256) k_bn_eval_affine(const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        const float* __restrict__ running_mean,
                                                        const float* __restrict__ running_var, int C, float eps,
                                                        float* __restrict__ scale, float* __restrict__ shift,
                                                        float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float rstd = (float)(1.0 / sqrt((double)running_var[c] + (double)eps));
  const float g = gamma ? gamma[c] : 1.0f, b = beta ? beta[c] : 0.0f;
  const float sc = g * rstd;
  scale[c] = sc;
  shift[c] = b - running_mean[c] * sc;
  if (mean_out) mean_out[c] = running_mean[c];
  if (rstd_out) rstd_out[c] = rstd;
}

struct BnSumsArgs {
  const float* z; Act act; const float* mean; const float* rstd;
  const float* du; const float* demb; const long long* ptr; long long B;
  int C, C4;
  float* partials;  // [grid][2*C4]
};

// s1 = sum dy, s2 = sum dy * xhat with dy = d act(z) * du.  Warp per row, lanes over channels.
template <int CC>
__global__ void __launch_bounds__(kThreads) k_bn_bwd_sums(BnSumsArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  const int C = p.C, C4 = p.C4;
  float* s_c = sm;               // [4][C4] scale, shift, mean, rstd
  float* s_red = sm + 4 * C4;    // [kWarps][2*C4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool affine = p.act.scale != nullptr;
  stage_affine(p.act, C, C4, s_c, s_c + C4);
  for (int c = tid; c < C4; c += kThreads) {
    s_c[2 * C4 + c] = c < C ? p.mean[c] : 0.0f;
    s_c[3 * C4 + c] = c < C ? p.rstd[c] : 0.0f;
  }
  __syncthreads();
  float s1[CC], s2[CC];
#pragma unroll
  for (int j = 0; j < CC; ++j) { s1[j] = 0.0f; s2[j] = 0.0f; }
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    const long long nb = p.ptr[g];
    const int n = (int)(p.ptr[g + 1] - nb);
    const float inv_n = pool_bwd_scale(n);
    for (int i = warp; i < n; i += kWarps) {
      const long long grow = nb + i;
      const uint32_t rh = p.act.drop ? drop_row_hash(p.act, p.act.row_base + grow) : 0u;
#pragma unroll
      for (int j = 0; j < CC; ++j) {
        const int ch = lane + 32 * j;
        if (ch < C) {
          const float t = p.z[grow * C + ch];
          const float up = p.du ? p.du[grow * C + ch] : p.demb[g * C + ch] * inv_n;
          const float dy = act_bwd(p.act, affine, t, s_c[ch], s_c[C4 + ch], rh, ch, up);
          bn_sums_add(s1[j], s2[j], dy, t, s_c[2 * C4 + ch], s_c[3 * C4 + ch]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < CC; ++j) {
    const int ch = lane + 32 * j;
    if (ch < C4) { s_red[warp * 2 * C4 + ch] = s1[j]; s_red[warp * 2 * C4 + C4 + ch] = s2[j]; }
  }
  __syncthreads();
  float* part = p.partials + (size_t)blockIdx.x * 2 * C4;
  for (int c = tid; c < 2 * C4; c += kThreads) part[c] = warp_rows_sum(s_red, 2 * C4, c);
}

#ifndef CGNN_EMU
// Channel-quad edition of k_bn_bwd_sums (C = 32 / 64 / 128 / 256, 16-byte aligned rows).
template <int Q>
__global__ void __launch_bounds__(kThreads, 2) k_bn_bwd_sums_quad(BnSumsArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  __shared__ float4 s_red[2 * kThreads];
  constexpr int RS = kThreads / Q;
  const int tid = threadIdx.x, q = tid % Q, r = tid / Q;
  const int C = p.C;
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act, 4 * q, C);
  const rt::RowKey rk = rt::row_key(p.act);
  float mean[4], rstd[4];
  rt::bn_stats_quad(mean, rstd, p.mean, p.rstd, 4 * q, 4 * Q, true);
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
  long long nb_next = 0, ne_next = 0;
  if ((long long)blockIdx.x < p.B) { nb_next = p.ptr[blockIdx.x]; ne_next = p.ptr[blockIdx.x + 1]; }
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    const long long nb = nb_next;                  // row range loaded one subject ahead
    const int n = (int)(ne_next - nb);
    if (g + gridDim.x < p.B) { nb_next = p.ptr[g + gridDim.x]; ne_next = p.ptr[g + gridDim.x + 1]; }
    float4 pooled = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!p.du) pooled = rt::pooled_quad<true>(p.demb, g, C, 4 * q, n);
    for (int i = r; i < n; i += 4 * RS) {
      float4 zv[4], uv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        uv[u] = pooled;
        if (i + u * RS < n) {
          zv[u] = rt::ld_quad<true>(p.z, nb + i + u * RS, C, 4 * q);
          if (p.du) uv[u] = rt::ld_quad<true>(p.du, nb + i + u * RS, C, 4 * q);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * RS < n) {
          const float4 dy = rt::act_bwd4(p.act, cq, zv[u], uv[u], rk, (uint32_t)(nb + i + u * RS));
          const float tv[4] = {zv[u].x, zv[u].y, zv[u].z, zv[u].w}, dv[4] = {dy.x, dy.y, dy.z, dy.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) bn_sums_add(s1[j], s2[j], dv[j], tv[j], mean[j], rstd[j]);
        }
    }
  }
  s_red[tid] = make_float4(s1[0], s1[1], s1[2], s1[3]);
  s_red[kThreads + tid] = make_float4(s2[0], s2[1], s2[2], s2[3]);
  __syncthreads();
  float* part = p.partials + (size_t)blockIdx.x * 2 * p.C4;
  for (int idx = tid; idx < 2 * C; idx += kThreads) {
    const int which = idx / C, c = idx - which * C;
    part[which * p.C4 + c] = quad_sum(reinterpret_cast<const float*>(s_red), 4, 4 * kThreads * which, kThreads, Q, c >> 2, c & 3);
  }
}
#endif


// ---------------------------------------------------------------------------------------------------------------------
// SyncBN exchange over peer memory (NVLink / NVSwitch): ONE kernel writes this rank's record straight into every peer's
// symmetric buffer, raises a flag there, waits for the peers' flags in its own buffer and then merges the records in rank
// order - identical on every rank.  It replaces an NCCL all-gather (or all-reduce) of a few hundred bytes plus the merge
// kernel behind it: three of these per training step and model sit on the critical path between two layer kernels.
//   symmetric buffer of a rank (doubles): [slots][world][rec_cap] records, then uint32 flags [slots][world]
//   flag (slot, r) in rank q's buffer = the sequence number of the last record rank r delivered to q in that slot
// A slot is written again only two uses later (the caller alternates two physical slots per logical one), by which time
// every peer has consumed it: a rank can only be one exchange ahead of the slowest one.
#ifndef CGNN_EMU
struct PeerArgs {
  const unsigned long long* bufs;   // [world] device pointers to the ranks' symmetric buffers
  int rank, world, slot, slots, rec_cap, n, mode, C;
  unsigned int seq;
  const double* mine; double* out; int* error;
};
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__global__ void __launch_bounds__(256) k_peer_exchange(PeerArgs p) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t rec0 = ((size_t)p.slot * p.world) * p.rec_cap;
  const size_t flags_off = (size_t)p.slots * p.world * p.rec_cap;      // in doubles
  for (int t = tid; t < p.n; t += blockDim.x) {
    const double v = p.mine[t];
    for (int r = 0; r < p.world; ++r) reinterpret_cast<double*>(p.bufs[r])[rec0 + (size_t)p.rank * p.rec_cap + t] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (tid < p.world) {
    unsigned int* peer_flags = reinterpret_cast<unsigned int*>(reinterpret_cast<double*>(p.bufs[tid]) + flags_off);
    st_release_sys(peer_flags + (size_t)p.slot * p.world + p.rank, p.seq);
    const unsigned int* my_flags = reinterpret_cast<const unsigned int*>(reinterpret_cast<const double*>(p.bufs[p.rank]) + flags_off);
    const long long t0 = clock64();
    while (ld_acquire_sys(my_flags + (size_t)p.slot * p.world + tid) != p.seq) {
      if (clock64() - t0 > 8000000000ll) { atomicExch(p.error, 1); break; }     // ~4 s: a peer died; do not hang the GPU
    }
  }
  __syncthreads();
  const double* recs = reinterpret_cast<const double*>(p.bufs[p.rank]) + rec0;
  if (p.mode == 1) {                     // plain sum in rank order
    for (int t = tid; t < p.n; t += blockDim.x) {
      double s = 0.0;
      for (int r = 0; r < p.world; ++r) s += recs[(size_t)r * p.rec_cap + t];
      p.out[t] = s;
    }
    return;
  }
  // BatchNorm statistics {count, mean[C], M2[C]}: the exact merge of k_stats_merge, one warp per channel
  const int C = p.C;
  for (int c = warp; c < C; c += (int)(blockDim.x >> 5)) {
    double n = 0.0, s = 0.0;
    for (int r = lane; r < p.world; r += 32) {
      const double nr = recs[(size_t)r * p.rec_cap];
      n += nr;
      s += nr * recs[(size_t)r * p.rec_cap + 1 + c];
    }
    n = warp_sum(n);
    s = warp_sum(s);
    const double mean = n > 0.0 ? s / n : 0.0;
    double q = 0.0;
    for (int r = lane; r < p.world; r += 32) {
      const double nr = recs[(size_t)r * p.rec_cap];
      if (nr > 0.0) {
        const double d = recs[(size_t)r * p.rec_cap + 1 + c] - mean;
        q += recs[(size_t)r * p.rec_cap + 1 + C + c] + nr * d * d;
      }
    }
    q = warp_sum(q);
    if (lane == 0) {
      p.out[1 + c] = mean;
      p.out[1 + C + c] = q;
      if (c == 0) p.out[0] = n;
    }
  }
}
#endif

}  // namespace cgnn

using namespace cgnn;

extern "C" {

int cgnn_bn_finalize(const double* stats, const float* gamma, const float* beta, int32_t C, float eps,
                     float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                     float* scale, float* shift, float* mean, float* rstd, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!stats || C <= 0 || !scale || !shift || !mean || !rstd) return CGNN_ERR_INVALID_ARG;
  auto kfn = k_bn_finalize;
  CGNN_LAUNCH(kfn, (C + 255) / 256, 256, 0, stream, stats, gamma, beta, (int)C, eps, momentum, running_mean,
              running_var, (long long*)num_batches_tracked, scale, shift, mean, rstd);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                        int32_t C, float eps, float* scale, float* shift, float* mean, float* rstd,
                        cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!running_mean || !running_var || C <= 0 || !scale || !shift) return CGNN_ERR_INVALID_ARG;
  auto kfn = k_bn_eval_affine;
  CGNN_LAUNCH(kfn, (C + 255) / 256, 256, 0, stream, gamma, beta, running_mean, running_var, (int)C, eps, scale,
              shift, mean, rstd);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_bn_bwd_sums(const float* z, const cgnn_act_t* act, const float* mean, const float* rstd, const float* du,
                     const float* demb, const int64_t* ptr, int64_t num_graphs, int64_t rows, int32_t C,
                     float* sums, double* sums64, void* workspace, size_t workspace_bytes, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!sums || C <= 0 || num_graphs < 0 || rows < 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0 || rows == 0) {
    cudaMemsetAsync(sums, 0, (size_t)2 * C * sizeof(float), stream);
    if (sums64) cudaMemsetAsync(sums64, 0, (size_t)2 * C * sizeof(double), stream);
    return CGNN_OK;
  }
  if ((du == nullptr) == (demb == nullptr)) return CGNN_ERR_INVALID_ARG;
  if (!z || !mean || !rstd || !ptr || !workspace) return CGNN_ERR_INVALID_ARG;
  const DeviceInfo dev = device_info();
  BnSumsArgs a;
  a.z = z; a.act = make_act(act); a.mean = mean; a.rstd = rstd; a.du = du; a.demb = demb;
  a.ptr = (const long long*)ptr; a.B = num_graphs; a.C = C; a.C4 = round_up(C, 4);
  if (a.C4 > 256) return CGNN_ERR_TILE_TOO_LARGE;
  const size_t smem = (size_t)(4 * a.C4 + kWarps * 2 * a.C4) * sizeof(float);
  int grid = persistent_grid(num_graphs, smem, dev, kThreads);
  const size_t rec = (size_t)2 * a.C4 * sizeof(float);
  if (workspace_bytes < rec) return CGNN_ERR_WORKSPACE;
  if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
  a.partials = (float*)workspace;
#ifndef CGNN_EMU
  if ((C == 32 || C == 64 || C == 128 || C == 256) && (((uintptr_t)z) & 15u) == 0 && (!du || (((uintptr_t)du) & 15u) == 0) &&
      (!demb || (((uintptr_t)demb) & 15u) == 0)) {
    long long g2 = 2LL * dev.sm_count;
    if (g2 > num_graphs) g2 = num_graphs;
    if ((size_t)g2 * rec > workspace_bytes) g2 = (long long)(workspace_bytes / rec);
    if (C == 32) { auto kfn = k_bn_bwd_sums_quad<8>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else if (C == 64) { auto kfn = k_bn_bwd_sums_quad<16>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else if (C == 128) { auto kfn = k_bn_bwd_sums_quad<32>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else { auto kfn = k_bn_bwd_sums_quad<64>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    CGNN_CHECK_LAUNCH();
    return launch_reduce_partials(a.partials, (int)g2, 2 * a.C4, 2, C, a.C4, sums, stream, 0, sums64);
  }
#endif
  const int cc = pick_hc(a.C4);
#define CGNN_BN_SUMS(CC_)                                                  \
  {                                                                        \
    auto kfn = k_bn_bwd_sums<CC_>;                                         \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);                     \
  }
  if (cc == 1) CGNN_BN_SUMS(1) else if (cc == 2) CGNN_BN_SUMS(2) else if (cc == 4) CGNN_BN_SUMS(4) else CGNN_BN_SUMS(8)
#undef CGNN_BN_SUMS
  CGNN_CHECK_LAUNCH();
  return launch_reduce_partials(a.partials, grid, 2 * a.C4, 2, C, a.C4, sums, stream, 0, sums64);
}

int cgnn_peer_exchange(const uint64_t* peer_buffers, int32_t rank, int32_t world, int32_t slot, int32_t slots, int32_t rec_cap,
                       uint32_t seq, int32_t mode, const double* mine, int32_t n, int32_t C, double* out, int32_t* error,
                       cgnn_stream_t stream_) {
#ifdef CGNN_EMU
  (void)peer_buffers; (void)rank; (void)world; (void)slot; (void)slots; (void)rec_cap; (void)seq; (void)mode; (void)mine; (void)n;
  (void)C; (void)out; (void)error; (void)stream_;
  return CGNN_ERR_UNSUPPORTED;
#else
  if (!peer_buffers || !mine || !out || !error || world < 1 || world > 64 || rank < 0 || rank >= world || slot < 0 || slot >= slots ||
      n < 1 || n > rec_cap || seq == 0 || (mode != 0 && mode != 1))
    return CGNN_ERR_INVALID_ARG;
  if (mode == 0 && n != 1 + 2 * C) return CGNN_ERR_INVALID_ARG;
  PeerArgs a;
  a.bufs = (const unsigned long long*)peer_buffers; a.rank = rank; a.world = world; a.slot = slot; a.slots = slots;
  a.rec_cap = rec_cap; a.n = n; a.mode = mode; a.C = C; a.seq = seq; a.mine = mine; a.out = out; a.error = error;
  auto kfn = k_peer_exchange;
  CGNN_LAUNCH(kfn, 1, 256, 0, (cudaStream_t)stream_, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
#endif
}

}  // extern "C"
