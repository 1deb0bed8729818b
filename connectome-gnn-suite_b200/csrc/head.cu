// head.cu - K4 / K5: mean-pool readout, MLP head, cross-entropy and their backward passes.
//
// Reference: models.py:57-59 (_graph_mean_pool -> _scatter_mean 40-47), models.py:196-201
// (Linear - ReLU - Dropout - Linear), train.py:39,49,64-66 (CrossEntropyLoss, argmax accuracy).
// These are O(B*H) - negligible next to the layer kernels - so they are written for
// clarity and determinism rather than peak throughput.
#include "tile.cuh"
#include "rowtile.cuh"

namespace cgnn {

constexpr int kHeadMaxC = 512;   // pooled width
constexpr int kHeadMaxM = 256;   // hidden width of the head
constexpr int kHeadMaxK = 64;    // classes
constexpr uint32_t kHeadSite = 0x48454144u;

// ---- mean pool ---------------------------------------------------------------------------
struct PoolArgs {
  const float* t; Act act; const long long* ptr; long long B; int C, C4; float* emb;
};

template <int CC>
__global__ void __launch_bounds__(kThreads) k_pool_fwd(PoolArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  const int C = p.C, C4 = p.C4;
  float* s_c = sm;             // [2][C4]
  float* s_red = sm + 2 * C4;  // [kWarps][C4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool affine = p.act.scale != nullptr;
  stage_affine(p.act, C, C4, s_c, s_c + C4);
  __syncthreads();
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    const long long nb = p.ptr[g];
    const int n = (int)(p.ptr[g + 1] - nb);
    float acc[CC];
#pragma unroll
    for (int j = 0; j < CC; ++j) acc[j] = 0.0f;
    for (int i = warp; i < n; i += kWarps) {
      const long long grow = nb + i;
      const uint32_t rh = p.act.drop ? drop_row_hash(p.act, p.act.row_base + grow) : 0u;
#pragma unroll
      for (int j = 0; j < CC; ++j) {
        const int ch = lane + 32 * j;
        if (ch < C) acc[j] += act_fwd(p.act, affine, p.t[grow * C + ch], s_c[ch], s_c[C4 + ch], rh, ch);
      }
    }
#pragma unroll
    for (int j = 0; j < CC; ++j) {
      const int ch = lane + 32 * j;
      if (ch < C4) s_red[warp * C4 + ch] = acc[j];
    }
    __syncthreads();
    const float denom = (float)n + 1e-8f;
    for (int c = tid; c < C; c += kThreads) p.emb[g * C + c] = warp_rows_sum(s_red, C4, c) / denom;
    __syncthreads();
  }
}

#ifndef CGNN_EMU
// Channel-quad edition (C = 32 / 64 / 128 / 256, 16-byte aligned rows): thread = one channel quad, four
// independent 16-byte loads in flight per thread, two CTAs of 512 threads per SM.
template <int Q>
__global__ void __launch_bounds__(kThreads, 2) k_pool_fwd_quad(PoolArgs p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
  __shared__ float4 s_red[kThreads];
  constexpr int RS = kThreads / Q;
  const int tid = threadIdx.x, q = tid % Q, r = tid / Q;
  const int C = p.C;
  rt::ChanQuad cq;
  rt::chan_quad_init(cq, p.act, 4 * q, C);
  const rt::RowKey rk = rt::row_key(p.act);
  long long nb_next = 0, ne_next = 0;
  if ((long long)blockIdx.x < p.B) { nb_next = p.ptr[blockIdx.x]; ne_next = p.ptr[blockIdx.x + 1]; }
  for (long long g = blockIdx.x; g < p.B; g += gridDim.x) {
    const long long nb = nb_next;                  // row range loaded one subject ahead
    const int n = (int)(ne_next - nb);
    if (g + gridDim.x < p.B) { nb_next = p.ptr[g + gridDim.x]; ne_next = p.ptr[g + gridDim.x + 1]; }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = r; i < n; i += 4 * RS) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * RS < n) v[u] = rt::ld_quad<true>(p.t, nb + i + u * RS, C, 4 * q);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * RS < n) {
          const float4 y = rt::act_fwd4(p.act, cq, v[u], rk, (uint32_t)(nb + i + u * RS));
          acc.x += y.x; acc.y += y.y; acc.z += y.z; acc.w += y.w;
        }
    }
    s_red[tid] = acc;
    __syncthreads();
    if (tid < C) p.emb[g * C + tid] = quad_sum(reinterpret_cast<const float*>(s_red), 4, 0, kThreads, Q, tid >> 2, tid & 3) / ((float)n + 1e-8f);
    __syncthreads();
  }
}
#endif

// ---- MLP head forward: one warp per graph -------------------------------------------------
struct HeadArgs {
  const float* emb; const float* W0; const float* b0; const float* W1; const float* b1;
  long long B; int C, M, K; Act drop;  // drop: dropout after the hidden ReLU (row id = graph id)
  float* hidden; float* logits;
};

__global__ void __launch_bounds__(kThreads) k_head_fwd(HeadArgs p) {
  act_salt(p.drop);   // device-side dropout salt (CUDA-graph replays)
  __shared__ float s_hid[kWarps][kHeadMaxM];
  __shared__ float s_emb[kWarps][kHeadMaxC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long g = (long long)blockIdx.x * kWarps + warp;
  if (g >= p.B) return;
  const int C = p.C, M = p.M, K = p.K;
  for (int c = lane; c < C; c += 32) s_emb[warp][c] = p.emb[g * C + c];
  __syncwarp();
  const uint32_t rh = p.drop.drop ? drop_row_hash(p.drop, p.drop.row_base + g) : 0u;
  for (int m = 0; m < M; ++m) {
    float part = 0.0f;
    for (int c = lane; c < C; c += 32) part = fmaf(p.W0[m * C + c], s_emb[warp][c], part);
    float h = warp_sum(part) + p.b0[m];
    h = fmaxf(h, 0.0f);
    if (p.drop.drop) h = drop_keep(p.drop, rh, m) ? h * p.drop.keep_scale : 0.0f;
    if (lane == 0) { s_hid[warp][m] = h; p.hidden[g * M + m] = h; }
  }
  __syncwarp();
  for (int k = 0; k < K; ++k) {
    float part = 0.0f;
    for (int m = lane; m < M; m += 32) part = fmaf(p.W1[k * M + m], s_hid[warp][m], part);
    const float v = warp_sum(part) + p.b1[k];
    if (lane == 0) p.logits[g * K + k] = v;
  }
}

// Small heads (C <= 128, M <= 64, K <= 8 - the reference's 64 -> 32 -> 2): the weights are staged once per CTA (W0
// transposed, so that lane = hidden unit reads consecutive words), every warp then walks graphs: the pooled row is
// broadcast from shared memory, 64 FMAs per lane and hidden unit, no shuffle in the first layer.
constexpr int kHeadSmallC = 128, kHeadSmallM = 64, kHeadSmallK = 8, kHeadSmallWarps = 8;
__global__ void __launch_bounds__(32 * kHeadSmallWarps) k_head_fwd_small(HeadArgs p) {
  act_salt(p.drop);   // device-side dropout salt (CUDA-graph replays)
  CGNN_SMEM_DECL;
  const int C = p.C, M = p.M, K = p.K, MP = M + 1;
  float* s_w0t = reinterpret_cast<float*>(cgnn_smem);       // [C][M + 1]
  float* s_w1 = s_w0t + C * MP;                             // [K][M]
  float* s_b0 = s_w1 + K * M;                               // [M]
  float* s_b1 = s_b0 + M;                                   // [K]
  float* s_emb = s_b1 + K;                                  // [warps][C]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < M * C; i += blockDim.x) { const int m = i / C, c = i - m * C; s_w0t[c * MP + m] = p.W0[i]; }
  for (int i = tid; i < K * M; i += blockDim.x) s_w1[i] = p.W1[i];
  for (int i = tid; i < M; i += blockDim.x) s_b0[i] = p.b0[i];
  for (int i = tid; i < K; i += blockDim.x) s_b1[i] = p.b1[i];
  __syncthreads();
  float* my_emb = s_emb + warp * C;
  const int m0 = lane, m1 = lane + 32;
  for (long long g = (long long)blockIdx.x * kHeadSmallWarps + warp; g < p.B; g += (long long)gridDim.x * kHeadSmallWarps) {
    for (int c = lane; c < C; c += 32) my_emb[c] = p.emb[g * C + c];
    __syncwarp();
    float h0 = 0.0f, h1 = 0.0f;
    if (m1 < M) {
      for (int c = 0; c < C; ++c) { const float e = my_emb[c]; h0 = fmaf(s_w0t[c * MP + m0], e, h0); h1 = fmaf(s_w0t[c * MP + m1], e, h1); }
    } else if (m0 < M) {
      for (int c = 0; c < C; ++c) h0 = fmaf(s_w0t[c * MP + m0], my_emb[c], h0);
    }
    const uint32_t rh = p.drop.drop ? drop_row_hash(p.drop, p.drop.row_base + g) : 0u;
    if (m0 < M) {
      h0 = fmaxf(h0 + s_b0[m0], 0.0f);
      if (p.drop.drop) h0 = drop_keep(p.drop, rh, m0) ? h0 * p.drop.keep_scale : 0.0f;
      p.hidden[g * M + m0] = h0;
    } else h0 = 0.0f;
    if (m1 < M) {
      h1 = fmaxf(h1 + s_b0[m1], 0.0f);
      if (p.drop.drop) h1 = drop_keep(p.drop, rh, m1) ? h1 * p.drop.keep_scale : 0.0f;
      p.hidden[g * M + m1] = h1;
    } else h1 = 0.0f;
    for (int k = 0; k < K; ++k) {
      float part = m0 < M ? s_w1[k * M + m0] * h0 : 0.0f;
      if (m1 < M) part = fmaf(s_w1[k * M + m1], h1, part);
      const float v = warp_sum(part) + s_b1[k];
      if (lane == 0) p.logits[g * K + k] = v;
    }
    __syncwarp();       // my_emb is rewritten for the next graph
  }
}

// ---- cross entropy --------------------------------------------------------------------------
// One CTA (the loss is one number; fixed summation order): 1024 threads, a warp-shuffle tree per warp, then warp 0 over
// the 32 warp sums - doubles, the same order every launch.
__global__ void __launch_bounds__(1024) k_ce_fwd(const float* __restrict__ logits, const long long* __restrict__ labels,
                                                 long long B, int K, float inv_count, float* __restrict__ nll,
                                                 float* __restrict__ loss, long long* __restrict__ correct) {
  __shared__ double s_loss[32];
  __shared__ long long s_corr[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double acc = 0.0;
  long long corr = 0;
  for (long long g = tid; g < B; g += blockDim.x) {
    const float* l = logits + g * K;
    float mx = l[0]; int arg = 0;
    for (int k = 1; k < K; ++k) if (l[k] > mx) { mx = l[k]; arg = k; }
    float se = 0.0f;
    for (int k = 0; k < K; ++k) se += expf(l[k] - mx);
    const float lse = mx + logf(se);
    long long y = labels[g];
    const bool ok = y >= 0 && y < K;
    // a label outside [0, K) is a caller error (torch's CrossEntropyLoss raises): poison the loss instead of
    // silently dropping the graph from the numerator
    const float v = ok ? lse - l[y] : __int_as_float(0x7fc00000);
    if (nll) nll[g] = v;
    acc += (double)v;
    corr += (ok && arg == (int)y) ? 1 : 0;
  }
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_down_sync(kFull, acc, o);
    corr += __shfl_down_sync(kFull, corr, o);
  }
  if (lane == 0) { s_loss[warp] = acc; s_corr[warp] = corr; }
  __syncthreads();
  if (warp == 0) {
    const int nw = (int)(blockDim.x >> 5);
    double s = lane < nw ? s_loss[lane] : 0.0;
    long long c = lane < nw ? s_corr[lane] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_down_sync(kFull, s, o);
      c += __shfl_down_sync(kFull, c, o);
    }
    if (lane == 0) {
      if (loss) loss[0] = (float)(s * (double)inv_count);
      if (correct) correct[0] = c;
    }
  }
}

__global__ void __launch_bounds__(256) k_ce_bwd(const float* __restrict__ logits, const long long* __restrict__ labels,
                                                long long B, int K, float inv_count, const float* __restrict__ gout,
                                                float* __restrict__ dlogits) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= B) return;
  const float* l = logits + g * K;
  float mx = l[0];
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, l[k]);
  float se = 0.0f;
  for (int k = 0; k < K; ++k) se += expf(l[k] - mx);
  const float scale = inv_count * (gout ? gout[0] : 1.0f);
  const long long y = labels[g];
  const bool ok = y >= 0 && y < K;
  for (int k = 0; k < K; ++k) {
    const float sm = expf(l[k] - mx) / se;
    dlogits[g * K + k] = ok ? (sm - (k == (int)y ? 1.0f : 0.0f)) * scale : 0.0f;
  }
}

// ---- MLP head backward ------------------------------------------------------------------------
struct HeadBwdArgs {
  const float* emb; const float* hidden; const float* dlogits; const float* W0; const float* W1;
  long long B; int C, M, K; float keep_scale;
  float* demb; float* partials; int part_stride, o_dw0, o_db0, o_dw1, o_db1;
  int o_acc, o_dhp, o_emb, o_dl, o_hid;  // smem float offsets
};

__global__ void __launch_bounds__(kThreads) k_head_bwd(HeadBwdArgs p) {
  CGNN_SMEM_DECL;
  float* sm = reinterpret_cast<float*>(cgnn_smem);
  const int C = p.C, M = p.M, K = p.K;
  float* s_acc = sm + p.o_acc;  // [part_stride] running sums of this CTA
  float* s_dhp = sm + p.o_dhp;  // [kWarps][M]  gradient w.r.t. the hidden pre-activation
  float* s_emb = sm + p.o_emb;  // [kWarps][C]
  float* s_dl = sm + p.o_dl;    // [kWarps][K]
  float* s_hid = sm + p.o_hid;  // [kWarps][M]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < p.part_stride; i += kThreads) s_acc[i] = 0.0f;
  __syncthreads();
  const long long groups = (p.B + kWarps - 1) / kWarps;
  for (long long grp = blockIdx.x; grp < groups; grp += gridDim.x) {
    const long long g = grp * kWarps + warp;
    const bool live = g < p.B;
    for (int k = lane; k < K; k += 32) s_dl[warp * K + k] = live ? p.dlogits[g * K + k] : 0.0f;
    for (int m = lane; m < M; m += 32) s_hid[warp * M + m] = live ? p.hidden[g * M + m] : 0.0f;
    for (int c = lane; c < C; c += 32) s_emb[warp * C + c] = live ? p.emb[g * C + c] : 0.0f;
    __syncwarp();
    for (int m = lane; m < M; m += 32) {
      float d = 0.0f;
      for (int k = 0; k < K; ++k) d = fmaf(s_dl[warp * K + k], p.W1[k * M + m], d);
      s_dhp[warp * M + m] = s_hid[warp * M + m] > 0.0f ? d * p.keep_scale : 0.0f;
    }
    __syncwarp();
    if (live) {
      for (int c = lane; c < C; c += 32) {
        float d = 0.0f;
        for (int m = 0; m < M; ++m) d = fmaf(s_dhp[warp * M + m], p.W0[m * C + c], d);
        p.demb[g * C + c] = d;
      }
    }
    __syncthreads();
    for (int idx = tid; idx < M * C; idx += kThreads) {
      const int m = idx / C, c = idx - m * C;
      float s = 0.0f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s = fmaf(s_dhp[w * M + m], s_emb[w * C + c], s);
      s_acc[p.o_dw0 + idx] += s;
    }
    for (int m = tid; m < M; m += kThreads) {
      float s = 0.0f;
      for (int w = 0; w < kWarps; ++w) s += s_dhp[w * M + m];
      s_acc[p.o_db0 + m] += s;
    }
    for (int idx = tid; idx < K * M; idx += kThreads) {
      const int k = idx / M, m = idx - k * M;
      float s = 0.0f;
      for (int w = 0; w < kWarps; ++w) s = fmaf(s_dl[w * K + k], s_hid[w * M + m], s);
      s_acc[p.o_dw1 + idx] += s;
    }
    for (int k = tid; k < K; k += kThreads) {
      float s = 0.0f;
      for (int w = 0; w < kWarps; ++w) s += s_dl[w * K + k];
      s_acc[p.o_db1 + k] += s;
    }
    __syncthreads();
  }
  float* part = p.partials + (size_t)blockIdx.x * p.part_stride;
  for (int i = tid; i < p.part_stride; i += kThreads) part[i] = s_acc[i];
}

}  // namespace cgnn

using namespace cgnn;

extern "C" {

int cgnn_pool_fwd(const float* t_in, const cgnn_act_t* act, const int64_t* ptr, int64_t num_graphs, int64_t rows,
                  int32_t C, float* emb, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || rows < 0 || C <= 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) return CGNN_OK;
  if (!ptr || !emb || (rows > 0 && !t_in)) return CGNN_ERR_INVALID_ARG;
  const DeviceInfo dev = device_info();
  PoolArgs a;
  a.t = t_in; a.act = make_act(act); a.ptr = (const long long*)ptr; a.B = num_graphs; a.C = C; a.C4 = round_up(C, 4);
  a.emb = emb;
  if (a.C4 > 256) return CGNN_ERR_TILE_TOO_LARGE;
#ifndef CGNN_EMU
  if ((C == 32 || C == 64 || C == 128 || C == 256) && (((uintptr_t)t_in) & 15u) == 0) {
    long long g2 = 2LL * dev.sm_count;
    if (g2 > num_graphs) g2 = num_graphs;
    if (C == 32) { auto kfn = k_pool_fwd_quad<8>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else if (C == 64) { auto kfn = k_pool_fwd_quad<16>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else if (C == 128) { auto kfn = k_pool_fwd_quad<32>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    else { auto kfn = k_pool_fwd_quad<64>; CGNN_LAUNCH(kfn, (unsigned)g2, kThreads, 0, stream, a); }
    CGNN_CHECK_LAUNCH();
    return CGNN_OK;
  }
#endif
  const size_t smem = (size_t)(2 * a.C4 + kWarps * a.C4) * sizeof(float);
  const int grid = persistent_grid(num_graphs, smem, dev, kThreads);
  const int cc = pick_hc(a.C4);
#define CGNN_POOL(CC_)                                       \
  {                                                          \
    auto kfn = k_pool_fwd<CC_>;                              \
    CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);       \
  }
  if (cc == 1) CGNN_POOL(1) else if (cc == 2) CGNN_POOL(2) else if (cc == 4) CGNN_POOL(4) else CGNN_POOL(8)
#undef CGNN_POOL
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_head_fwd(const float* emb, const float* W0, const float* b0, const float* W1, const float* b1,
                  int64_t num_graphs, int32_t C, int32_t M, int32_t K, float p_drop, uint64_t seed,
                  int64_t graph_base, const uint32_t* salt, float* hidden, float* logits, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || C <= 0 || M <= 0 || K <= 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) return CGNN_OK;
  if (!emb || !W0 || !b0 || !W1 || !b1 || !hidden || !logits) return CGNN_ERR_INVALID_ARG;
  if (C > kHeadMaxC || M > kHeadMaxM || K > kHeadMaxK) return CGNN_ERR_TILE_TOO_LARGE;
  HeadArgs a;
  a.emb = emb; a.W0 = W0; a.b0 = b0; a.W1 = W1; a.b1 = b1; a.B = num_graphs; a.C = C; a.M = M; a.K = K;
  cgnn_act_t d{};
  d.p_drop = p_drop; d.seed = seed; d.site = kHeadSite; d.row_base = graph_base; d.salt = salt;
  a.drop = make_act(&d);
  a.hidden = hidden; a.logits = logits;
  if (C <= kHeadSmallC && M <= kHeadSmallM && K <= kHeadSmallK) {
    const size_t smem = (size_t)(C * (M + 1) + K * M + M + K + kHeadSmallWarps * C) * sizeof(float);
    long long grid = (num_graphs + kHeadSmallWarps - 1) / kHeadSmallWarps;
    const long long cap = 4ll * device_info().sm_count;        // persistent: the weights are staged once per CTA
    if (grid > cap) grid = cap;
    auto kfs = k_head_fwd_small;
#ifndef CGNN_EMU
    if (smem > 48 * 1024) cudaFuncSetAttribute(kfs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
    CGNN_LAUNCH(kfs, (unsigned)grid, 32 * kHeadSmallWarps, smem, stream, a);
    CGNN_CHECK_LAUNCH();
    return CGNN_OK;
  }
  auto kfn = k_head_fwd;
  CGNN_LAUNCH(kfn, (unsigned)((num_graphs + kWarps - 1) / kWarps), kThreads, 0, stream, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_ce_fwd(const float* logits, const int64_t* labels, int64_t num_graphs, int32_t K, float inv_count,
                float* nll, float* loss, int64_t* correct, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || K <= 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs > 0 && (!logits || !labels)) return CGNN_ERR_INVALID_ARG;
  auto kfn = k_ce_fwd;
  CGNN_LAUNCH(kfn, 1, num_graphs > 256 ? 1024 : 256, 0, stream, logits, (const long long*)labels, (long long)num_graphs, (int)K,
              inv_count, nll, loss, (long long*)correct);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_ce_bwd(const float* logits, const int64_t* labels, int64_t num_graphs, int32_t K, float inv_count,
                const float* gout, float* dlogits, cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || K <= 0) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) return CGNN_OK;
  if (!logits || !labels || !dlogits) return CGNN_ERR_INVALID_ARG;
  auto kfn = k_ce_bwd;
  CGNN_LAUNCH(kfn, (unsigned)((num_graphs + 255) / 256), 256, 0, stream, logits, (const long long*)labels,
              (long long)num_graphs, (int)K, inv_count, gout, dlogits);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int cgnn_head_bwd(const float* emb, const float* hidden, const float* dlogits, const float* W0, const float* W1,
                  int64_t num_graphs, int32_t C, int32_t M, int32_t K, float p_drop, float* demb, float* dW0,
                  float* db0, float* dW1, float* db1, void* workspace, size_t workspace_bytes,
                  cgnn_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_graphs < 0 || C <= 0 || M <= 0 || K <= 0 || !dW0 || !db0 || !dW1 || !db1) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) {
    cudaMemsetAsync(dW0, 0, (size_t)M * C * sizeof(float), stream);
    cudaMemsetAsync(db0, 0, (size_t)M * sizeof(float), stream);
    cudaMemsetAsync(dW1, 0, (size_t)K * M * sizeof(float), stream);
    cudaMemsetAsync(db1, 0, (size_t)K * sizeof(float), stream);
    return CGNN_OK;
  }
  if (!emb || !hidden || !dlogits || !W0 || !W1 || !demb || !workspace) return CGNN_ERR_INVALID_ARG;
  if (C > kHeadMaxC || M > kHeadMaxM || K > kHeadMaxK) return CGNN_ERR_TILE_TOO_LARGE;
  const DeviceInfo dev = device_info();
  HeadBwdArgs a;
  a.emb = emb; a.hidden = hidden; a.dlogits = dlogits; a.W0 = W0; a.W1 = W1;
  a.B = num_graphs; a.C = C; a.M = M; a.K = K;
  a.keep_scale = p_drop > 0.0f ? 1.0f / (1.0f - p_drop) : 1.0f;
  a.demb = demb;
  a.o_dw0 = 0; a.o_db0 = M * C; a.o_dw1 = a.o_db0 + M; a.o_db1 = a.o_dw1 + K * M;
  a.part_stride = a.o_db1 + K;
  int off = 0;
  a.o_acc = off; off += round_up(a.part_stride, 4);
  a.o_dhp = off; off += kWarps * M;
  a.o_emb = off; off += kWarps * C;
  a.o_dl = off; off += kWarps * K;
  a.o_hid = off; off += kWarps * M;
  const size_t smem = (size_t)off * sizeof(float);
  if (smem > (size_t)dev.smem_optin) return CGNN_ERR_TILE_TOO_LARGE;
  const long long groups = (num_graphs + kWarps - 1) / kWarps;
  int grid = persistent_grid(groups, smem, dev, kThreads);
  if (grid > 2 * dev.sm_count) grid = 2 * dev.sm_count;
  const size_t rec = (size_t)a.part_stride * sizeof(float);
  if (workspace_bytes < rec) return CGNN_ERR_WORKSPACE;
  if ((size_t)grid * rec > workspace_bytes) grid = (int)(workspace_bytes / rec);
  a.partials = (float*)workspace;
  auto kfn = k_head_bwd;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  CGNN_LAUNCH(kfn, grid, kThreads, smem, stream, a);
  CGNN_CHECK_LAUNCH();
  ReduceQueue rq(stream);
  rq.add(a.partials + a.o_dw0, grid, a.part_stride, M, C, C, dW0);
  rq.add(a.partials + a.o_db0, grid, a.part_stride, 1, M, M, db0);
  rq.add(a.partials + a.o_dw1, grid, a.part_stride, K, M, M, dW1);
  rq.add(a.partials + a.o_db1, grid, a.part_stride, 1, K, K, db1);
  return rq.flush();
}

}  // extern "C"
