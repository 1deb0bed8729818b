// tile.cuh - building blocks shared by the GCN / GraphSAGE layer kernels: per-channel constant staging, the output
// gradient of the backward kernels, per-CTA reductions, Welford statistics epilogue, CSR rows in shared memory.
#pragma once
#include "common.cuh"

namespace cgnn {

// Per-channel affine constants of an Act into shared memory, padded to C4 with zeros
// (identity -> scale 1, shift 0).  Caller syncs.
__device__ __forceinline__ void stage_affine(const Act& a, int C, int C4, float* s_scale, float* s_shift) {
  for (int c = threadIdx.x; c < C4; c += blockDim.x) {
    float sc = 0.0f, sh = 0.0f;
    if (c < C) { sc = a.scale ? a.scale[c] : 1.0f; sh = a.scale ? a.shift[c] : 0.0f; }
    s_scale[c] = sc;
    s_shift[c] = sh;
  }
}

// Per-channel constants of the output gradient dz of a GCN / GraphSAGE backward, [DZ_ROWS][H4] in shared memory: the
// output activation's affine map and the BatchNorm-backward coefficients.  CTAs of kThreads; caller syncs.
enum { DZ_SCALE = 0, DZ_SHIFT, DZ_BSC, DZ_MEAN, DZ_RSTD, DZ_S1N, DZ_S2N, DZ_ROWS };
__device__ __forceinline__ void stage_dz_consts(const Act& act_out, const BnBwdDev& bn, int H, int H4, float* s) {
  stage_affine(act_out, H, H4, s + DZ_SCALE * H4, s + DZ_SHIFT * H4);
  for (int c = threadIdx.x; c < H4; c += kThreads) {
    const BnCoef k = bn_bwd_coef(bn, c, H);
    s[DZ_BSC * H4 + c] = k.bsc;
    s[DZ_MEAN * H4 + c] = k.mean;
    s[DZ_RSTD * H4 + c] = k.rstd;
    s[DZ_S1N * H4 + c] = k.s1n;
    s[DZ_S2N * H4 + c] = k.s2n;
  }
}
// dz of one element: dropout/ReLU backward of the upstream gradient, then BatchNorm backward
__device__ __forceinline__ float staged_dz(const Act& act_out, const BnBwdDev& bn, const float* s, int H4, bool aff_out, float t,
                                           float up, uint32_t rh, int c) {
  const float dy = act_bwd(act_out, aff_out, t, s[DZ_SCALE * H4 + c], s[DZ_SHIFT * H4 + c], rh, c, up);
  if (!bn.has) return dy;
  if (!bn.train) return s[DZ_BSC * H4 + c] * dy;
  return bn_bwd_dz(BnCoef{s[DZ_MEAN * H4 + c], s[DZ_RSTD * H4 + c], s[DZ_BSC * H4 + c], s[DZ_S1N * H4 + c], s[DZ_S2N * H4 + c]}, t, dy);
}

// The per-CTA reductions of per-thread partial sums, each in one fixed order.
// Element j of channel quad q summed over the threads th = q, q + Q, q + 2Q, ... < nt that own that quad:
// rec[th * stride + off + j].
__device__ __forceinline__ float quad_sum(const float* rec, int stride, int off, int nt, int Q, int q, int j) {
  float s = 0.0f;
  for (int th = q; th < nt; th += Q) s += rec[th * stride + off + j];
  return s;
}
// Column c of a lane-per-channel record summed over the warps 0, 1, ..., kWarps - 1: s_red[w * ld + c].
__device__ __forceinline__ float warp_rows_sum(const float* s_red, int ld, int c) {
  float s = 0.0f;
  for (int w = 0; w < kWarps; ++w) s += s_red[w * ld + c];
  return s;
}

// Per-warp running Welford state for HC channels per lane (channel = lane + 32*j).
template <int HC>
struct WarpStats {
  Welford w[HC];
  int rows;
  __device__ __forceinline__ void init() {
    rows = 0;
#pragma unroll
    for (int j = 0; j < HC; ++j) w[j].init();
  }
  __device__ __forceinline__ void begin_row(float& inv) { rows += 1; inv = fast_rcp((float)rows); }
  // Deposit into shared scratch: s_cnt[warp], s_mean[warp*ldc + c], s_m2[...]
  __device__ __forceinline__ void deposit(float* s_cnt, float* s_mean, float* s_m2, int ldc, int C4) const {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_cnt[warp] = (float)rows;
#pragma unroll
    for (int j = 0; j < HC; ++j) {
      const int c = lane + 32 * j;
      if (c < C4) { s_mean[warp * ldc + c] = w[j].mean; s_m2[warp * ldc + c] = w[j].m2; }
    }
  }
};

// ---- one subject's CSR rows, either staged in shared memory or read in place ---------------
// All three arrays are indexed with ABSOLUTE positions (rp[i] are global edge positions, col/w are
// pre-offset by -first_edge when they live in shared memory), so the same loop serves both homes.
struct RowCsr {
  const int* rp;     // [n+1] row i owns edges [rp[i], rp[i+1])
  const int* col;    // global row id of the neighbour
  const float* w;
};

static inline __host__ __device__ int csr_words(int max_nodes, int max_edges) {
  return round_up(max_nodes + 1, 4) + 2 * round_up(max_edges, 4) + round_up(max_nodes, 4);
}

// Start the async copy of a subject's CSR slice (+ one per-row float array) into shared memory.
// s_base layout: [rp: max_nodes+1][col: max_edges][w: max_edges][extra: max_nodes] (each rounded up to 4 words).
__device__ __forceinline__ void stage_csr_async(float* s_base, int max_nodes, int max_edges, const int32_t* rowptr,
                                                const int32_t* col, const float* w, const float* extra, long long nb,
                                                int n, int eb, int m) {
  int* s_rp = reinterpret_cast<int*>(s_base);
  int* s_col = s_rp + round_up(max_nodes + 1, 4);
  float* s_w = reinterpret_cast<float*>(s_col + round_up(max_edges, 4));
  float* s_extra = s_w + round_up(max_edges, 4);
  cp_async_words(s_rp, rowptr + nb, n + 1);
  cp_async_words(s_col, col + eb, m);
  cp_async_words(s_w, w + eb, m);
  if (extra) cp_async_words(s_extra, extra + nb, n);
}
__device__ __forceinline__ RowCsr staged_csr(float* s_base, int max_nodes, int max_edges, int eb, const float** extra) {
  int* s_rp = reinterpret_cast<int*>(s_base);
  int* s_col = s_rp + round_up(max_nodes + 1, 4);
  float* s_w = reinterpret_cast<float*>(s_col + round_up(max_edges, 4));
  *extra = s_w + round_up(max_edges, 4);
  return RowCsr{s_rp, s_col - eb, s_w - eb};
}

// acc[j] (+)= sum over the edges of row i of w_e * tile[(col_e - nb) * ld + lane + 32 j].
// EXACT keeps the reference's rounding (product rounded, then added, in COO order); otherwise FMA.
template <int HC, bool EXACT>
__device__ __forceinline__ void gather_row(const RowCsr& c, int i, long long nb, int n, const float* __restrict__ tile,
                                           int ld, int C4, float (&acc)[HC]) {
  const int lane = threadIdx.x & 31;
  const int e0 = c.rp[i], e1 = c.rp[i + 1];
  for (int e = e0; e < e1; ++e) {
    const int src = (int)(c.col[e] - nb);
    const float w = c.w[e];
    if ((unsigned)src < (unsigned)n) {
#pragma unroll
      for (int j = 0; j < HC; ++j) {
        const int ch = lane + 32 * j;
        if (ch < C4) {
          const float v = tile[src * ld + ch];
          acc[j] = EXACT ? __fadd_rn(acc[j], __fmul_rn(v, w)) : fmaf(v, w, acc[j]);
        }
      }
    }
  }
}

static inline int pick_hc(int C4) { return C4 <= 32 ? 1 : (C4 <= 64 ? 2 : (C4 <= 128 ? 4 : 8)); }

}  // namespace cgnn
