// rowtile.cuh - building blocks of the row-tile streaming kernels in gemm_tc.cu (sm_100a only).
//
// A row tile is TR consecutive rows of the batch (TR = 128 or 64).  Every thread owns ONE channel quad (4 consecutive
// channels) of a tile and the rows r, r + RS, r + 2 RS, ... of it, so everything per channel - BatchNorm scale/shift,
// dropout stream constants, bias, column sums, swizzled operand offsets - is computed once and lives in registers;
// per tile a thread only adds a constant byte stride to its operand addresses.
#pragma once
#include "tc05.cuh"

#ifndef CGNN_EMU
namespace cgnn {
namespace rt {

// thread <-> (quad column q, first row r) for a tile of TR rows x 4*Q channels; Q in {8, 16, 32}
template <int Q, int TR, int NT = kThreads>
struct QuadMap {
  static constexpr int RS = NT / Q;          // rows between two quads of one thread
  static constexpr int NQ = TR / RS;         // quads per thread per tile
  static_assert(NT % Q == 0 && RS % 8 == 0 && TR % RS == 0 && NQ >= 1, "unsupported tile shape");
};

// byte offset of the quad (row, 4q) in a K-major 128B-swizzled operand of `rows` rows per 32-channel block
__device__ __forceinline__ uint32_t kmajor_quad_offset(int row, int q, int rows) {
  return (uint32_t)((q >> 3) * rows * 128 + (row >> 3) * 1024 + (row & 7) * 128 + ((((q & 7) ^ (row & 7))) << 4));
}
// the same quad in an MN-major SWIZZLE_128B_BASE32B operand (row = contraction index, `rows` of them)
__device__ __forceinline__ uint32_t mnmajor_quad_offset(int row, int q, int rows) {
  return (uint32_t)((q >> 3) * rows * 128 + (row >> 2) * 512 + (row & 3) * 128 + (((((q & 7) >> 1) ^ (row & 3))) << 5) + ((q & 1) << 4));
}
// advancing a thread's row by RS (a multiple of 8) moves either offset by RS * 128 bytes
constexpr uint32_t kRowBytes = 128;

__device__ __forceinline__ void sts4(unsigned char* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// ---- per-thread constants of one channel quad of an Act ---------------------------------------------------------
struct ChanQuad {
  float sc[4], sh[4];
  uint32_t ck;         // dropout: drop_quad_key of this quad
};
__device__ __forceinline__ void chan_quad_init(ChanQuad& cq, const Act& a, int c0, int C) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const bool ok = a.scale != nullptr && c0 + j < C;
    cq.sc[j] = ok ? a.scale[c0 + j] : 1.0f;
    cq.sh[j] = ok ? a.shift[c0 + j] : 0.0f;
  }
  cq.ck = drop_quad_key(a, c0 >> 2);
}
// Dropout row key: the per-row hash of common.cuh::drop_row_hash for global row ids (row_base + row) computed from
// 32-bit pieces - the high word's hash is formed once per kernel (and once more for rows behind a 2^32 boundary).
struct RowKey {
  uint32_t lo0, hh0, hh1;
};
__device__ __forceinline__ RowKey row_key(const Act& a) {
  RowKey k;
  const unsigned long long base = (unsigned long long)a.row_base;
  k.lo0 = (uint32_t)base;
  const uint32_t hi = (uint32_t)(base >> 32);
  k.hh0 = fmix32(hi + a.k1);
  k.hh1 = fmix32(hi + 1u + a.k1);
  return k;
}
__device__ __forceinline__ uint32_t row_hash_at(const Act& a, const RowKey& k, uint32_t row) {
  const uint32_t lo = k.lo0 + row;
  const uint32_t hh = lo >= k.lo0 ? k.hh0 : k.hh1;
  return (lo * 0x9E3779B1u) ^ a.k0 ^ hh;
}
// u = dropout(relu?(sc t + sh)) on the quad
__device__ __forceinline__ float4 act_fwd4(const Act& a, const ChanQuad& cq, float4 t, const RowKey& rk, uint32_t row) {
  float y[4] = {t.x, t.y, t.z, t.w};
  if (a.scale != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) y[j] = fmaf(y[j], cq.sc[j], cq.sh[j]);
  }
  if (a.relu) {
#pragma unroll
    for (int j = 0; j < 4; ++j) y[j] = fmaxf(y[j], 0.0f);
  }
  if (a.drop) {
    const uint32_t keep = drop_keep4(a, row_hash_at(a, rk, row), cq.ck);
#pragma unroll
    for (int j = 0; j < 4; ++j) y[j] = ((keep >> j) & 1u) ? y[j] * a.keep_scale : 0.0f;
  }
  return make_float4(y[0], y[1], y[2], y[3]);
}
// dy = d act / d y * du on the quad (t = the stored pre-activation value)
__device__ __forceinline__ float4 act_bwd4(const Act& a, const ChanQuad& cq, float4 t, float4 du, const RowKey& rk, uint32_t row) {
  const float tv[4] = {t.x, t.y, t.z, t.w};
  float d[4] = {du.x, du.y, du.z, du.w};
  uint32_t pass = 0xfu;
  if (a.relu) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float y = a.scale != nullptr ? fmaf(tv[j], cq.sc[j], cq.sh[j]) : tv[j];
      if (!(y > 0.0f)) pass &= ~(1u << j);
    }
  }
  if (a.drop) {
    pass &= drop_keep4(a, row_hash_at(a, rk, row), cq.ck);
#pragma unroll
    for (int j = 0; j < 4; ++j) d[j] *= a.keep_scale;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) d[j] = ((pass >> j) & 1u) ? d[j] : 0.0f;
  return make_float4(d[0], d[1], d[2], d[3]);
}

// BatchNorm-backward coefficients of one channel quad
struct BnQuad {
  BnCoef k[4];
};
__device__ __forceinline__ void bn_quad_init(BnQuad& b, const BnBwdDev& bn, int c0, int C) {
#pragma unroll
  for (int j = 0; j < 4; ++j) b.k[j] = bn_bwd_coef(bn, c0 + j, C);
}
__device__ __forceinline__ float4 bn_bwd4(const BnBwdDev& bn, const BnQuad& b, float4 t, float4 dy) {
  if (!bn.has) return dy;
  const float tv[4] = {t.x, t.y, t.z, t.w};
  float d[4] = {dy.x, dy.y, dy.z, dy.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) d[j] = bn.train ? bn_bwd_dz(b.k[j], tv[j], d[j]) : b.k[j].bsc * d[j];
  return make_float4(d[0], d[1], d[2], d[3]);
}
// dz of the quad of the layer output z from the upstream gradient up: dropout / ReLU backward of the output activation,
// then BatchNorm backward; RELU_MASK: then the layer's own ReLU (GraphSAGE, z = relu(.))
template <bool RELU_MASK>
__device__ __forceinline__ float4 dz4(const Act& act_out, const ChanQuad& cq, const BnBwdDev& bn, const BnQuad& bq, float4 z, float4 up,
                                      const RowKey& rk, uint32_t row) {
  float4 dz = bn_bwd4(bn, bq, z, act_bwd4(act_out, cq, z, up, rk, row));
  if (RELU_MASK) {
    if (!(z.x > 0.0f)) dz.x = 0.0f;
    if (!(z.y > 0.0f)) dz.y = 0.0f;
    if (!(z.z > 0.0f)) dz.z = 0.0f;
    if (!(z.w > 0.0f)) dz.w = 0.0f;
  }
  return dz;
}
// mean / rstd of the BatchNorm of the layer below for the quad c0.. (zero unless `want` and c < C), for bn_sums_add
__device__ __forceinline__ void bn_stats_quad(float (&mean)[4], float (&rstd)[4], const float* m, const float* r, int c0, int C, bool want) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const bool ok = want && c0 + j < C;
    mean[j] = ok ? m[c0 + j] : 0.0f;
    rstd[j] = ok ? r[c0 + j] : 0.0f;
  }
}

// 4 channels c0.. of row `row` of a dense [rows, C] tensor; VEC: one 16-byte load, else bounded scalar loads
template <bool VEC>
__device__ __forceinline__ float4 ld_quad(const float* __restrict__ base, long long row, int C, int c0) {
  if (VEC) return *reinterpret_cast<const float4*>(base + row * C + c0);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  const float* s = base + row * C + c0;
  if (c0 + 0 < C) v.x = s[0];
  if (c0 + 1 < C) v.y = s[1];
  if (c0 + 2 < C) v.z = s[2];
  if (c0 + 3 < C) v.w = s[3];
  return v;
}
template <bool VEC>
__device__ __forceinline__ void st_quad(float* __restrict__ base, long long row, int C, int c0, float4 v) {
  float* d = base + row * C + c0;
  if (VEC) { *reinterpret_cast<float4*>(d) = v; return; }
  if (c0 + 0 < C) d[0] = v.x;
  if (c0 + 1 < C) d[1] = v.y;
  if (c0 + 2 < C) d[2] = v.z;
  if (c0 + 3 < C) d[3] = v.w;
}
// the upstream gradient of every row of subject g (n rows) under a mean pool: the quad c0.. of demb[g] / (n + 1e-8)
template <bool VEC>
__device__ __forceinline__ float4 pooled_quad(const float* __restrict__ demb, long long g, int C, int c0, int n) {
  const float inv_n = pool_bwd_scale(n);
  const float4 e = ld_quad<VEC>(demb, g, C, c0);
  return make_float4(e.x * inv_n, e.y * inv_n, e.z * inv_n, e.w * inv_n);
}
__device__ __forceinline__ float4 mask_quad(float4 v, int c0, int C) {   // zero the channels >= C
  if (c0 + 0 >= C) v.x = 0.0f;
  if (c0 + 1 >= C) v.y = 0.0f;
  if (c0 + 2 >= C) v.z = 0.0f;
  if (c0 + 3 >= C) v.w = 0.0f;
  return v;
}

// ---- accumulator tile -> XOR-swizzled staging [TR][NC] in shared memory (lane = row) ----------------------------
// float4 index of quad q of row r: r * (NC/4) + (q ^ (r & 7)): conflict-free for the row-per-lane writes below and for
// the quad-per-thread reads of the epilogues.
__device__ __forceinline__ int stage_index(int row, int q, int QN) { return row * QN + (q ^ (row & 7)); }

template <int NC, int NT = kThreads>
__device__ __forceinline__ void drain_rows_to_staging(uint32_t taddr, float4* stage, int warp, int lane) {
  constexpr int CW = NC / (NT / 128);   // columns per warp: 4 lane quarters x NT / 128 column groups
  const int lq = warp & 3, cg = warp >> 2, row = 32 * lq + lane;
  float v[CW];
  tc::tmem_ld<CW>(taddr + ((uint32_t)(32 * lq) << 16) + (uint32_t)(cg * CW), v);
  tc::tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < CW / 4; ++j)
    stage[stage_index(row, cg * (CW / 4) + j, NC / 4)] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

// ---- MMA issue loops (one thread) -----------------------------------------------------------------------------------
// The 64-bit shared-memory descriptors of the four operand tiles are formed once per kernel; per MMA the issuing
// thread only adds a compile-time byte offset (>> 4) to the low word, so a whole K loop is a straight run of
// tcgen05.mma instructions with immediate adds in between.
struct OperandDescs {
  uint64_t a_hi, a_lo, b_hi, b_lo;
};
__device__ __forceinline__ OperandDescs kmajor_descs(uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo) {
  return OperandDescs{tc::smem_desc_sw128(a_hi), tc::smem_desc_sw128(a_lo), tc::smem_desc_sw128(b_hi), tc::smem_desc_sw128(b_lo)};
}
__device__ __forceinline__ OperandDescs mnmajor_descs(uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, int krows) {
  const uint32_t lbo = (uint32_t)krows * 128u;
  return OperandDescs{tc::smem_desc_mn32(a_hi, lbo, 512u), tc::smem_desc_mn32(a_lo, lbo, 512u), tc::smem_desc_mn32(b_hi, lbo, 512u),
                      tc::smem_desc_mn32(b_lo, lbo, 512u)};
}
// D (+)= A B^T with K-major 128B-swizzled operands of A_ROWS / B_ROWS rows per 32-channel block; KSTEPS steps of 8
// channels are unrolled, `ksteps` (<= KSTEPS) of them are issued.
template <int KSTEPS, int A_ROWS, int B_ROWS>
__device__ __forceinline__ void issue_kmajor_x3(uint32_t d_tmem, const OperandDescs& od, int ksteps, uint32_t idesc, bool accumulate) {
#pragma unroll
  for (int ks = 0; ks < KSTEPS; ++ks) {
    if (ks < ksteps) {
      const uint64_t ao = (uint64_t)(((ks >> 2) * A_ROWS * 128 + (ks & 3) * 32) >> 4);
      const uint64_t bo = (uint64_t)(((ks >> 2) * B_ROWS * 128 + (ks & 3) * 32) >> 4);
      tc::mma_tf32x3_step(d_tmem, od.a_hi + ao, od.a_lo + ao, od.b_hi + bo, od.b_lo + bo, idesc, (accumulate || ks > 0) ? 1u : 0u);
    }
  }
}
// D (+)= A^T B with MN-major operands whose contraction index is the tile row (KROWS rows, 8 per step)
template <int KROWS>
__device__ __forceinline__ void issue_mnmajor_x3(uint32_t d_tmem, const OperandDescs& od, uint32_t idesc, bool accumulate) {
#pragma unroll
  for (int ks = 0; ks < KROWS / 8; ++ks) {
    const uint64_t off = (uint64_t)((ks * 1024) >> 4);
    tc::mma_tf32x3_step(d_tmem, od.a_hi + off, od.a_lo + off, od.b_hi + off, od.b_lo + off, idesc, (accumulate || ks > 0) ? 1u : 0u);
  }
}

}  // namespace rt
}  // namespace cgnn
#endif
