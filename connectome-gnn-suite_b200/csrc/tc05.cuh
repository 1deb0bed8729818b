// tc05.cuh - thin inline-PTX layer over the Blackwell tensor-core path as the cgnn kernels use it: fp32-grade projections
// P[rows, N] = X[rows, K] W[N, K]^T done as three TF32 MMAs (x = hi + lo split of both operands: hi*hi + hi*lo + lo*hi,
// fp32 accumulation in tensor memory), fed by mbarrier pipelines, TMA loads (cp.async.bulk / cp.async.bulk.tensor) and
// tcgen05.st / tcgen05.ld.
//
// Shared-memory operands are K-major, 128-byte swizzled "canonical" tiles (what TMA would write):
//   one block = [rows][32 tf32] (128 B per row), rows grouped by 8 (1024 B), 16-byte chunk index XORed
//   with (row % 8).  A K of 64 is two such blocks; one MMA consumes K = 8 (32 B) of a block.
//
// Two implementations of the primitives the warp-specialised kernels (engine.cu, eval_fused.cu) use:
//   * device (nvcc, sm_100a): inline PTX;
//   * -DCGNN_EMU (g++, tests/emu): a functional model - mbarriers are phase/count words polled by fibers, TMA
//     copies complete at issue, tensor memory is a [128][512] array, tcgen05.mma with A in tensor memory is a
//     TF32-truncating triple loop that decodes the SAME shared-memory descriptors.  It checks the protocol (phases,
//     counts, lane quadrants, indexing, layouts as this file states them), not the hardware; the layouts themselves
//     were pinned on a B200 (tests/test_gpu_parity.py).
// The SS-mode MMA and the MN-major operands have the device form only.
#pragma once
#include "common.cuh"

#ifndef CGNN_EMU
#include <cuda.h>   // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)
#endif

namespace cgnn {
namespace tc {

// ------------------------------------------------------------------------------------------------------------------
// shared-memory addresses
// ------------------------------------------------------------------------------------------------------------------
#ifdef CGNN_EMU
// "shared address" = byte offset into the block's dynamic shared memory (what descriptors carry)
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)(reinterpret_cast<const unsigned char*>(p) - cgnn_emu::g_dyn_smem);
}
#else
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
#endif
// 1024-byte aligned start of the dynamic shared memory, as a pointer the compiler still knows to be shared
// (an integer round trip would turn every access into a generic LD/ST with descriptor moves).
__device__ __forceinline__ unsigned char* smem_align1024(unsigned char* smem_raw) {
  return smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
}

// ------------------------------------------------------------------------------------------------------------------
// operand staging
// ------------------------------------------------------------------------------------------------------------------
// byte offset of element (row, k) of a K-major 128B-swizzled operand with `rows` rows per 32-wide K block
__device__ __forceinline__ uint32_t kmajor_offset(int row, int k, int rows) {
  return (uint32_t)((k >> 5) * rows * 128 + (row >> 3) * 1024 + (row & 7) * 128 + (((((k & 31) >> 2) ^ (row & 7))) << 4) + ((k & 3) << 2));
}
// hi part of the split: x rounded to the nearest tf32 (10 explicit mantissa bits) with an integer add + mask, two
// instructions where cvt.rna.tf32 compiles to four.  x - hi is exact and |x - hi| <= 2^-11 |x|; the tensor core
// ignores the low 13 bits of a tf32 operand, so the three-term product keeps ~2^-21 relative accuracy (measured
// in tests/test_gpu_parity.py).
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
// hi / lo parts of 4 values
__device__ __forceinline__ void split4(float4 v, float4& h, float4& l) {
  h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
  l = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
}
// write 4 consecutive k (k % 4 == 0) of one row as hi / lo parts
__device__ __forceinline__ void store_split4(unsigned char* hi_base, unsigned char* lo_base, int row, int k, int rows, float4 v) {
  const uint32_t off = kmajor_offset(row, k, rows);
  float4 h, l;
  split4(v, h, l);
  *reinterpret_cast<float4*>(hi_base + off) = h;
  *reinterpret_cast<float4*>(lo_base + off) = l;
}

// ------------------------------------------------------------------------------------------------------------------
// descriptors
// ------------------------------------------------------------------------------------------------------------------
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, sm_100):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major, 1)
//   [32,46) stride byte offset >> 4 (1024 B between 8-row groups) | [46,48) version = 1 | [61,64) layout = 2
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32; bit 15 / 16 = A / B is
// MN-major (0 = K-major)
__device__ __forceinline__ uint32_t idesc_tf32(int M, int N, int a_mn = 0, int b_mn = 0) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(a_mn & 1) << 15) | ((uint32_t)(b_mn & 1) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
#ifndef CGNN_EMU
// MN-major operands (the contraction runs over the ROWS of a staged tile X[r][c], i.e. X^T Y products).  For 32-bit
// (tf32) elements the only MN-major layout the tensor core accepts is SWIZZLE_128B_BASE32B (cute
// Layout_MN_SW128_32B_Atom, layout type 1): 128-byte rows hold 32 consecutive M (or N) indices as four 32-byte
// chunks, chunk index XORed with (k mod 4); 4 consecutive K indices form one 512-byte atom.  lbo = bytes between
// 32-wide MN groups, sbo = bytes between 4-deep K groups.  This is NOT the byte image of the K-major 128B swizzle,
// so a tile that feeds both X W and X^T Y is staged twice.
__device__ __forceinline__ uint64_t smem_desc_mn32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (1ull << 61);
}
#endif

// ------------------------------------------------------------------------------------------------------------------
// mbarrier.  mbar_init leaves the init fence to fence_mbar_init(), issued once after all inits and before the
// __syncthreads() that publishes them.
// ------------------------------------------------------------------------------------------------------------------
#ifdef CGNN_EMU
// word layout of the model: [0,20) pending arrivals | [20,40) arrival count per phase | [40,63) pending tx bytes | 63 phase
namespace emu {
inline void settle(uint64_t* bar) {
  uint64_t v = *bar;
  const uint64_t pending = v & 0xFFFFFu, init = (v >> 20) & 0xFFFFFu, tx = (v >> 40) & 0x7FFFFFu;
  if (pending == 0 && tx == 0) {
    v = (v & (1ull << 63)) ^ (1ull << 63);
    v |= init | (init << 20);
    *bar = v;
  }
  cgnn_emu::note_event();
}
inline void complete_tx(uint64_t* bar, uint32_t bytes) {
  const uint64_t tx = (*bar >> 40) & 0x7FFFFFu;
  if (tx < bytes) { fprintf(stderr, "[cuda_emu] complete_tx of %u bytes with %llu expected\n", bytes, (unsigned long long)tx); abort(); }
  *bar -= (uint64_t)bytes << 40;
  settle(bar);
}
}  // namespace emu
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { *bar = (uint64_t)count | ((uint64_t)count << 20); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  if ((*bar & 0xFFFFFu) == 0) { fprintf(stderr, "[cuda_emu] mbarrier over-arrival (thread %u)\n", threadIdx.x); abort(); }
  *bar -= 1;
  emu::settle(bar);
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  *bar += (uint64_t)bytes << 40;
  mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (((*bar >> 63) & 1u) == (uint64_t)(parity & 1u)) cgnn_emu::poll_yield();
}
__device__ __forceinline__ void fence_mbar_init() {}
__device__ __forceinline__ void fence_proxy_async() {}
__device__ __forceinline__ void named_sync(int id, int nthreads) { cgnn_emu::named_barrier(id, nthreads); }
#else
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// (a poll loop with __nanosleep between the try_waits was measured in the fused eval kernel: 400 M of its 680 M warp
// instructions were the sleeping loop and every hand-over gained its latency; the plain try_wait suspends in hardware)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
#endif

// ------------------------------------------------------------------------------------------------------------------
// TMA: 1-D bulk copies and 2-D tiled loads of a row-major fp32 matrix with the 128-byte swizzle
// ------------------------------------------------------------------------------------------------------------------
// A box is 32 fp32 columns (128 B) x BOX_ROWS rows; in shared memory row r of the box sits at r * 128 and its 16-byte
// chunk j at position j ^ (r & 7) (CU_TENSOR_MAP_SWIZZLE_128B; the destination must be 1024-byte aligned).
// Rows / columns outside the matrix arrive as zeros.
constexpr int kBoxCols = 32;
__device__ __host__ __forceinline__ uint32_t box_chunk_offset(int r, int j) { return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)); }

#ifdef CGNN_EMU
struct TensorMap {
  const float* base; long long rows; int cols, box_rows;
};
static inline int make_tensor_map(TensorMap* m, const float* base, long long rows, int cols, int box_rows) {
  m->base = base; m->rows = rows; m->cols = cols; m->box_rows = box_rows;
  return CGNN_OK;
}
__device__ __forceinline__ void tma_load_box(void* dst, const TensorMap* m, int col0, long long row0, uint64_t* bar) {
  if (smem_u32(dst) & 1023u) { fprintf(stderr, "[cuda_emu] TMA box destination not 1024-byte aligned\n"); abort(); }
  unsigned char* d = reinterpret_cast<unsigned char*>(dst);
  for (int r = 0; r < m->box_rows; ++r)
    for (int j = 0; j < 8; ++j) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      const long long gr = row0 + r;
      for (int e = 0; e < 4; ++e) {
        const int c = col0 + 4 * j + e;
        if (gr >= 0 && gr < m->rows && c < m->cols) v[e] = m->base[gr * m->cols + c];
      }
      memcpy(d + box_chunk_offset(r, j), v, 16);
    }
  emu::complete_tx(bar, (uint32_t)m->box_rows * 128u);
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  if ((bytes & 15u) || (smem_u32(dst) & 15u) || (((uintptr_t)src) & 15u)) { fprintf(stderr, "[cuda_emu] bulk copy alignment\n"); abort(); }
  memcpy(dst, src, bytes);
  emu::complete_tx(bar, bytes);
}
__device__ __forceinline__ void prefetch_tensor_map(const TensorMap*) {}
#else
using TensorMap = CUtensorMap;
// host: encode a [rows, cols] fp32 row-major matrix with 32-column x box_rows boxes (defined in engine.cu)
int make_tensor_map(TensorMap* m, const float* base, long long rows, int cols, int box_rows);
__device__ __forceinline__ void tma_load_box(void* dst, const TensorMap* m, int col0, long long row0, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(col0), "r"((int)row0), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void prefetch_tensor_map(const TensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
#endif

// ------------------------------------------------------------------------------------------------------------------
// tensor memory + MMA.  taddr = (lane << 16) | column; a warp reaches lanes [32 * (warp % 4), +32) only.
//   tmem_st<N> (N = 8, 16): N consecutive 32-bit columns of this thread's lane; tmem_st_wait() before the hand-over.
//   tmem_ld<N> (N = 8, 16, 32): the same read back WITHOUT the wait - issue several, then tmem_ld_wait() once, before
//   any of the values is used.
// ------------------------------------------------------------------------------------------------------------------
#ifdef CGNN_EMU
namespace emu {
inline int my_quadrant() { return (int)((threadIdx.x >> 5) & 3u); }
inline float* cell(uint32_t taddr, int lane_off, int col_off) {
  const int lane = (int)(taddr >> 16) + lane_off, col = (int)(taddr & 0xffffu) + col_off;
  if (lane < 0 || lane >= 128 || col < 0 || col >= 512) { fprintf(stderr, "[cuda_emu] tensor memory access out of range (lane %d col %d)\n", lane, col); abort(); }
  return cgnn_emu::tmem() + lane * 512 + col;
}
inline void check_quadrant(uint32_t taddr) {
  if ((int)(taddr >> 16) != 32 * my_quadrant()) {
    fprintf(stderr, "[cuda_emu] warp %u touches tensor-memory lane base %u outside its quadrant\n", threadIdx.x >> 5, taddr >> 16);
    abort();
  }
}
inline float trunc_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
}  // namespace emu
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t cols) { (void)cols; *smem_result = 0; }
__device__ __forceinline__ void tmem_dealloc(uint32_t, uint32_t) {}
__device__ __forceinline__ void fence_before_sync() {}
__device__ __forceinline__ void fence_after_sync() {}
template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const float (&v)[N]) {
  emu::check_quadrant(taddr);
  for (int i = 0; i < N; ++i) *emu::cell(taddr, (int)(threadIdx.x & 31u), i) = v[i];
}
__device__ __forceinline__ void tmem_st_wait() {}
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[N]) {
  emu::check_quadrant(taddr);
  for (int i = 0; i < N; ++i) v[i] = *emu::cell(taddr, (int)(threadIdx.x & 31u), i);
}
__device__ __forceinline__ void tmem_ld_wait() {}
// D[128 x N] (+)= A[tmem: lane = row, 8 columns = K] * B[smem, K-major SW128, N rows x 8 K]^T
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  const int N = (int)((idesc >> 17) & 0x3Fu) << 3, M = (int)((idesc >> 24) & 0x1Fu) << 4;
  if (M != 128) { fprintf(stderr, "[cuda_emu] mma: M = %d\n", M); abort(); }
  const uint32_t start = (uint32_t)(b_desc & 0x3FFFu) << 4;
  const uint32_t sbo = (uint32_t)((b_desc >> 32) & 0x3FFFu) << 4;
  for (int m = 0; m < 128; ++m)
    for (int n = 0; n < N; ++n) {
      float acc = accumulate ? *emu::cell(d_tmem, m, n) : 0.0f;
      for (int kk = 0; kk < 8; ++kk) {
        uint32_t addr = start + (uint32_t)(n >> 3) * sbo + (uint32_t)(n & 7) * 128u + 4u * (uint32_t)kk;
        addr ^= ((addr >> 7) & 7u) << 4;      // the 128-byte swizzle is a function of the address bits
        float b;
        memcpy(&b, cgnn_emu::g_dyn_smem + addr, 4);
        acc += emu::trunc_tf32(*emu::cell(a_tmem, m, kk)) * emu::trunc_tf32(b);
      }
      *emu::cell(d_tmem, m, n) = acc;
    }
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) { mbar_arrive(bar); }
#else
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t cols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {        // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const float (&v)[N]) {
  static_assert(N == 8 || N == 16, "tmem_st: 8 or 16 columns");
  if constexpr (N == 8) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
  } else {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
  }
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[N]) {
  static_assert(N == 8 || N == 16 || N == 32, "tmem_ld: 8, 16 or 32 columns");
  uint32_t r[N];
  if constexpr (N == 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr) : "memory");
  } else if constexpr (N == 16) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
  }
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]^T, one K = 8 step: A is read from tensor memory (lane = row of the tile, one 32-bit
// column per K element), so the instruction takes no shared-memory bandwidth for A.  Issued by ONE thread.
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrive on `bar` once every MMA issued so far by this thread has completed (implies fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- SS form: both operands in shared memory ----------------------------------------------------------------------
// D[tmem] (+)= A[smem] * B[smem]^T, one K = 8 step.  Issued by ONE thread.
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// One K = 8 step of the three-term product with explicit descriptors (hi/lo operand pairs).
__device__ __forceinline__ void mma_tf32x3_step(uint32_t d_tmem, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                                uint32_t idesc, uint32_t accumulate) {
  mma_tf32(d_tmem, a_lo, b_hi, idesc, accumulate);   // small terms first
  mma_tf32(d_tmem, a_hi, b_lo, idesc, 1u);
  mma_tf32(d_tmem, a_hi, b_hi, idesc, 1u);
}
// All K steps of the three-term product for one [M x N] tile: operands made of K/32 blocks.
//   a_hi/a_lo: [K/32][M rows][128 B]   b_hi/b_lo: [K/32][N rows][128 B]
__device__ __forceinline__ void mma_tf32x3(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, int M,
                                           int N, int K) {
  const uint32_t idesc = idesc_tf32(M, N);
  uint32_t acc = 0;
  // small terms first, the dominant hi*hi term last
  for (int term = 0; term < 3; ++term) {
    const uint32_t a = term == 0 ? a_lo : a_hi;
    const uint32_t b = term == 1 ? b_lo : b_hi;
    for (int k = 0; k < K; k += 8) {
      const uint32_t kb = (uint32_t)(k >> 5), ko = (uint32_t)((k & 31) * 4);
      mma_tf32(d_tmem, smem_desc_sw128(a + kb * (uint32_t)M * 128u + ko), smem_desc_sw128(b + kb * (uint32_t)N * 128u + ko), idesc, acc);
      acc = 1;
    }
  }
}
#endif

// One K = 8 step of the fp32-grade product with A = (a_hi, a_lo) in tensor memory and B = (b_hi, b_lo) descriptors:
// small terms first, the dominant hi * hi term last.
__device__ __forceinline__ void mma_tf32x3_ts(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, uint64_t b_hi, uint64_t b_lo, uint32_t idesc,
                                              uint32_t accumulate) {
  mma_tf32_ts(d_tmem, a_lo, b_hi, idesc, accumulate);
  mma_tf32_ts(d_tmem, a_hi, b_lo, idesc, 1u);
  mma_tf32_ts(d_tmem, a_hi, b_hi, idesc, 1u);
}

}  // namespace tc
}  // namespace cgnn
