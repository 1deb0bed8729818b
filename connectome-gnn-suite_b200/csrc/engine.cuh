// engine.cuh - the warp-specialised engine's roles, shared by its two kernels (engine.cu: one hidden layer;
// eval_fused.cu: the whole network in eval mode): role layout, tensor-memory column plan, unit geometry and table, the
// P-tile swizzle, the pipeline barriers and the role steps both kernels take in the same way.
#pragma once
#include "agg.cuh"
#include "tc05.cuh"

namespace cgnn {
namespace eng {

constexpr int kC = 64;                    // channels in and out
constexpr int kTR = 128;                  // rows per tile (MMA M)
constexpr int kMaxTiles = 3;              // tiles per unit
constexpr int kMaxUnitRows = kTR * kMaxTiles;
constexpr int kMaxSub = 16;               // subjects per unit
constexpr int kStageBytes = kTR * 128;    // one box: 128 rows x 32 channels
constexpr int kNS = 2;                    // staging slots (slot = channel half)
constexpr int kWarpTile = 0, kWarpMma = 1, kWarpAlloc = 2, kWarpBlob = 3;
constexpr int kConvWarp0 = 4, kConvWarps = 8, kGathWarp0 = 12, kGathWarps = 16;
constexpr int kNT = 32 * (kGathWarp0 + kGathWarps);
constexpr int kGathThreads = 32 * kGathWarps;
constexpr uint32_t kColAHi = 0, kColALo = 64, kColD = 128, kTmemCols = 512;
constexpr size_t kStaticSmem = 1024;        // barriers + tensor-memory address, rounded up by the alignment of the dynamic part

// the rings between converters, MMA issuer, blob producer and gather warps
struct PipeBars {
  uint64_t a_full[2], a_free[2];                  // A columns of a channel half
  uint64_t d_full[kMaxTiles], d_free[kMaxTiles];  // accumulator slot of a tile of the unit
  uint64_t blob_full[2], blob_free[2];            // blob buffer
};
__device__ __forceinline__ void init_pipe_bars(PipeBars& b) {
  for (int i = 0; i < 2; ++i) { tc::mbar_init(&b.a_full[i], 4 * 32); tc::mbar_init(&b.a_free[i], 1); }
  for (int i = 0; i < kMaxTiles; ++i) { tc::mbar_init(&b.d_full[i], 1); tc::mbar_init(&b.d_free[i], kGathWarps); }
  for (int i = 0; i < 2; ++i) { tc::mbar_init(&b.blob_full[i], 1); tc::mbar_init(&b.blob_free[i], kGathWarps); }
}

// how a launch cuts the batch into units, and where their records are
struct UnitPlan {
  const int32_t* blob; const int32_t* meta;   // packed in-edge records (agg.cuh), per-subject {first row, rows, first edge, edges}
  long long B, units;
  int spu;                 // subjects per unit
  int blob_cap_bytes;      // one blob buffer
  int nblob;               // 1 or 2 blob buffers
};

// geometry of unit u
struct Unit {
  long long g0; int nsub;
  long long row0; int rows, tiles;
  long long blob_word0; int blob_bytes;
};
__device__ __forceinline__ Unit unit_geom(const UnitPlan& p, long long u) {
  Unit r;
  r.g0 = u * p.spu;
  long long g1 = r.g0 + p.spu;
  if (g1 > p.B) g1 = p.B;
  r.nsub = (int)(g1 - r.g0);
  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  const int4 m0 = meta[r.g0], m1 = meta[g1 - 1];
  r.row0 = m0.x;
  r.rows = m1.x + m1.y - m0.x;
  if (r.rows > kMaxUnitRows) r.rows = kMaxUnitRows;       // host contract; never index past the tiles
  r.tiles = (r.rows + kTR - 1) / kTR;
  r.blob_word0 = agg_base_words(m0.x, m0.z, r.g0);
  const long long end = agg_base_words(m1.x, m1.z, g1 - 1) + ((agg_copy_words(m1.y, m1.w) + 3) & ~3);
  long long bytes = (end - r.blob_word0) * 4;
  if (bytes > p.blob_cap_bytes) bytes = p.blob_cap_bytes;
  r.blob_bytes = (int)bytes;
  return r;
}

// the unit table the gather warps build one unit ahead in shared memory
struct SubRec {
  int row;       // first row in the unit's tiles
  int prow;      // first row in P (8-aligned)
  int rows;
  int blob;      // word offset of the subject's records in the unit's blob
  int pair;      // first flat pair index of the unit
  int pad_[3];
};
struct UnitTab {
  int rows, nsub, groups, tiles;   // groups: row pairs of the unit
  long long row0, g0;
  SubRec sub[kMaxSub];
};

// one warp: lane j < nsub writes subject j's record, lane 0 the header
__device__ __forceinline__ void build_unit_tab(const UnitPlan& p, long long u, UnitTab* tab, int lane) {
  const Unit un = unit_geom(p, u);
  const int4* meta = reinterpret_cast<const int4*>(p.meta);
  int4 m = make_int4(0, 0, 0, 0);
  if (lane < un.nsub) m = meta[un.g0 + lane];
  const int n = lane < un.nsub ? m.y : 0;
  int pincl = (n + 7) & ~7, gincl = (n + 1) >> 1;
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(kFull, pincl, o), b = __shfl_up_sync(kFull, gincl, o);
    if (lane >= o) { pincl += a; gincl += b; }
  }
  const int groups = __shfl_sync(kFull, gincl, 31);
  if (lane < un.nsub) {
    SubRec& e = tab->sub[lane];
    e.row = (int)(m.x - un.row0);
    e.prow = pincl - ((n + 7) & ~7);
    e.rows = n;
    e.blob = (int)(agg_base_words(m.x, m.z, un.g0 + lane) - un.blob_word0);
    e.pair = gincl - ((n + 1) >> 1);
  }
  if (lane == 0) {
    tab->rows = un.rows; tab->nsub = un.nsub; tab->groups = groups; tab->tiles = un.tiles;
    tab->row0 = un.row0; tab->g0 = un.g0;
  }
}

// byte offset of 16-byte chunk c (0..15) of row `prow` of the P tile; `key` = the row's index inside its subject
__device__ __forceinline__ uint32_t p_chunk_offset(int prow, int key, int c) {
  return (uint32_t)(prow * 256 + ((((c ^ key) & 7) | (c & 8)) << 4));
}

// W [64 out][64 in] -> K-major operand rows n = output channel, hi / lo parts; threads tid, tid + nthreads, ...
__device__ __forceinline__ void stage_w_split(unsigned char* hi, unsigned char* lo, const float* W, int tid, int nthreads) {
  for (int idx = tid; idx < kC * (kC / 4); idx += nthreads) {
    const int n = idx / (kC / 4), k = (idx - n * (kC / 4)) * 4;
    tc::store_split4(hi, lo, n, k, kC, *reinterpret_cast<const float4*>(W + n * kC + k));
  }
}

// ---- roles ------------------------------------------------------------------------------------------------------------
// blob producer (one thread): every unit's records into the blob ring
__device__ __forceinline__ void blob_producer(const UnitPlan& p, PipeBars& bars, unsigned char* s_blob) {
  uint32_t ucount = 0;
  for (long long u = blockIdx.x; u < p.units; u += gridDim.x, ++ucount) {
    const Unit un = unit_geom(p, u);
    const uint32_t b = ucount % (uint32_t)p.nblob, use = ucount / (uint32_t)p.nblob;
    tc::mbar_wait(&bars.blob_free[b], (use & 1u) ^ 1u);
    tc::mbar_arrive_expect_tx(&bars.blob_full[b], (uint32_t)un.blob_bytes);
    tc::bulk_load(s_blob + (size_t)b * p.blob_cap_bytes, p.blob + un.blob_word0, (uint32_t)un.blob_bytes, &bars.blob_full[b]);
  }
}

// MMA issuer: P = u W^T of tile t, the `tq`-th tile of this CTA, into accumulator slot t (in its `use`-th use)
__device__ __forceinline__ void mma_tile(PipeBars& bars, uint32_t tmem, int t, uint32_t& use, uint32_t tq, uint32_t idesc,
                                         uint64_t b_hi, uint64_t b_lo) {
  tc::mbar_wait(&bars.d_free[t], (use & 1u) ^ 1u);     // the gather warps have drained this slot's previous tile
  ++use;
  const uint32_t d = tmem + kColD + (uint32_t)(kC * t);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    tc::mbar_wait(&bars.a_full[h], tq & 1u);
    tc::fence_after_sync();
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t bo = (uint64_t)((h * kC * 128 + ks * 32) >> 4);
      const uint32_t ac = (uint32_t)(32 * h + 8 * ks);
      tc::mma_tf32x3_ts(d, tmem + kColAHi + ac, tmem + kColALo + ac, b_hi + bo, b_lo + bo, idesc, (h | ks) ? 1u : 0u);
    }
    tc::mma_commit(&bars.a_free[h]);       // this half of the A columns may be rewritten once these MMAs are done
  }
  tc::mma_commit(&bars.d_full[t]);
}

// converters (thread = row of the tile): the row's 32 channels of channel half h from a box-swizzled slot
__device__ __forceinline__ void load_box_row(const unsigned char* slot, int row, float4 (&v)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const float4*>(slot + tc::box_chunk_offset(row, j));
}
// ... and, once the MMAs of the `tq`-th tile's predecessor have read channel half h, its TF32 hi / lo parts into the A
// columns at tensor-memory lane address `lane_addr`
__device__ __forceinline__ void store_a_row(PipeBars& bars, uint32_t lane_addr, int h, uint32_t tq, const float4 (&v)[8]) {
  tc::mbar_wait(&bars.a_free[h], (tq & 1u) ^ 1u);
  tc::fence_after_sync();
#pragma unroll
  for (int part = 0; part < 2; ++part) {
    float hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 hq, lq;
      tc::split4(v[4 * part + j], hq, lq);
      hi[4 * j + 0] = hq.x; hi[4 * j + 1] = hq.y; hi[4 * j + 2] = hq.z; hi[4 * j + 3] = hq.w;
      lo[4 * j + 0] = lq.x; lo[4 * j + 1] = lq.y; lo[4 * j + 2] = lq.z; lo[4 * j + 3] = lq.w;
    }
    const uint32_t col = (uint32_t)(32 * h + 16 * part);
    tc::tmem_st<16>(lane_addr + kColAHi + col, hi);
    tc::tmem_st<16>(lane_addr + kColALo + col, lo);
  }
  tc::tmem_st_wait();
  tc::fence_before_sync();
  tc::mbar_arrive(&bars.a_full[h]);
}

// gather warps: the unit's projected tiles, tensor memory -> P (rows of a subject start at a multiple of 8); warp of lane
// quarter q moves the 16 columns of group cg
__device__ __forceinline__ void drain_tiles(PipeBars& bars, const UnitTab& tab, uint32_t tmem, int q, int cg, int lane,
                                            unsigned char* s_p, uint32_t (&uses)[kMaxTiles]) {
  const int rows = tab.rows, nsub = tab.nsub, tiles = tab.tiles;
  for (int t = 0; t < tiles; ++t) {
    tc::mbar_wait(&bars.d_full[t], uses[t] & 1u);
    ++uses[t];
    tc::fence_after_sync();
    float v[16];
    tc::tmem_ld<16>(tmem + ((uint32_t)(32 * q) << 16) + kColD + (uint32_t)(kC * t + 16 * cg), v);
    tc::tmem_ld_wait();
    const int drow = t * kTR + 32 * q + lane;
    if (drow < rows) {
      int j = 0;
      while (j + 1 < nsub && drow >= tab.sub[j + 1].row) ++j;
      const int i = drow - tab.sub[j].row, prow = tab.sub[j].prow + i;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        *reinterpret_cast<float4*>(s_p + p_chunk_offset(prow, i, 4 * cg + k)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    }
    tc::fence_before_sync();
    __syncwarp();
    if (lane == 0) tc::mbar_arrive(&bars.d_free[t]);
  }
}

// sum_e w^_e P_src(e) of a row with descriptor d (zero for a lane without a row) in this lane's channel quad; the two
// rows of a pair (half warps) walk their records in lock step, 4 at a time up to the shorter row, then 2 at a time with
// zero weights (reading row 0) for the row that has ended
__device__ __forceinline__ float4 gather_row(int4 d, const int4* rec2, const unsigned char* pbase, uint32_t lane_const) {
  const int len = d.y - d.x;
  const int lmin = min(len, __shfl_xor_sync(kFull, len, 16)), lmax = max(len, __shfl_xor_sync(kFull, len, 16));
  const int4* rp = rec2 + (d.x >> 1);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  int k = 0;
#pragma unroll 1
  for (; k + 4 <= lmin; k += 4, rp += 2) {
    const int4 r = rp[0], s = rp[1];
    const float4 v0 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.x ^ lane_const));
    const float4 v1 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.z ^ lane_const));
    const float4 v2 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)s.x ^ lane_const));
    const float4 v3 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)s.z ^ lane_const));
    fma_quad(a, v0, __int_as_float(r.y));
    fma_quad(a, v1, __int_as_float(r.w));
    fma_quad(a, v2, __int_as_float(s.y));
    fma_quad(a, v3, __int_as_float(s.w));
  }
#pragma unroll 1
  for (; k < lmax; k += 2, ++rp) {
    int4 r = make_int4(0, 0, 0, 0);
    if (k < len) r = *rp;
    const float4 v0 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.x ^ lane_const));
    const float4 v1 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.z ^ lane_const));
    fma_quad(a, v0, __int_as_float(r.y));
    fma_quad(a, v1, __int_as_float(r.w));
  }
  return a;
}

// pooled readout: s_pool [subjects of the unit][16 warps][64].  Warp gw's share of subject j: the pair's two rows in a fixed
// order, one slot per (subject, warp)
__device__ __forceinline__ void pool_put(float* s_pool, int j, int gw, int lane, float4 pool) {
  pool.x += __shfl_xor_sync(kFull, pool.x, 16); pool.y += __shfl_xor_sync(kFull, pool.y, 16);
  pool.z += __shfl_xor_sync(kFull, pool.z, 16); pool.w += __shfl_xor_sync(kFull, pool.w, 16);
  if ((lane >> 4) == 0) *reinterpret_cast<float4*>(s_pool + ((size_t)j * kGathWarps + gw) * kC + 4 * (lane & 15)) = pool;
}
// subject j's sum of channel c over the 16 warps, in warp order: the same in every batch the subject is in
__device__ __forceinline__ float pool_sum(const float* s_pool, int j, int c) {
  float sum = 0.0f;
  for (int w = 0; w < kGathWarps; ++w) sum += s_pool[((size_t)j * kGathWarps + w) * kC + c];
  return sum;
}

// ---- host plan ---------------------------------------------------------------------------------------------------------
// subjects per unit before a launcher fits its shared memory: as many as the tiles hold, at most kMaxSub, and for small
// batches fewer, so that the units cover the SMs (16 x 84-node subjects: 16 CTAs of one tile each instead of 4 CTAs of
// three) - the launch is latency-bound there, not throughput-bound
inline int plan_spu(int max_nodes, long long num_graphs, int sm_count) {
  int spu = kMaxUnitRows / max_nodes;
  if (spu > kMaxSub) spu = kMaxSub;
  const long long fill = (num_graphs + sm_count - 1) / sm_count;
  if ((long long)spu > fill) spu = (int)fill;
  return spu < 1 ? 1 : spu;
}
// bytes of one blob buffer: the records of spu subjects of the largest shape
inline size_t plan_blob_cap(int spu, int max_nodes, int max_edges) {
  return (size_t)(((long long)spu * (agg_copy_words(max_nodes, max_edges) + 8) + 3) & ~3ll) * 4;
}

}  // namespace eng
}  // namespace cgnn
