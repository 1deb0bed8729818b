// engine.cuh - shared pieces of the warp-specialised kernels (engine.cu: one hidden layer; eval_fused.cu: the whole
// network in eval mode): role layout, tensor-memory column plan, unit geometry, the P-tile swizzle.
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
constexpr int kTabInts = 8 + 8 * kMaxSub;   // header + per-subject records of the unit table
constexpr size_t kStaticSmem = 1024;        // barriers + tensor-memory address, rounded up by the alignment of the dynamic part


struct Barriers {
  uint64_t stage_full[kNS], stage_free[kNS];
  uint64_t a_full[2], a_free[2];
  uint64_t d_full[kMaxTiles], d_free[kMaxTiles];
  uint64_t blob_full[2], blob_free[2];
};

// geometry of unit u, from the per-subject records {first row, rows, first edge, edges}
struct Unit {
  long long g0; int nsub;
  long long row0; int rows, tiles;
  long long blob_word0; int blob_bytes;
};
// what unit_geom needs from a kernel's arguments
struct UnitSrc {
  const int32_t* meta; long long B; int spu; int blob_cap_bytes;
};
__device__ __forceinline__ Unit unit_geom(const UnitSrc& p, long long u) {
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

// byte offset of 16-byte chunk c (0..15) of row `prow` of the P tile; `key` = the row's index inside its subject
__device__ __forceinline__ uint32_t p_chunk_offset(int prow, int key, int c) {
  return (uint32_t)(prow * 256 + ((((c ^ key) & 7) | (c & 8)) << 4));
}


}  // namespace eng
}  // namespace cgnn
