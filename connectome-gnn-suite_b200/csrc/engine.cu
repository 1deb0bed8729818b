// engine.cu - warp-specialised hidden-layer forward (64 -> 64 channels), one persistent CTA per SM.
//
//   GCN (reference models.py:84-114 after models.py:208-210):   z = A^ (u W^T) + b,   u = dropout(relu(bn(t_in)))
//
// A UNIT is one subject, or several consecutive small subjects, of at most 384 rows.  Five roles run concurrently and
// hand tiles to each other through mbarriers, so the HBM stream, the tensor core and the shared-memory gather of
// different tiles / units overlap instead of taking turns:
//
//   tile producer   1 thread    TMA (cp.async.bulk.tensor, 128-byte swizzle): 128 rows x 32 channels of t_in per
//                               box into a two-slot staging ring
//   blob producer   1 thread    cp.async.bulk: the unit's packed in-edge records (agg.cuh) into the blob ring
//   converters      8 warps     thread = row: read the row's 32 channels from the staging slot (conflict-free
//                               thanks to the swizzle), apply BatchNorm/ReLU/dropout, split into TF32 hi/lo and
//                               store both straight into TENSOR MEMORY (tcgen05.st) - the A operand never
//                               touches shared memory
//   MMA issuer      1 thread    P = u W^T as 3 x TF32 tcgen05.mma with A from tensor memory, W^T hi/lo from
//                               shared memory, accumulators P[128 x 64] per tile in tensor memory
//   gather warps    16 warps    drain the unit's P tiles tensor memory -> shared memory (XOR-swizzled rows),
//                               then z_i = sum_e w^_e P_src(e) + dinv_i^2 P_i + b: half a warp per row, float4
//                               lanes, records two at a time; write z (coalesced), BatchNorm statistics
//
// Only t_in, the records and z cross HBM.  The same sources run on the test-only simulator (tc05.cuh).
#include "engine.cuh"

namespace cgnn {
namespace eng {

struct Args {
  Act act;
  const float* W; const float* bias;
  const int32_t* blob; const int32_t* meta;
  long long B, units;
  int spu;                 // subjects per unit
  int blob_cap_bytes;      // one blob buffer
  int nblob;               // 1 or 2 blob buffers
  float* z; double* partials;
  // POOL variant (eval-mode last layer): emb[g] = mean_i relu2(z_i * scale2 + shift2); z itself is not written
  const float* scale2; const float* shift2; int relu2; float* emb;
  int o_stage, o_p, o_blob, o_const, o_tab, o_pool;   // byte offsets from the 1024-aligned base (W operands at 0)
  __host__ __device__ UnitSrc src() const { return UnitSrc{meta, B, spu, blob_cap_bytes}; }
};

template <bool POOL>
__global__ void __launch_bounds__(kNT, 1) k_gcn_fwd_ws(const __grid_constant__ tc::TensorMap tmap, Args p) {
  act_salt(p.act);   // device-side dropout salt (CUDA-graph replays)
#ifdef CGNN_EMU
  CGNN_SMEM_DECL;
  unsigned char* smem_raw = cgnn_smem;
#else
  extern __shared__ __align__(1024) unsigned char smem_raw[];
#endif
  __shared__ Barriers bars;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  unsigned char* w_hi = base;                           // [2 K blocks][64 rows][128 B]
  unsigned char* w_lo = base + 2 * kC * 128;
  unsigned char* s_stage = base + p.o_stage;
  unsigned char* s_p = base + p.o_p;
  unsigned char* s_blob = base + p.o_blob;
  float* s_scale = reinterpret_cast<float*>(base + p.o_const);   // [64] scale, [64] shift, [64] bias
  float* s_shift = s_scale + kC;
  float* s_bias = s_shift + kC;
  int* s_tab = reinterpret_cast<int*>(base + p.o_tab);           // [2][kTabInts]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- one-time setup ------------------------------------------------------------------------------------------
  if (warp == kWarpAlloc) tc::tmem_alloc(&tmem_base_s, kTmemCols);
  if (tid == 0) {
    for (int i = 0; i < kNS; ++i) { tc::mbar_init(&bars.stage_full[i], 1); tc::mbar_init(&bars.stage_free[i], 4 * 32); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&bars.a_full[i], 4 * 32); tc::mbar_init(&bars.a_free[i], 1); }
    for (int i = 0; i < kMaxTiles; ++i) { tc::mbar_init(&bars.d_full[i], 1); tc::mbar_init(&bars.d_free[i], kGathWarps); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&bars.blob_full[i], 1); tc::mbar_init(&bars.blob_free[i], kGathWarps); }
    tc::fence_mbar_init();
  }
  if (warp == kWarpTile && lane == 0) tc::prefetch_tensor_map(&tmap);
  // W [64 out][64 in] -> K-major operand rows n = output channel, hi / lo parts
  for (int idx = tid; idx < kC * (kC / 4); idx += kNT) {
    const int n = idx / (kC / 4), k = (idx - n * (kC / 4)) * 4;
    tc::store_split4(w_hi, w_lo, n, k, kC, *reinterpret_cast<const float4*>(p.W + n * kC + k));
  }
  for (int c = tid; c < kC; c += kNT) {
    s_scale[c] = p.act.scale ? p.act.scale[c] : 1.0f;
    s_shift[c] = p.act.scale ? p.act.shift[c] : 0.0f;
    s_bias[c] = p.bias ? p.bias[c] : 0.0f;
  }
  tc::fence_proxy_async();        // the W operands are read by the tensor core (async proxy)
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_base_s;

  if (warp == kWarpTile) {
    // ================================ tile producer ================================================================
    if (lane == 0) {
      uint32_t tcount = 0;     // tiles issued so far: slot h of tile k is in its k-th use
      for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
        const Unit un = unit_geom(p.src(), u);
        for (int t = 0; t < un.tiles; ++t, ++tcount)
          for (int h = 0; h < 2; ++h) {
            tc::mbar_wait(&bars.stage_free[h], (tcount & 1u) ^ 1u);
            tc::mbar_arrive_expect_tx(&bars.stage_full[h], kStageBytes);
            tc::tma_load_box(s_stage + h * kStageBytes, &tmap, 32 * h, un.row0 + (long long)t * kTR, &bars.stage_full[h]);
          }
      }
    }
  } else if (warp == kWarpBlob) {
    // ================================ blob producer ================================================================
    if (lane == 0) {
      uint32_t ucount = 0;
      for (long long u = blockIdx.x; u < p.units; u += gridDim.x, ++ucount) {
        const Unit un = unit_geom(p.src(), u);
        const uint32_t b = ucount % (uint32_t)p.nblob, use = ucount / (uint32_t)p.nblob;
        tc::mbar_wait(&bars.blob_free[b], (use & 1u) ^ 1u);
        tc::mbar_arrive_expect_tx(&bars.blob_full[b], (uint32_t)un.blob_bytes);
        tc::bulk_load(s_blob + (size_t)b * p.blob_cap_bytes, p.blob + un.blob_word0, (uint32_t)un.blob_bytes, &bars.blob_full[b]);
      }
    }
  } else if (warp == kWarpMma) {
    // ================================ MMA issuer ===================================================================
    if (lane == 0) {
      const uint32_t idesc = tc::idesc_tf32(kTR, kC);
      const uint64_t b_hi = tc::smem_desc_sw128(tc::smem_u32(w_hi)), b_lo = tc::smem_desc_sw128(tc::smem_u32(w_lo));
      uint32_t tcount = 0, uses[kMaxTiles] = {0, 0, 0};
      for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
        const Unit un = unit_geom(p.src(), u);
        for (int t = 0; t < un.tiles; ++t, ++tcount) {
          tc::mbar_wait(&bars.d_free[t], (uses[t] & 1u) ^ 1u);     // the gather warps have drained this slot's previous tile
          ++uses[t];
          const uint32_t d = tmem + kColD + (uint32_t)(kC * t);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            tc::mbar_wait(&bars.a_full[h], tcount & 1u);
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
      }
    }
  } else if (warp >= kConvWarp0 && warp < kConvWarp0 + kConvWarps) {
    // ================================ converters ===================================================================
    const int q = warp & 3, h = (warp - kConvWarp0) >> 2;    // tensor-memory lane quarter, channel half
    const int row = 32 * q + lane;                           // row of the tile = tensor-memory lane
    const unsigned char* slot = s_stage + h * kStageBytes;
    const uint32_t lane_addr = tmem + ((uint32_t)(32 * q) << 16);
    const bool affine = p.act.scale != nullptr;
    uint32_t tcount = 0;
    for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
      const Unit un = unit_geom(p.src(), u);
      for (int t = 0; t < un.tiles; ++t, ++tcount) {
        tc::mbar_wait(&bars.stage_full[h], tcount & 1u);
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const float4*>(slot + tc::box_chunk_offset(row, j));
        tc::mbar_arrive(&bars.stage_free[h]);      // the values are in registers: the slot may be refilled
        const long long grow = un.row0 + (long long)t * kTR + row;
        const uint32_t rh = p.act.drop ? drop_row_hash(p.act, p.act.row_base + grow) : 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c0 = 32 * h + 4 * j;
          float y[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
          if (affine) {
            const float4 sc = *reinterpret_cast<const float4*>(s_scale + c0), sh = *reinterpret_cast<const float4*>(s_shift + c0);
            y[0] = fmaf(y[0], sc.x, sh.x); y[1] = fmaf(y[1], sc.y, sh.y); y[2] = fmaf(y[2], sc.z, sh.z); y[3] = fmaf(y[3], sc.w, sh.w);
          }
          if (p.act.relu) {
#pragma unroll
            for (int e = 0; e < 4; ++e) y[e] = fmaxf(y[e], 0.0f);
          }
          if (p.act.drop) {
            const uint32_t keep = drop_keep4(p.act, rh, drop_quad_key(p.act, c0 >> 2));
#pragma unroll
            for (int e = 0; e < 4; ++e) y[e] = ((keep >> e) & 1u) ? y[e] * p.act.keep_scale : 0.0f;
          }
          v[j] = make_float4(y[0], y[1], y[2], y[3]);
        }
        tc::mbar_wait(&bars.a_free[h], (tcount & 1u) ^ 1u);    // the MMAs that read these columns for the previous tile are done
        tc::fence_after_sync();
#pragma unroll
        for (int part = 0; part < 2; ++part) {
          float hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float4 h, l;
            tc::split4(v[4 * part + j], h, l);
            hi[4 * j + 0] = h.x; hi[4 * j + 1] = h.y; hi[4 * j + 2] = h.z; hi[4 * j + 3] = h.w;
            lo[4 * j + 0] = l.x; lo[4 * j + 1] = l.y; lo[4 * j + 2] = l.z; lo[4 * j + 3] = l.w;
          }
          const uint32_t col = (uint32_t)(32 * h + 16 * part);
          tc::tmem_st<16>(lane_addr + kColAHi + col, hi);
          tc::tmem_st<16>(lane_addr + kColALo + col, lo);
        }
        tc::tmem_st_wait();
        tc::fence_before_sync();
        tc::mbar_arrive(&bars.a_full[h]);
      }
    }
  } else if (warp >= kGathWarp0) {
    // ================================ gather warps =================================================================
    const int gw = warp - kGathWarp0, q = warp & 3, cg = gw >> 2;   // lane quarter and 16-column group of the drain
    const int cl = lane & 15, half = lane >> 4;                     // gather: channel quad, which row of the pair
    const uint32_t lane_const = (uint32_t)(((cl & 7) << 4) | ((cl & 8) << 4));
    const float4 bias4 = *reinterpret_cast<const float4*>(s_bias + 4 * cl);
    float4 sc2 = make_float4(1.f, 1.f, 1.f, 1.f), sh2 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (POOL && p.scale2) { sc2 = *reinterpret_cast<const float4*>(p.scale2 + 4 * cl); sh2 = *reinterpret_cast<const float4*>(p.shift2 + 4 * cl); }
    float* s_pool = reinterpret_cast<float*>(base + p.o_pool);      // [subjects per unit][16 warps][64]
    const bool want_stats = p.partials != nullptr;
    // BatchNorm statistics of this thread's channel quad as shifted sums: s1 = sum (z - c), s2 = sum (z - c)^2 with
    // c = the thread's first value (no cancellation: |z - c| is of the order of the spread); turned into
    // {count, mean, M2} in double at the end.  6 packed instructions per row instead of 16 for a Welford update.
    float4 sh = make_float4(0.f, 0.f, 0.f, 0.f), s1 = sh, s2 = sh;
    int cnt = 0;
    uint32_t ucount = 0, uses[kMaxTiles] = {0, 0, 0};

    // unit table: header {rows, nsub, groups, tiles, row0 lo, row0 hi, -, -}, then per subject
    // {first row in the tiles, first row in P (8-aligned), rows, blob word offset, first flat pair index, -, -, -}
    auto build_table = [&](long long u, int* tab) {
      const Unit un = unit_geom(p.src(), u);
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
        int* e = tab + 8 + 8 * lane;
        e[0] = (int)(m.x - un.row0);
        e[1] = pincl - ((n + 7) & ~7);
        e[2] = n;
        e[3] = (int)(agg_base_words(m.x, m.z, un.g0 + lane) - un.blob_word0);
        e[4] = gincl - ((n + 1) >> 1);
      }
      if (lane == 0) {
        tab[0] = un.rows; tab[1] = un.nsub; tab[2] = groups; tab[3] = un.tiles;
        tab[4] = (int)(un.row0 & 0xffffffffll); tab[5] = (int)(un.row0 >> 32);
        tab[6] = (int)un.g0;
      }
    };
    if (gw == 0 && (long long)blockIdx.x < p.units) build_table(blockIdx.x, s_tab);
    tc::named_sync(1, kGathThreads);

    for (long long u = blockIdx.x; u < p.units; u += gridDim.x, ++ucount) {
      const int* tab = s_tab + (ucount & 1u) * kTabInts;
      const int rows = tab[0], nsub = tab[1], groups = tab[2], tiles = tab[3];
      const long long row0 = (long long)(uint32_t)tab[4] | ((long long)tab[5] << 32);
      // ---- drain: the unit's projected tiles, tensor memory -> P (rows of a subject start at a multiple of 8) ----
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
          while (j + 1 < nsub && drow >= tab[8 + 8 * (j + 1)]) ++j;
          const int i = drow - tab[8 + 8 * j], prow = tab[8 + 8 * j + 1] + i;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(s_p + p_chunk_offset(prow, i, 4 * cg + k)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
        }
        tc::fence_before_sync();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&bars.d_free[t]);
      }
      const uint32_t b = ucount % (uint32_t)p.nblob;
      tc::mbar_wait(&bars.blob_full[b], (ucount / (uint32_t)p.nblob) & 1u);
      // the next unit's table goes into the other buffer now; it becomes visible at the barrier that ends this unit
      if (gw == 0 && u + gridDim.x < p.units) build_table(u + gridDim.x, s_tab + ((ucount + 1) & 1u) * kTabInts);
      tc::named_sync(1, kGathThreads);            // P is complete

      // ---- gather: half a warp per row, pairs of rows in lock step -------------------------------------------------
      const int32_t* blob = reinterpret_cast<const int32_t*>(s_blob + (size_t)b * p.blob_cap_bytes);
      // POOL: pair k of a subject always goes to warp k % 16, whatever else shares the unit - the subject's sum is then
      // formed in the same order in every batch (eval logits are bit-identical under any batch split)
      const int n_outer = POOL ? nsub : 1;
      for (int jo = 0; jo < n_outer; ++jo) {
      float4 pool = make_float4(0.f, 0.f, 0.f, 0.f);
      const int g_lo = POOL ? tab[8 + 8 * jo + 4] + gw : gw;
      const int g_hi = POOL ? tab[8 + 8 * jo + 4] + ((tab[8 + 8 * jo + 2] + 1) >> 1) : groups;
      for (int gi = g_lo; gi < g_hi; gi += kGathWarps) {
        int j = POOL ? jo : 0;
        if (!POOL) while (j + 1 < nsub && gi >= tab[8 + 8 * (j + 1) + 4]) ++j;
        const int* e = tab + 8 + 8 * j;
        const int n = e[2], i = 2 * (gi - e[4]) + half;
        const bool valid = i < n;
        const int4* desc = reinterpret_cast<const int4*>(blob + e[3]);
        const int4* rec2 = reinterpret_cast<const int4*>(blob + e[3] + 4 * n);
        int4 d = make_int4(0, 0, 0, 0);
        if (valid) d = desc[i];
        const int len = d.y - d.x;
        const int lmin = min(len, __shfl_xor_sync(kFull, len, 16)), lmax = max(len, __shfl_xor_sync(kFull, len, 16));
        const unsigned char* pbase = s_p + (size_t)e[1] * 256;
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
        for (; k < lmax; k += 2, ++rp) {      // rows that have ended contribute zero weights (and read row 0)
          int4 r = make_int4(0, 0, 0, 0);
          if (k < len) r = *rp;
          const float4 v0 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.x ^ lane_const));
          const float4 v1 = *reinterpret_cast<const float4*>(pbase + ((uint32_t)r.z ^ lane_const));
          fma_quad(a, v0, __int_as_float(r.y));
          fma_quad(a, v1, __int_as_float(r.w));
        }
        if (!valid) continue;
        a.x += bias4.x; a.y += bias4.y; a.z += bias4.z; a.w += bias4.w;
        if (POOL) {       // the next BatchNorm (running statistics) + ReLU on the value, straight into the subject's sum
          if (p.scale2) { a.x = fmaf(a.x, sc2.x, sh2.x); a.y = fmaf(a.y, sc2.y, sh2.y); a.z = fmaf(a.z, sc2.z, sh2.z); a.w = fmaf(a.w, sc2.w, sh2.w); }
          if (p.relu2) { a.x = fmaxf(a.x, 0.0f); a.y = fmaxf(a.y, 0.0f); a.z = fmaxf(a.z, 0.0f); a.w = fmaxf(a.w, 0.0f); }
          pool.x += a.x; pool.y += a.y; pool.z += a.z; pool.w += a.w;
          continue;
        }
        *reinterpret_cast<float4*>(p.z + (row0 + e[0] + i) * kC + 4 * cl) = a;
        if (want_stats) {
          if (cnt == 0) sh = a;
          cnt += 1;
          const float4 dv = make_float4(a.x - sh.x, a.y - sh.y, a.z - sh.z, a.w - sh.w);
          s1.x += dv.x; s1.y += dv.y; s1.z += dv.z; s1.w += dv.w;
          s2.x = fmaf(dv.x, dv.x, s2.x); s2.y = fmaf(dv.y, dv.y, s2.y); s2.z = fmaf(dv.z, dv.z, s2.z); s2.w = fmaf(dv.w, dv.w, s2.w);
        }
      }
      if (POOL) {       // this warp's share of subject jo: even rows + odd rows, one slot per (subject, warp)
        pool.x += __shfl_xor_sync(kFull, pool.x, 16); pool.y += __shfl_xor_sync(kFull, pool.y, 16);
        pool.z += __shfl_xor_sync(kFull, pool.z, 16); pool.w += __shfl_xor_sync(kFull, pool.w, 16);
        if (half == 0) *reinterpret_cast<float4*>(s_pool + ((size_t)jo * kGathWarps + gw) * kC + 4 * cl) = pool;
      }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars.blob_free[b]);     // this warp has read its last record of the unit
      if (POOL) {
        tc::named_sync(1, kGathThreads);          // every warp's partial sums are in place
        const long long g0 = (long long)tab[6];
        for (int j = gw; j < nsub; j += kGathWarps) {
          // mean over the subject's rows (models.py:57-59)
          for (int c = lane; c < kC; c += 32) {
            float sum = 0.0f;
            for (int w = 0; w < kGathWarps; ++w) sum += s_pool[((size_t)j * kGathWarps + w) * kC + c];
            p.emb[(g0 + j) * kC + c] = sum / ((float)tab[8 + 8 * j + 2] + 1e-8f);
          }
        }
      }
      tc::named_sync(1, kGathThreads);            // every warp is done with P: the next drain may overwrite it
    }

    // ---- BatchNorm statistics of this CTA: {count, mean[64], M2[64]} as doubles --------------------------------------
    if (want_stats) {
      float* rec = reinterpret_cast<float*>(s_p);   // [kGathThreads][9]
      const int gt = tid - 32 * kGathWarp0;
      rec[gt * 9] = (float)cnt;
      {
        const float shv[4] = {sh.x, sh.y, sh.z, sh.w}, s1v[4] = {s1.x, s1.y, s1.z, s1.w}, s2v[4] = {s2.x, s2.y, s2.z, s2.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double n_ = cnt > 0 ? (double)cnt : 1.0, m1 = (double)s1v[j] / n_;
          rec[gt * 9 + 1 + j] = (float)((double)shv[j] + m1);
          rec[gt * 9 + 5 + j] = (float)fmax((double)s2v[j] - (double)s1v[j] * m1, 0.0);
        }
      }
      tc::named_sync(1, kGathThreads);
      cta_write_quad_stats(rec, kGathThreads, 16, kC, gt, p.partials + (size_t)blockIdx.x * (1 + 2 * kC));
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == kWarpAlloc) tc::tmem_dealloc(tmem, kTmemCols);
}

}  // namespace eng

#ifndef CGNN_EMU
// ---- host: tensor-map encoder through the runtime's driver entry point (no -lcuda) ---------------------------------
namespace tc {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}
int make_tensor_map(TensorMap* m, const float* base, long long rows, int cols, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return CGNN_ERR_CUDA;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)kBoxCols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? CGNN_OK : CGNN_ERR_CUDA;
}
}  // namespace tc
#endif

// Returns CGNN_OK when launched (grid in *grid_out: the caller merges `partials`), -1 when the shape is not covered.
// emb != nullptr: the POOL variant - act_out (BatchNorm affine + ReLU of the layer's output, no dropout) and the mean-pool
// readout are applied in the epilogue, emb [num_graphs, 64] is written instead of z.
static int launch_ws(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                     int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z,
                     double* partials, const cgnn_act_t* act_out, float* emb, int* grid_out, size_t workspace_bytes,
                     cudaStream_t stream) {
  using namespace eng;
  if (!csr->agg_in || csr->agg_kind != AGG_GCN) return -1;
  if (d_in != kC || H != kC) return -1;
  if (max_nodes < 1 || max_nodes > kMaxUnitRows) return -1;
  if ((((uintptr_t)t_in) & 15u) != 0 || (z && (((uintptr_t)z) & 15u) != 0) || (((uintptr_t)W) & 15u) != 0) return -1;
  const bool pool = emb != nullptr;
  if (pool && act_out && act_out->p_drop > 0.0f) return -1;       // eval mode only
  if (pool && act_out && act_out->scale && ((((uintptr_t)act_out->scale) & 15u) != 0 || (((uintptr_t)act_out->shift) & 15u) != 0)) return -1;
  const DeviceInfo dev = device_info();
  Args a;
  a.act = make_act(act); a.W = W; a.bias = bias;
  a.blob = csr->agg_in; a.meta = csr->graph_meta; a.B = num_graphs;
  int spu = kMaxUnitRows / max_nodes;
  if (spu > kMaxSub) spu = kMaxSub;
  // small batches: fewer subjects per unit so that the units cover the SMs (16 x 84-node subjects: 16 CTAs of one tile each
  // instead of 4 CTAs of three) - the launch is latency-bound there, not throughput-bound
  {
    const long long fill = (num_graphs + dev.sm_count - 1) / dev.sm_count;
    if ((long long)spu > fill) spu = (int)fill;
  }
  if (spu < 1) spu = 1;
  a.spu = spu;
  a.units = (num_graphs + spu - 1) / spu;
  a.z = z; a.partials = partials;
  a.scale2 = (pool && act_out) ? act_out->scale : nullptr;
  a.shift2 = (pool && act_out) ? act_out->shift : nullptr;
  a.relu2 = (pool && act_out) ? act_out->relu : 0;
  a.emb = emb;
  // P rows: every subject starts at a multiple of 8
  const int p_rows = spu * ((max_nodes + 7) & ~7);
  const size_t blob_cap = (size_t)(((long long)spu * (agg_copy_words(max_nodes, max_edges) + 8) + 3) & ~3ll) * 4;
  size_t off = (size_t)4 * kC * 128;                      // W hi / lo
  a.o_stage = (int)off; off += (size_t)kNS * kStageBytes;
  a.o_p = (int)off; off += (size_t)p_rows * 256;
  if (off < (size_t)a.o_p + (size_t)kGathThreads * 9 * 4) off = (size_t)a.o_p + (size_t)kGathThreads * 9 * 4;
  off = (off + 15) & ~(size_t)15;
  a.o_blob = (int)off;
  const size_t pool_bytes = pool ? (size_t)spu * kGathWarps * kC * 4 : 0;
  const size_t tail = (size_t)3 * kC * 4 + (size_t)2 * kTabInts * 4 + 32 + pool_bytes;
  const size_t limit = (size_t)dev.smem_optin - kStaticSmem;       // the kernel's static shared memory counts too
  int nblob = 2;
  if (off + 2 * blob_cap + tail + 1024 > limit) nblob = 1;
  if (off + (size_t)nblob * blob_cap + tail + 1024 > limit) return -1;
  a.nblob = nblob;
  a.blob_cap_bytes = (int)blob_cap;
  off += (size_t)nblob * blob_cap;
  a.o_const = (int)off; off += (size_t)3 * kC * 4;
  a.o_tab = (int)off; off += (size_t)2 * kTabInts * 4;
  off = (off + 15) & ~(size_t)15;
  a.o_pool = (int)off; off += pool_bytes;
  const size_t smem = off + 1024;
  long long grid = dev.sm_count;
  if (grid > a.units) grid = a.units;
  if (partials) {
    const size_t rec = (size_t)(1 + 2 * kC) * sizeof(double);
    if ((size_t)grid * rec > workspace_bytes) grid = (long long)(workspace_bytes / rec);
  }
  if (grid < 1) return -1;
  *grid_out = (int)grid;
  tc::TensorMap tmap;
  if (tc::make_tensor_map(&tmap, t_in, rows, kC, kTR) != CGNN_OK) return -1;
  if (pool) {
    auto kfn = k_gcn_fwd_ws<true>;
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    CGNN_LAUNCH(kfn, (unsigned)grid, kNT, smem, stream, tmap, a);
  } else {
    auto kfn = k_gcn_fwd_ws<false>;
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    CGNN_LAUNCH(kfn, (unsigned)grid, kNT, smem, stream, tmap, a);
  }
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

int launch_gcn_fwd_ws(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                      int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z,
                      double* partials, int* grid_out, size_t workspace_bytes, cudaStream_t stream) {
  return launch_ws(t_in, act, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, z, partials, nullptr, nullptr, grid_out,
                   workspace_bytes, stream);
}

int launch_gcn_fwd_ws_pool(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                           int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges,
                           const cgnn_act_t* act_out, float* emb, cudaStream_t stream) {
  int grid = 0;
  return launch_ws(t_in, act, W, bias, csr, num_graphs, rows, d_in, H, max_nodes, max_edges, nullptr, nullptr, act_out, emb, &grid, 0,
                   stream);
}

}  // namespace cgnn
