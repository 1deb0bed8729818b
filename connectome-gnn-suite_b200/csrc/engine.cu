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
  UnitPlan plan;
  float* z; double* partials;
  // POOL variant (eval-mode last layer): emb[g] = mean_i relu2(z_i * scale2 + shift2); z itself is not written
  const float* scale2; const float* shift2; int relu2; float* emb;
  int o_stage, o_p, o_blob, o_const, o_tab, o_pool;   // byte offsets from the 1024-aligned base (W operands at 0)
};

struct Barriers {
  uint64_t stage_full[kNS], stage_free[kNS];
  PipeBars pipe;
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
  UnitTab* s_tab = reinterpret_cast<UnitTab*>(base + p.o_tab);   // [2]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- one-time setup ------------------------------------------------------------------------------------------
  if (warp == kWarpAlloc) tc::tmem_alloc(&tmem_base_s, kTmemCols);
  if (tid == 0) {
    for (int i = 0; i < kNS; ++i) { tc::mbar_init(&bars.stage_full[i], 1); tc::mbar_init(&bars.stage_free[i], 4 * 32); }
    init_pipe_bars(bars.pipe);
    tc::fence_mbar_init();
  }
  if (warp == kWarpTile && lane == 0) tc::prefetch_tensor_map(&tmap);
  stage_w_split(w_hi, w_lo, p.W, tid, kNT);
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
      for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x) {
        const Unit un = unit_geom(p.plan, u);
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
    if (lane == 0) blob_producer(p.plan, bars.pipe, s_blob);
  } else if (warp == kWarpMma) {
    // ================================ MMA issuer ===================================================================
    if (lane == 0) {
      const uint32_t idesc = tc::idesc_tf32(kTR, kC);
      const uint64_t b_hi = tc::smem_desc_sw128(tc::smem_u32(w_hi)), b_lo = tc::smem_desc_sw128(tc::smem_u32(w_lo));
      uint32_t tcount = 0, uses[kMaxTiles] = {0, 0, 0};
      for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x) {
        const Unit un = unit_geom(p.plan, u);
        for (int t = 0; t < un.tiles; ++t, ++tcount) mma_tile(bars.pipe, tmem, t, uses[t], tcount, idesc, b_hi, b_lo);
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
    for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x) {
      const Unit un = unit_geom(p.plan, u);
      for (int t = 0; t < un.tiles; ++t, ++tcount) {
        tc::mbar_wait(&bars.stage_full[h], tcount & 1u);
        float4 v[8];
        load_box_row(slot, row, v);
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
        store_a_row(bars.pipe, lane_addr, h, tcount, v);
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

    if (gw == 0 && (long long)blockIdx.x < p.plan.units) build_unit_tab(p.plan, blockIdx.x, s_tab, lane);
    tc::named_sync(1, kGathThreads);

    for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x, ++ucount) {
      const UnitTab& tab = s_tab[ucount & 1u];
      const int nsub = tab.nsub;
      drain_tiles(bars.pipe, tab, tmem, q, cg, lane, s_p, uses);
      const uint32_t b = ucount % (uint32_t)p.plan.nblob;
      tc::mbar_wait(&bars.pipe.blob_full[b], (ucount / (uint32_t)p.plan.nblob) & 1u);
      // the next unit's table goes into the other buffer now; it becomes visible at the barrier that ends this unit
      if (gw == 0 && u + gridDim.x < p.plan.units) build_unit_tab(p.plan, u + gridDim.x, &s_tab[(ucount + 1) & 1u], lane);
      tc::named_sync(1, kGathThreads);            // P is complete

      // ---- gather: half a warp per row, pairs of rows in lock step -------------------------------------------------
      const int32_t* blob = reinterpret_cast<const int32_t*>(s_blob + (size_t)b * p.plan.blob_cap_bytes);
      // POOL: pair k of a subject always goes to warp k % 16, whatever else shares the unit - the subject's sum is then
      // formed in the same order in every batch (eval logits are bit-identical under any batch split)
      const int n_outer = POOL ? nsub : 1;
      for (int jo = 0; jo < n_outer; ++jo) {
      float4 pool = make_float4(0.f, 0.f, 0.f, 0.f);
      const int g_lo = POOL ? tab.sub[jo].pair + gw : gw;
      const int g_hi = POOL ? tab.sub[jo].pair + ((tab.sub[jo].rows + 1) >> 1) : tab.groups;
      for (int gi = g_lo; gi < g_hi; gi += kGathWarps) {
        int j = POOL ? jo : 0;
        if (!POOL) while (j + 1 < nsub && gi >= tab.sub[j + 1].pair) ++j;
        const SubRec& e = tab.sub[j];
        const int n = e.rows, i = 2 * (gi - e.pair) + half;
        const bool valid = i < n;
        const int4* desc = reinterpret_cast<const int4*>(blob + e.blob);
        int4 d = make_int4(0, 0, 0, 0);
        if (valid) d = desc[i];
        float4 a = gather_row(d, desc + n, s_p + (size_t)e.prow * 256, lane_const);
        if (!valid) continue;
        a.x += bias4.x; a.y += bias4.y; a.z += bias4.z; a.w += bias4.w;
        if (POOL) {       // the next BatchNorm (running statistics) + ReLU on the value, straight into the subject's sum
          if (p.scale2) { a.x = fmaf(a.x, sc2.x, sh2.x); a.y = fmaf(a.y, sc2.y, sh2.y); a.z = fmaf(a.z, sc2.z, sh2.z); a.w = fmaf(a.w, sc2.w, sh2.w); }
          if (p.relu2) { a.x = fmaxf(a.x, 0.0f); a.y = fmaxf(a.y, 0.0f); a.z = fmaxf(a.z, 0.0f); a.w = fmaxf(a.w, 0.0f); }
          pool.x += a.x; pool.y += a.y; pool.z += a.z; pool.w += a.w;
          continue;
        }
        *reinterpret_cast<float4*>(p.z + (tab.row0 + e.row + i) * kC + 4 * cl) = a;
        if (want_stats) {
          if (cnt == 0) sh = a;
          cnt += 1;
          const float4 dv = make_float4(a.x - sh.x, a.y - sh.y, a.z - sh.z, a.w - sh.w);
          s1.x += dv.x; s1.y += dv.y; s1.z += dv.z; s1.w += dv.w;
          s2.x = fmaf(dv.x, dv.x, s2.x); s2.y = fmaf(dv.y, dv.y, s2.y); s2.z = fmaf(dv.z, dv.z, s2.z); s2.w = fmaf(dv.w, dv.w, s2.w);
        }
      }
      if (POOL) pool_put(s_pool, jo, gw, lane, pool);
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars.pipe.blob_free[b]);     // this warp has read its last record of the unit
      if (POOL) {
        tc::named_sync(1, kGathThreads);          // every warp's partial sums are in place
        for (int j = gw; j < nsub; j += kGathWarps)
          for (int c = lane; c < kC; c += 32)     // mean over the subject's rows (models.py:57-59)
            p.emb[(tab.g0 + j) * kC + c] = pool_sum(s_pool, j, c) / ((float)tab.sub[j].rows + 1e-8f);
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
  const int spu = plan_spu(max_nodes, num_graphs, dev.sm_count);
  a.plan.blob = csr->agg_in; a.plan.meta = csr->graph_meta; a.plan.B = num_graphs;
  a.plan.spu = spu;
  a.plan.units = (num_graphs + spu - 1) / spu;
  a.z = z; a.partials = partials;
  a.scale2 = (pool && act_out) ? act_out->scale : nullptr;
  a.shift2 = (pool && act_out) ? act_out->shift : nullptr;
  a.relu2 = (pool && act_out) ? act_out->relu : 0;
  a.emb = emb;
  // P rows: every subject starts at a multiple of 8
  const int p_rows = spu * ((max_nodes + 7) & ~7);
  const size_t blob_cap = plan_blob_cap(spu, max_nodes, max_edges);
  size_t off = (size_t)4 * kC * 128;                      // W hi / lo
  a.o_stage = (int)off; off += (size_t)kNS * kStageBytes;
  a.o_p = (int)off; off += (size_t)p_rows * 256;
  if (off < (size_t)a.o_p + (size_t)kGathThreads * 9 * 4) off = (size_t)a.o_p + (size_t)kGathThreads * 9 * 4;
  off = (off + 15) & ~(size_t)15;
  a.o_blob = (int)off;
  const size_t pool_bytes = pool ? (size_t)spu * kGathWarps * kC * 4 : 0;
  const size_t tail = (size_t)3 * kC * 4 + 2 * sizeof(UnitTab) + 32 + pool_bytes;
  const size_t limit = (size_t)dev.smem_optin - kStaticSmem;       // the kernel's static shared memory counts too
  int nblob = 2;
  if (off + 2 * blob_cap + tail + 1024 > limit) nblob = 1;
  if (off + (size_t)nblob * blob_cap + tail + 1024 > limit) return -1;
  a.plan.nblob = nblob;
  a.plan.blob_cap_bytes = (int)blob_cap;
  off += (size_t)nblob * blob_cap;
  a.o_const = (int)off; off += (size_t)3 * kC * 4;
  a.o_tab = (int)off; off += 2 * sizeof(UnitTab);
  off = (off + 15) & ~(size_t)15;
  a.o_pool = (int)off; off += pool_bytes;
  const size_t smem = off + 1024;
  long long grid = dev.sm_count;
  if (grid > a.plan.units) grid = a.plan.units;
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
