// eval_fused.cu - K9: the whole eval-mode network of a GCNConnectome in ONE kernel (reference train.py:56-68 forward,
// models.py:203-216 with BatchNorm in eval mode = a per-channel affine map, dropout off).
//
// In eval mode nothing couples two subjects (SURVEY 3.2), so a unit (one subject, or several small ones, <= 384 rows)
// runs through all L layers, the mean-pool readout and the MLP head without its activations ever leaving the SM:
// HBM sees the node features (4 N F bytes), the packed in-edge records and C logits per subject - 33 KB instead of
// 638 KB for a 360-node subject.
//
//   layer 1          gather warps: a_i = sum_e w^_e x_src(e) in the F (<= 8) input channels, z = a W1^T + b1 (FMAs)
//   layers 2..L      P = u W_l^T on the tensor core (3 x TF32, A operand in tensor memory), drained into the P tile,
//                    then z_i = sum_e w^_e P_src(e) + b_l by the gather warps - the roles of engine.cuh, except that
//                    the rows reach the converters through a shared-memory ring written by the PREVIOUS layer's
//                    epilogue (u = relu(scale z + shift)) instead of by TMA
//   readout + head   per-warp partial sums in a fixed order (the result does not depend on how subjects are batched),
//                    emb = sum / (N + 1e-8), logits = W1 relu(W0 emb + b0) + b1
//
// Roles: W loader (cp.async.bulk of the pre-split weight image of the next layer), blob loader, MMA issuer, 8 converter
// warps (ring -> TF32 hi/lo -> tcgen05.st), 16 gather warps.  Also runs on the test-only simulator.
#include "engine.cuh"

namespace cgnn {
namespace evf {
using namespace eng;

constexpr int kMaxLayers = 4;
constexpr int kFeat = 8;                   // input channels, padded
constexpr int kWImgBytes = 4 * kC * 128;   // one hidden layer's weights: hi | lo K-major operands
constexpr int kHeadMaxM = 64, kHeadMaxK = 8;

struct Args {
  const float* x; int F;
  const float* W1; const float* b1;          // first layer [64, F], [64]
  const unsigned char* wimg;                 // [L - 1][kWImgBytes]
  const float* hbias;                        // [L - 1][64]
  const float* affine;                       // [L][2][64] scale, shift of the eval-mode BatchNorm after every layer
  int L;
  const float* W0; const float* b0; const float* Wc; const float* bc; int M, K;   // head
  UnitPlan plan;
  float* emb; float* logits;
  int o_ring, o_p, o_blob, o_x, o_pool, o_const, o_head, o_tab;   // byte offsets from the 1024-aligned base (W buffer at 0)
};

struct EvalBarriers {
  uint64_t w_full, w_free;
  uint64_t ring_full[2], ring_free[2];
  PipeBars pipe;
};

struct PrepArgs {
  const float* W[kMaxLayers]; const float* bias[kMaxLayers];
  const float* gamma[kMaxLayers]; const float* beta[kMaxLayers]; const float* rmean[kMaxLayers]; const float* rvar[kMaxLayers];
  float eps[kMaxLayers];
  int L;
  unsigned char* wimg; float* hbias; float* affine;
};

// block b < L - 1: the K-major hi / lo image of hidden layer b + 2; block L - 1: the affine maps and hidden biases
__global__ void __launch_bounds__(256) k_eval_prep(PrepArgs p) {
  const int b = blockIdx.x, tid = threadIdx.x;
  if (b < p.L - 1) {
    unsigned char* hi = p.wimg + (size_t)b * kWImgBytes;
    stage_w_split(hi, hi + 2 * kC * 128, p.W[b + 1], tid, blockDim.x);
    return;
  }
  for (int idx = tid; idx < p.L * kC; idx += blockDim.x) {
    const int l = idx / kC, c = idx - l * kC;
    // same arithmetic as cgnn_bn_eval_affine (norm.cu)
    const float rstd = (float)(1.0 / sqrt((double)p.rvar[l][c] + (double)p.eps[l]));
    const float g = p.gamma[l] ? p.gamma[l][c] : 1.0f, be = p.beta[l] ? p.beta[l][c] : 0.0f;
    const float sc = g * rstd;
    p.affine[(2 * l) * kC + c] = sc;
    p.affine[(2 * l + 1) * kC + c] = be - p.rmean[l][c] * sc;
    if (l >= 1) p.hbias[(l - 1) * kC + c] = p.bias[l] ? p.bias[l][c] : 0.0f;
  }
}

__global__ void __launch_bounds__(kNT, 1) k_gcn_eval_fused(Args p) {
#ifdef CGNN_EMU
  CGNN_SMEM_DECL;
  unsigned char* smem_raw = cgnn_smem;
#else
  extern __shared__ __align__(1024) unsigned char smem_raw[];
#endif
  __shared__ EvalBarriers bars;
  __shared__ uint32_t tmem_base_s;
  unsigned char* base = tc::smem_align1024(smem_raw);
  unsigned char* w_hi = base;
  unsigned char* w_lo = base + 2 * kC * 128;
  unsigned char* s_ring = base + p.o_ring;          // [2 channel halves][128 rows][128 B], TMA-box swizzle
  unsigned char* s_p = base + p.o_p;
  unsigned char* s_blob = base + p.o_blob;
  float* s_x = reinterpret_cast<float*>(base + p.o_x);          // [unit rows][8]
  float* s_pool = reinterpret_cast<float*>(base + p.o_pool);    // [subjects][16 warps][64]
  float* s_b1 = reinterpret_cast<float*>(base + p.o_const);     // [64]
  float* s_w1 = s_b1 + kC;                                      // [8][64]: W1 transposed (input channel major)
  float* s_hb = s_w1 + kC * kFeat;                              // [L - 1][64]
  float* s_aff = s_hb + (kMaxLayers - 1) * kC;                  // [L][2][64]
  float* s_head = reinterpret_cast<float*>(base + p.o_head);    // W0 [M][64], b0 [M], Wc [K][M], bc [K], then [16 warps][64 + M]
  UnitTab* s_tab = reinterpret_cast<UnitTab*>(base + p.o_tab);  // [2]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int L = p.L, NH = p.L - 1;

  if (warp == kWarpAlloc) tc::tmem_alloc(&tmem_base_s, kTmemCols);
  if (tid == 0) {
    tc::mbar_init(&bars.w_full, 1); tc::mbar_init(&bars.w_free, 1);
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&bars.ring_full[i], kGathWarps); tc::mbar_init(&bars.ring_free[i], 4 * 32); }
    init_pipe_bars(bars.pipe);
    tc::fence_mbar_init();
  }
  for (int c = tid; c < kC; c += kNT) s_b1[c] = p.b1 ? p.b1[c] : 0.0f;
  for (int i = tid; i < kC * kFeat; i += kNT) { const int k = i >> 6, c = i & 63; s_w1[i] = k < p.F ? p.W1[c * p.F + k] : 0.0f; }
  for (int i = tid; i < NH * kC; i += kNT) s_hb[i] = p.hbias[i];
  for (int i = tid; i < L * 2 * kC; i += kNT) s_aff[i] = p.affine[i];
  if (p.logits) {
    const int M = p.M, K = p.K;
    float* w0 = s_head; float* b0 = w0 + M * kC; float* wc = b0 + M; float* bc = wc + K * M;
    for (int i = tid; i < M * kC; i += kNT) w0[i] = p.W0[i];
    for (int i = tid; i < M; i += kNT) b0[i] = p.b0[i];
    for (int i = tid; i < K * M; i += kNT) wc[i] = p.Wc[i];
    for (int i = tid; i < K; i += kNT) bc[i] = p.bc[i];
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_base_s;

  if (warp == kWarpTile) {
    // ================================ W loader =====================================================================
    if (lane == 0 && NH >= 1) {
      if (NH == 1) {                       // one hidden layer: its weights stay for the whole kernel
        tc::mbar_arrive_expect_tx(&bars.w_full, kWImgBytes);
        tc::bulk_load(w_hi, p.wimg, kWImgBytes, &bars.w_full);
      } else {
        uint32_t wq = 0;
        for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x)
          for (int hl = 0; hl < NH; ++hl, ++wq) {
            tc::mbar_wait(&bars.w_free, (wq & 1u) ^ 1u);    // the previous layer's MMAs no longer read the buffer
            tc::mbar_arrive_expect_tx(&bars.w_full, kWImgBytes);
            tc::bulk_load(w_hi, p.wimg + (size_t)hl * kWImgBytes, kWImgBytes, &bars.w_full);
          }
      }
    }
  } else if (warp == kWarpBlob) {
    // ================================ blob loader ==================================================================
    if (lane == 0) blob_producer(p.plan, bars.pipe, s_blob);
  } else if (warp == kWarpMma) {
    // ================================ MMA issuer ===================================================================
    if (lane == 0 && NH >= 1) {
      const uint32_t idesc = tc::idesc_tf32(kTR, kC);
      const uint64_t b_hi = tc::smem_desc_sw128(tc::smem_u32(w_hi)), b_lo = tc::smem_desc_sw128(tc::smem_u32(w_lo));
      uint32_t tq = 0, wq = 0, uses[kMaxTiles] = {0, 0, 0};
      for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x) {
        const Unit un = unit_geom(p.plan, u);
        for (int hl = 0; hl < NH; ++hl) {
          if (NH > 1 || wq == 0) { tc::mbar_wait(&bars.w_full, wq & 1u); ++wq; }
          for (int t = 0; t < un.tiles; ++t, ++tq) mma_tile(bars.pipe, tmem, t, uses[t], tq, idesc, b_hi, b_lo);
          if (NH > 1) tc::mma_commit(&bars.w_free);     // fires when this layer's last MMA has read the weights
        }
      }
    }
  } else if (warp >= kConvWarp0 && warp < kConvWarp0 + kConvWarps) {
    // ================================ converters: ring -> TF32 hi / lo -> tensor memory ============================
    const int q = warp & 3, h = (warp - kConvWarp0) >> 2;
    const int row = 32 * q + lane;
    const unsigned char* slot = s_ring + h * kStageBytes;
    const uint32_t lane_addr = tmem + ((uint32_t)(32 * q) << 16);
    uint32_t tq = 0;
    for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x) {
      const Unit un = unit_geom(p.plan, u);
      for (int hl = 0; hl < NH; ++hl)
        for (int t = 0; t < un.tiles; ++t, ++tq) {
          tc::mbar_wait(&bars.ring_full[h], tq & 1u);
          float4 v[8];
          load_box_row(slot, row, v);
          tc::mbar_arrive(&bars.ring_free[h]);
          store_a_row(bars.pipe, lane_addr, h, tq, v);
        }
    }
  } else if (warp >= kGathWarp0) {
    // ================================ gather warps =================================================================
    const int gw = warp - kGathWarp0, q = warp & 3, cg = gw >> 2;
    const int cl = lane & 15, half = lane >> 4;
    const int gt = tid - 32 * kGathWarp0;
    const uint32_t lane_const = (uint32_t)(((cl & 7) << 4) | ((cl & 8) << 4));
    const int M = p.M, K = p.K;
    const float4 b1q = *reinterpret_cast<const float4*>(s_b1 + 4 * cl);
    uint32_t ucount = 0, rq = 0, uses[kMaxTiles] = {0, 0, 0};   // rq: ring tiles written so far (all warps count alike)

    if (gw == 0 && (long long)blockIdx.x < p.plan.units) build_unit_tab(p.plan, blockIdx.x, s_tab, lane);
    tc::named_sync(1, kGathThreads);

    for (long long u = blockIdx.x; u < p.plan.units; u += gridDim.x, ++ucount) {
      const UnitTab& tab = s_tab[ucount & 1u];
      const int rows = tab.rows, nsub = tab.nsub, tiles = tab.tiles;
      const long long row0 = tab.row0, g0 = tab.g0;
      // ---- the unit's node features: [rows][8], zero padded --------------------------------------------------------
      for (int idx = gt; idx < rows * kFeat; idx += kGathThreads) {
        const int r = idx >> 3, k = idx & 7;
        s_x[idx] = k < p.F ? p.x[(row0 + r) * p.F + k] : 0.0f;
      }
      const uint32_t b = ucount % (uint32_t)p.plan.nblob;
      tc::mbar_wait(&bars.pipe.blob_full[b], (ucount / (uint32_t)p.plan.nblob) & 1u);
      if (gw == 0 && u + gridDim.x < p.plan.units) build_unit_tab(p.plan, u + gridDim.x, &s_tab[(ucount + 1) & 1u], lane);
      tc::named_sync(1, kGathThreads);
      const int32_t* blob = reinterpret_cast<const int32_t*>(s_blob + (size_t)b * p.plan.blob_cap_bytes);

      for (int l = 0; l < L; ++l) {          // l = 0: the narrow first layer; l >= 1: hidden layer over the P tile
        const bool last = l == L - 1;
        if (l >= 1) {
          // ---- drain this layer's projected tiles, tensor memory -> P ------------------------------------------------
          drain_tiles(bars.pipe, tab, tmem, q, cg, lane, s_p, uses);
        } else {
          // ---- first layer: P = x W1^T with plain FMAs (F <= 8 input channels), written like a drained tile ------------
          // (reference models.py:111 projects first as well; the gather below is the one every layer shares)
          float4 wq[kFeat];
#pragma unroll
          for (int k = 0; k < kFeat; ++k) wq[k] = *reinterpret_cast<const float4*>(s_w1 + k * kC + 4 * cl);
          for (int j = 0; j < nsub; ++j) {
            const SubRec& e = tab.sub[j];
            const int n = e.rows;
            for (int i = 2 * gw + half; i < n; i += 2 * kGathWarps) {
              const float* xr = s_x + (size_t)(e.row + i) * kFeat;
              const float4 xa = *reinterpret_cast<const float4*>(xr), xb = *reinterpret_cast<const float4*>(xr + 4);
              const float xv[kFeat] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
              float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
              for (int k = 0; k < kFeat; ++k) {
                o.x = fmaf(xv[k], wq[k].x, o.x); o.y = fmaf(xv[k], wq[k].y, o.y);
                o.z = fmaf(xv[k], wq[k].z, o.z); o.w = fmaf(xv[k], wq[k].w, o.w);
              }
              *reinterpret_cast<float4*>(s_p + p_chunk_offset(e.prow + i, i, cl)) = o;
            }
          }
        }
        tc::named_sync(1, kGathThreads);            // P is complete
        const float4 bq = l == 0 ? b1q : *reinterpret_cast<const float4*>(s_hb + (l - 1) * kC + 4 * cl);
        const float4 scq = *reinterpret_cast<const float4*>(s_aff + (2 * l) * kC + 4 * cl);
        const float4 shq = *reinterpret_cast<const float4*>(s_aff + (2 * l + 1) * kC + 4 * cl);
        int cur = -1;                               // ring tile this warp is writing (layers that feed a projection)
        auto advance_to = [&](int t) {              // every warp enters and leaves every tile of the layer exactly once
          while (cur < t) {
            if (cur >= 0) {
              __syncwarp();
              if (lane == 0) { tc::mbar_arrive(&bars.ring_full[0]); tc::mbar_arrive(&bars.ring_full[1]); }
            }
            ++cur;
            const uint32_t par = ((rq + (uint32_t)cur) & 1u) ^ 1u;     // the converters have read the slot's previous tile
            tc::mbar_wait(&bars.ring_free[0], par);
            tc::mbar_wait(&bars.ring_free[1], par);
          }
        };
        for (int j = 0; j < nsub; ++j) {
          const SubRec& e = tab.sub[j];
          const int n = e.rows;
          const int4* desc = reinterpret_cast<const int4*>(blob + e.blob);
          float4 pool = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int lp = gw; 2 * lp < n; lp += kGathWarps) {       // subject-local pairs: the same warp for the same row in any batch
            const int i = 2 * lp + half;
            const bool valid = i < n;
            int4 d = make_int4(0, 0, 0, 0);
            if (valid) d = desc[i];
            const float4 a = gather_row(d, desc + n, s_p + (size_t)e.prow * 256, lane_const);
            // z = a + b; u = relu(scale z + shift)   (GCN: conv -> BatchNorm -> ReLU, reference models.py:207-209)
            float4 uo;
            uo.x = fmaxf(fmaf(a.x + bq.x, scq.x, shq.x), 0.0f);
            uo.y = fmaxf(fmaf(a.y + bq.y, scq.y, shq.y), 0.0f);
            uo.z = fmaxf(fmaf(a.z + bq.z, scq.z, shq.z), 0.0f);
            uo.w = fmaxf(fmaf(a.w + bq.w, scq.w, shq.w), 0.0f);
            if (last) {
              if (valid) { pool.x += uo.x; pool.y += uo.y; pool.z += uo.z; pool.w += uo.w; }
            } else {
              // the row goes to the converters through the ring, in the layout a TMA box would have
              const int ur = e.row + (valid ? i : (n - 1));               // row of the unit
              const int t_mine = ur >> 7;
              const int t0 = __shfl_sync(kFull, t_mine, 0), t1 = __shfl_sync(kFull, t_mine, 16);
              const int hh = cl >> 3, jc = cl & 7, rr = ur & 127;
              unsigned char* dst = s_ring + hh * kStageBytes + tc::box_chunk_offset(rr, jc);
              advance_to(t0);
              if (valid && t_mine == t0) *reinterpret_cast<float4*>(dst) = uo;
              if (t1 != t0) {
                advance_to(t1);
                if (valid && t_mine == t1) *reinterpret_cast<float4*>(dst) = uo;
              }
            }
          }
          if (last) pool_put(s_pool, j, gw, lane, pool);
        }
        if (!last) {
          advance_to(tiles - 1);
          if (cur >= 0) {
            __syncwarp();
            if (lane == 0) { tc::mbar_arrive(&bars.ring_full[0]); tc::mbar_arrive(&bars.ring_full[1]); }
          }
          rq += (uint32_t)tiles;
          tc::named_sync(1, kGathThreads);          // every warp is done with P (and x): the next drain may overwrite it
        }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars.pipe.blob_free[b]);
      tc::named_sync(1, kGathThreads);              // the readout partials are complete; P, x and the blob are free

      // ---- mean-pool readout and MLP head: one warp per subject ------------------------------------------------------
      {
        const float* w0 = s_head; const float* b0 = w0 + M * kC; const float* wc = b0 + M; const float* bc = wc + K * M;
        float* my = s_head + M * kC + M + K * M + K + (size_t)gw * (kC + M);    // [64] emb, [M] hidden
        for (int j = gw; j < nsub; j += kGathWarps) {
          const float inv = 1.0f / ((float)tab.sub[j].rows + 1e-8f);          // reference models.py:40-47: sum / (count + 1e-8)
          for (int c = lane; c < kC; c += 32) {
            const float v = pool_sum(s_pool, j, c) * inv;
            my[c] = v;
            if (p.emb) p.emb[(g0 + j) * kC + c] = v;
          }
          __syncwarp();
          if (p.logits) {
            for (int m = 0; m < M; ++m) {                 // same loops as k_head_fwd (head.cu)
              float part = 0.0f;
              for (int c = lane; c < kC; c += 32) part = fmaf(w0[m * kC + c], my[c], part);
              const float hsum = fmaxf(warp_sum(part) + b0[m], 0.0f);
              if (lane == 0) my[kC + m] = hsum;
            }
            __syncwarp();
            for (int k = 0; k < K; ++k) {
              float part = 0.0f;
              for (int m = lane; m < M; m += 32) part = fmaf(wc[k * M + m], my[kC + m], part);
              const float v = warp_sum(part) + bc[k];
              if (lane == 0) p.logits[(g0 + j) * K + k] = v;
            }
          }
          __syncwarp();
        }
      }
      tc::named_sync(1, kGathThreads);              // s_pool is rewritten by the next unit
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == kWarpAlloc) tc::tmem_dealloc(tmem, kTmemCols);
}

}  // namespace evf

// Returns CGNN_OK when launched, -1 when the shape is not covered (the caller reports CGNN_ERR_UNSUPPORTED).
int launch_eval_fused(int kind, const float* x, int F, const cgnn_eval_layer_t* layers, int L, int H, const float* W0,
                      const float* b0, const float* Wc, const float* bc, int M, int K, const cgnn_csr_t* csr, int64_t num_graphs,
                      int32_t max_nodes, int32_t max_edges, float* emb, float* logits, void* workspace, size_t workspace_bytes,
                      cudaStream_t stream) {
  using namespace eng;
  using namespace evf;
  if (kind != AGG_GCN || !csr->agg_in || csr->agg_kind != AGG_GCN) return -1;
  if (H != kC || L < 2 || L > kMaxLayers || F < 1 || F > kFeat || M < 1 || M > kHeadMaxM || K < 1 || K > kHeadMaxK) return -1;
  if (max_nodes < 1 || max_nodes > kMaxUnitRows) return -1;
  for (int l = 1; l < L; ++l)
    if ((((uintptr_t)layers[l].W) & 15u) != 0) return -1;
  const DeviceInfo dev = device_info();
  const int NH = L - 1;
  // workspace: weight images, hidden biases, affine maps
  const size_t ws_need = (size_t)NH * kWImgBytes + (size_t)NH * kC * 4 + (size_t)L * 2 * kC * 4;
  if (!workspace || workspace_bytes < ws_need || (((uintptr_t)workspace) & 15u) != 0) return -1;
  PrepArgs pa{};
  for (int l = 0; l < L; ++l) {
    pa.W[l] = layers[l].W; pa.bias[l] = layers[l].bias; pa.gamma[l] = layers[l].gamma; pa.beta[l] = layers[l].beta;
    pa.rmean[l] = layers[l].running_mean; pa.rvar[l] = layers[l].running_var; pa.eps[l] = layers[l].eps;
    if (!layers[l].W || !layers[l].running_mean || !layers[l].running_var) return -1;
  }
  pa.L = L;
  pa.wimg = reinterpret_cast<unsigned char*>(workspace);
  pa.hbias = reinterpret_cast<float*>(pa.wimg + (size_t)NH * kWImgBytes);
  pa.affine = pa.hbias + (size_t)NH * kC;

  Args a{};
  a.x = x; a.F = F; a.W1 = layers[0].W; a.b1 = layers[0].bias;
  a.wimg = pa.wimg; a.hbias = pa.hbias; a.affine = pa.affine; a.L = L;
  a.W0 = W0; a.b0 = b0; a.Wc = Wc; a.bc = bc; a.M = M; a.K = K;
  a.plan.blob = csr->agg_in; a.plan.meta = csr->graph_meta; a.plan.B = num_graphs;
  a.emb = emb; a.logits = logits;
  int spu = plan_spu(max_nodes, num_graphs, dev.sm_count);
  size_t smem = 0;
  for (; spu >= 1; --spu) {         // the largest number of subjects per unit whose tiles, records and readout partials fit
    const int p_rows = spu * ((max_nodes + 7) & ~7);
    const size_t blob_cap = plan_blob_cap(spu, max_nodes, max_edges);
    size_t off = kWImgBytes;
    a.o_ring = (int)off; off += 2 * kStageBytes;
    a.o_p = (int)off; off += (size_t)p_rows * 256;
    off = (off + 15) & ~(size_t)15;
    a.o_x = (int)off; off += (size_t)spu * max_nodes * kFeat * 4;
    off = (off + 15) & ~(size_t)15;
    a.o_pool = (int)off; off += (size_t)spu * kGathWarps * kC * 4;
    a.o_const = (int)off; off += (size_t)(kC + kC * kFeat + (kMaxLayers - 1) * kC + kMaxLayers * 2 * kC) * 4;
    a.o_head = (int)off; off += (size_t)(M * kC + M + K * M + K + kGathWarps * (kC + M)) * 4;
    off = (off + 15) & ~(size_t)15;
    a.o_tab = (int)off; off += 2 * sizeof(UnitTab);
    off = (off + 15) & ~(size_t)15;
    a.o_blob = (int)off;
    const size_t limit = (size_t)dev.smem_optin - kStaticSmem;     // the kernel's static shared memory counts too
    int nblob = 2;
    if (off + 2 * blob_cap + 1024 > limit) nblob = 1;
    if (off + (size_t)nblob * blob_cap + 1024 > limit) continue;
    a.plan.nblob = nblob; a.plan.blob_cap_bytes = (int)blob_cap;
    smem = off + (size_t)nblob * blob_cap + 1024;
    break;
  }
  if (spu < 1) return -1;
  a.plan.spu = spu;
  a.plan.units = (num_graphs + spu - 1) / spu;
  long long grid = dev.sm_count;
  if (grid > a.plan.units) grid = a.plan.units;
  if (grid < 1) return -1;
  {
    auto kp = evf::k_eval_prep;
    CGNN_LAUNCH(kp, (unsigned)L, 256, 0, stream, pa);
    CGNN_CHECK_LAUNCH();
  }
  auto kfn = evf::k_gcn_eval_fused;
  cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  CGNN_LAUNCH(kfn, (unsigned)grid, kNT, smem, stream, a);
  CGNN_CHECK_LAUNCH();
  return CGNN_OK;
}

}  // namespace cgnn

extern "C" {

int cgnn_eval_fused_fwd(int32_t kind, const float* x, int32_t num_features, const cgnn_eval_layer_t* layers, int32_t num_layers,
                        int32_t H, const float* W0, const float* b0, const float* W1, const float* b1, int32_t M, int32_t K,
                        const cgnn_csr_t* csr, const int64_t* ptr, int64_t num_graphs, int64_t rows, int32_t max_nodes,
                        int32_t max_edges, float* emb, float* logits, void* workspace, size_t workspace_bytes,
                        cgnn_stream_t stream_) {
  (void)ptr;
  if (!layers || num_layers <= 0 || H <= 0 || num_graphs < 0 || rows < 0 || (!emb && !logits)) return CGNN_ERR_INVALID_ARG;
  if (num_graphs == 0) return CGNN_OK;
  if (!x || !csr || !csr->graph_meta) return CGNN_ERR_INVALID_ARG;
  if (logits && (!W0 || !b0 || !W1 || !b1)) return CGNN_ERR_INVALID_ARG;
  const int rc = cgnn::launch_eval_fused(kind, x, num_features, layers, num_layers, H, W0, b0, W1, b1, M, K, csr, num_graphs,
                                         max_nodes, max_edges, emb, logits, workspace, workspace_bytes, (cudaStream_t)stream_);
  return rc < 0 ? CGNN_ERR_UNSUPPORTED : rc;
}

}  // extern "C"
