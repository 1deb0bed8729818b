// agg.cuh - packed per-subject aggregation blobs and the warp-per-row gather over them.
//
// The generic kernels walk {rowptr, col, w} arrays: three dependent scalar loads per edge.  Measured on B200
// (tools/ubench/ldtm_gather.cu) every LSU instruction costs ~1.9 issue cycles per SM whatever its width, so the
// tensor-core generation of kernels reads the structure as 16-byte records instead:
//   row descriptor  int4 {rec_begin, rec_end, aux bits, row}        one broadcast load per row
//   record pair     int4 {nbr0, w0 bits, nbr1, w1 bits}             one broadcast load per two edges
// Rows are padded to an even number of records (zero weight), GCN rows end with their self-loop record.
// Descriptor k stands for row k (its fourth word repeats k).  Measured on B200 and dropped: descriptors sorted by record
// count, so that rows walked in lock step have equal lengths - the ranking cost the collate kernel 17 % of its time and the
// gathers did not get faster (352 us per layer either way).
// The neighbour word of the by-destination blob (agg_in) is stored as agg_rec_x(nbr) = the byte offset of the
// neighbour's row in a 256-byte-pitch tile with its XOR-swizzle key (row & 7) in the 16-byte-chunk bits: the
// warp-specialised forward kernels (engine.cu) turn it into a shared-memory address with one XOR.  Everybody else
// takes agg_rec_row().  The by-source blob (agg_out) carries plain row indices.
#pragma once
#include "common.cuh"

namespace cgnn {

enum { AGG_GCN = 0, AGG_SAGE = 1 };

static inline __host__ __device__ int agg_rec_x(int nbr) { return (nbr << 8) | ((nbr & 7) << 4); }
static inline __host__ __device__ int agg_rec_row(int x) { return x >> 8; }

// word offset of subject g's blob: 8 words per row + 2 per edge (edge base rounded up to even) + 4 per subject;
// a blob uses at most 4n (descriptors) + 2(m + 2n) (records incl. self-loop and padding) words.
static inline __host__ __device__ long long agg_base_words(long long nb, long long eb, long long g) {
  return 8 * nb + 2 * (eb + (eb & 1)) + 4 * g;
}
static inline size_t agg_total_words(long long rows, long long edges, long long graphs) {
  return (size_t)(8 * rows + 2 * (edges + 1) + 4 * graphs + 8);
}

// ---- gather over a blob staged in shared memory -------------------------------------------------------------------
// words a CTA copies for one subject: descriptors + records + padding, always inside the blob buffer (the next blob
// starts 8n + 2m (+2) + 4 words further, agg_total_words adds 8 words of slack at the end)
static inline __host__ __device__ int agg_copy_words(int n, int m) { return 8 * n + 2 * m + 4; }
static inline __host__ __device__ int agg_smem_words(int max_nodes, int max_edges) { return 8 * max_nodes + 2 * max_edges + 8; }

// One warp, 32 / LPR consecutive rows at a time: lane owns the channel quad (lane % LPR) of row i0 + lane / LPR and
// returns acc = sum over that row's records of w * tile[nbr][quad] (tile rows are LPR float4 wide), the row's aux
// word and whether the row exists.  Records are read two at a time (rows are padded to an even count); the rows of a
// group run in lock step up to the shortest one, the remainder is predicated.
// acc += w * v on a channel quad.  Device build: two packed fp32 FMAs (fma.rn.f32x2 -> FFMA2 with the weight as a
// broadcast scalar) - the same IEEE fused multiply-adds as four FFMAs, half the issue slots.
__device__ __forceinline__ void fma_quad(float4& a, const float4& v, float w) {
#ifdef CGNN_EMU
  a.x = fmaf(v.x, w, a.x); a.y = fmaf(v.y, w, a.y); a.z = fmaf(v.z, w, a.z); a.w = fmaf(v.w, w, a.w);
#else
  float2 a0 = make_float2(a.x, a.y), a1 = make_float2(a.z, a.w);
  const float2 v0 = make_float2(v.x, v.y), v1 = make_float2(v.z, v.w), w2 = make_float2(w, w);
  unsigned long long d0 = reinterpret_cast<unsigned long long&>(a0), d1 = reinterpret_cast<unsigned long long&>(a1);
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d0) : "l"(reinterpret_cast<const unsigned long long&>(v0)), "l"(reinterpret_cast<const unsigned long long&>(w2)));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d1) : "l"(reinterpret_cast<const unsigned long long&>(v1)), "l"(reinterpret_cast<const unsigned long long&>(w2)));
  a0 = reinterpret_cast<float2&>(d0); a1 = reinterpret_cast<float2&>(d1);
  a = make_float4(a0.x, a0.y, a1.x, a1.y);
#endif
}

// the channel quad of tile row `nbr` for this lane: one shared-space address = one multiply-add per record
struct TileQuads {
#ifdef CGNN_EMU
  const float4* t4; int pitch;
  __device__ __forceinline__ float4 at(int nbr) const { return t4[nbr * pitch]; }
#else
  uint32_t base, pitch_bytes;
  __device__ __forceinline__ float4 at(int nbr) const {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(base + (uint32_t)nbr * pitch_bytes));
    return v;
  }
#endif
};
__device__ __forceinline__ TileQuads tile_quads(const float4* t4, int pitch) {
#ifdef CGNN_EMU
  return TileQuads{t4, pitch};
#else
  return TileQuads{(uint32_t)__cvta_generic_to_shared(t4), (uint32_t)pitch * 16u};
#endif
}

// PRE: the records' neighbour words are agg_rec_x() encoded (agg_in); false: plain row indices (agg_out)
template <int LPR, int PITCH = LPR, bool PRE = true>
static __device__ __forceinline__ bool agg_gather_group(const int4* __restrict__ s_desc, const int4* __restrict__ s_rec2,
                                                        const float4* __restrict__ tile4, int i0, int n, float4& acc, float& aux,
                                                        int& row) {
  const int lane = threadIdx.x & 31, cl = lane % LPR;
  row = i0 + lane / LPR;
  const bool valid = row < n;
  int4 d = make_int4(0, 0, 0, 0);
  if (valid) d = s_desc[row];
  const int len = d.y - d.x;
  int lmin = len, lmax = len;
#pragma unroll
  for (int o = LPR; o < 32; o <<= 1) {
    lmin = min(lmin, __shfl_xor_sync(kFull, lmin, o));
    lmax = max(lmax, __shfl_xor_sync(kFull, lmax, o));
  }
  const TileQuads t = tile_quads(tile4 + cl, PITCH);
  const int4* rp = s_rec2 + (d.x >> 1);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  int k = 0;
#pragma unroll 1
  for (; k + 4 <= lmin; k += 4, rp += 2) {   // four records per step: half the loop overhead, four tile loads in flight
    const int4 r = rp[0], s = rp[1];
    const float4 v0 = t.at(PRE ? agg_rec_row(r.x) : r.x), v1 = t.at(PRE ? agg_rec_row(r.z) : r.z);
    const float4 v2 = t.at(PRE ? agg_rec_row(s.x) : s.x), v3 = t.at(PRE ? agg_rec_row(s.z) : s.z);
    fma_quad(a, v0, __int_as_float(r.y));
    fma_quad(a, v1, __int_as_float(r.w));
    fma_quad(a, v2, __int_as_float(s.y));
    fma_quad(a, v3, __int_as_float(s.w));
  }
#pragma unroll 1
  for (; k < lmin; k += 2, ++rp) {        // every row of the group has these records
    const int4 r = *rp;
    const float4 v0 = t.at(PRE ? agg_rec_row(r.x) : r.x), v1 = t.at(PRE ? agg_rec_row(r.z) : r.z);
    fma_quad(a, v0, __int_as_float(r.y));
    fma_quad(a, v1, __int_as_float(r.w));
  }
#pragma unroll 1
  for (; k < lmax; k += 2, ++rp) {        // rows that have ended contribute zero weights (and read row 0)
    int4 r = make_int4(0, 0, 0, 0);
    if (k < len) r = *rp;
    const float4 v0 = t.at(PRE ? agg_rec_row(r.x) : r.x), v1 = t.at(PRE ? agg_rec_row(r.z) : r.z);
    fma_quad(a, v0, __int_as_float(r.y));
    fma_quad(a, v1, __int_as_float(r.w));
  }
  acc = a;
  aux = __int_as_float(d.z);
  return valid;
}

enum { GATHER_SAGE_FWD = 0, GATHER_GCN_BWD = 1, GATHER_SAGE_BWD = 2, GATHER_GCN_FWD = 3 };
enum { GC_SCALE = 0, GC_SHIFT, GC_BSC, GC_MEAN, GC_RSTD, GC_S1N, GC_S2N, GC_ROWS };   // per-channel constant rows

struct GatherArgs {
  const int32_t* meta; long long B; const int32_t* blob;
  int C, max_nodes, max_edges, nslab;
  // tile source
  const float* src;        // SAGE_FWD / GCN_FWD: t_in   GCN_BWD: z   SAGE_BWD: d_agg
  Act act;                 // SAGE_FWD: act on load   GCN_BWD: act_out (its backward)   SAGE_BWD: act_in (for the sums)
  const float* du; const float* demb;                                    // GCN_BWD upstream
  BnBwdDev bn;
  // SAGE_BWD
  const float* direct;     // d_u [rows, C]
  const float* t_raw;      // this layer's stored input (for the sums of the layer below)
  const float* prev_mean; const float* prev_rstd; int want_prev;
  float* out;              // [rows, C]
  float* out_u;            // SAGE_FWD, optional: the transformed input rows act(t_in) are also written here (wide layers)
  float* partials; int part_stride;   // GCN_BWD: dbias [C]; SAGE_BWD: prev sums [2C]
};

// Launchers.  A path that launches one kernel asks its launcher directly: -1 = not covered, nothing was launched (the
// caller tries the next path), > 0 = an error.  A path of several kernels settles the coverage of all of them before the
// first launch, through the *_supported predicate next to each later launcher; those launchers only return CGNN_OK or
// an error.

// engine.cu: warp-specialised hidden-layer forward (64 -> 64 channels; also built for the simulator)
int launch_gcn_fwd_ws(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                      int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z,
                      double* partials, int* grid_out, size_t workspace_bytes, cudaStream_t stream);
// eval-mode last layer: BatchNorm affine + ReLU of the output and the mean-pool readout in the epilogue (emb instead of z)
int launch_gcn_fwd_ws_pool(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                           int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges,
                           const cgnn_act_t* act_out, float* emb, cudaStream_t stream);
#ifndef CGNN_EMU
// agg.cu: one gather kernel (grid in *grid_out: the caller reduces `partials` over it), for C channels when
// gather_supported(C, ...)
bool gather_supported(int C, int max_nodes, int max_edges);
int launch_gather(int mode, GatherArgs& a, int* grid_out, cudaStream_t stream);
// gemm_tc.cu: tensor-core contractions.  The GraphSAGE forward and GCN backward ones run after a gather, when their
// predicate holds for the same arguments (`shape`: where the launcher takes its launch shape from); the GraphSAGE
// backward one runs first (-1 when not covered).
struct GemmShape;
bool sage_fwd_gemm_supported(const float* t_in, const float* agg, const float* z, int64_t rows, int32_t C, int32_t H,
                             bool want_stats, size_t workspace_bytes, GemmShape* shape = nullptr);
int launch_sage_fwd_gemm(const float* t_in, const cgnn_act_t* act, const float* agg, const float* W, const float* bias,
                         int64_t rows, int32_t C, int32_t H, float* z, double* partials, int* grid_out,
                         size_t workspace_bytes, cudaStream_t stream);
bool gcn_bwd_gemm_supported(const float* dP, const float* t_in, const float* du_in, int64_t rows, int32_t d_in, int32_t H,
                            int part_stride, size_t partial_bytes, GemmShape* shape = nullptr);
int launch_gcn_bwd_gemm(const float* dP, const float* t_in, const cgnn_act_t* act_in, const float* W, int64_t rows,
                        int32_t d_in, int32_t H, float* du_in, const float* prev_mean, const float* prev_rstd, int want_prev,
                        float* partials, int part_stride, int o_pprev, int* grid_out, size_t partial_bytes,
                        cudaStream_t stream);
int launch_sage_bwd_gemm(const float* du, const float* demb, const int32_t* row_graph, const int32_t* meta, const float* z,
                         const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn, const float* t_in, const float* agg,
                         const cgnn_act_t* act_in, const float* W, int64_t rows, int32_t C, int32_t H, float* direct,
                         float* nbr, float* partials, int part_stride, int o_pdb, int* grid_out, size_t partial_bytes,
                         cudaStream_t stream);
// first_layer.cu: narrow-input (d_in <= 8) layers without tensor cores; kind = AGG_GCN / AGG_SAGE
int launch_first_fwd(int kind, const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                     int64_t num_graphs, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z, float* agg_out,
                     double* partials, int* grid_out, size_t workspace_bytes, cudaStream_t stream);
int launch_first_bwd(int kind, const float* du, const float* demb, const float* z, const cgnn_act_t* act_out,
                     const cgnn_bn_bwd_t* bn, const float* t_in, const float* agg, const cgnn_act_t* act_in, const cgnn_csr_t* csr,
                     int64_t num_graphs, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* partials,
                     int* grid_out, size_t partial_bytes, cudaStream_t stream);
// wide_tc.cu: H = d_in = 256 (gather + K-looped tcgen05 contraction; forward runs in place in z)
bool wide_shape(int d_in, int H);
int launch_gcn_fwd_wide(const float* t_in, const cgnn_act_t* act, const float* W, const float* bias, const cgnn_csr_t* csr,
                        int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* z,
                        int want_stats, int* grid_out, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int launch_sage_fwd_wide(const float* t_in, const cgnn_act_t* act, float* agg, const float* W, const float* bias,
                         const cgnn_csr_t* csr, int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes,
                         int32_t max_edges, float* z, int want_stats, int* grid_out, void* workspace, size_t workspace_bytes,
                         cudaStream_t stream);
int launch_sage_bwd_wide(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn,
                         const float* t_in, const float* agg, const cgnn_act_t* act_in, const float* W, const cgnn_csr_t* csr,
                         int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges, float* dW,
                         float* dbias, float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64, float* scratch,
                         void* workspace, size_t workspace_bytes, cudaStream_t stream);
int launch_gcn_bwd_wide(const float* du, const float* demb, const float* z, const cgnn_act_t* act_out, const cgnn_bn_bwd_t* bn,
                        const float* t_in, const cgnn_act_t* act_in, const float* W, const cgnn_csr_t* csr, const int64_t* ptr,
                        int64_t num_graphs, int64_t rows, int32_t d_in, int32_t H, int32_t max_nodes, int32_t max_edges,
                        float* dW, float* dbias, float* du_in, const float* prev_mean, const float* prev_rstd, float* prev_sums, double* prev_sums64,
                        float* scratch, void* workspace, size_t workspace_bytes, cudaStream_t stream);
#endif
// agg.cu: blob builder; subjects with <= skip_edge_cap edges (and < 65536 rows) are skipped (built by the collate kernel)
int launch_build_agg(const cgnn_csr_t* csr, int32_t kind, int64_t num_graphs, int32_t max_nodes, int32_t* agg_in, int32_t* agg_out,
                     int32_t* row_graph, int skip_edge_cap, cudaStream_t stream);

}  // namespace cgnn
