// Work tiles of the pair kernels: which rows / history cells a 128-cell tile covers, for both layouts of NaisPairs
// (include/nais_b200.h): dense [B, H] rows that each carry their own history, and the segmented (multi-user) layout where the
// rows of a segment share one history stored once.
#pragma once
#include "nais_common.cuh"

namespace nais {

constexpr int PAIR_MAXROWS = 16;  // rows sharing one 128-cell tile when the history is short

// floor(a / b) for 0 <= a <= 128, 1 <= b <= 128 without the ~25-instruction integer division sequence: (a + 0.5) / b is at least
// 1 / 256 away from every integer, far more than the approximate divide's error (the pair kernels do this per cell and work unit)
__device__ __forceinline__ int div_small(int a, int b) { return (int)__fdividef((float)a + 0.5f, (float)b); }

__host__ __device__ inline int pair_rows_per_tile(int H) {
#ifdef __CUDA_ARCH__
  int r = H <= TC ? div_small(TC, H > 0 ? H : 1) : 1;
#else
  int r = H <= TC ? TC / (H > 0 ? H : 1) : 1;
#endif
  return r > PAIR_MAXROWS ? PAIR_MAXROWS : r;
}

struct PairTile {
  int64_t row0;     // first row of the tile (global row index)
  int nrows;        // rows in the tile (all of one segment)
  int H;            // their history length
  int64_t hist0;    // index of (row0, h = 0) in hist / hreg / hist_coords
  int64_t hist_rs;  // history-index stride between consecutive rows: H (dense) or 0 (segmented: shared history)
  int64_t cell0;    // index of (row0, h = 0) in the per-cell arrays (aux, act_mask, dq positions): cell (r, h) = cell0 + r*H + h
};

// The disentangled two-branch layout (include/nais_b200.h): branch 0 owns the POI tables, branch 1 the region table, so no id list is
// in both branches; the fused optimizer paths take it with NAIS_DIST_NONE or NAIS_DIST_KM.
__host__ __device__ inline bool pairs_disentangled(const NaisParams& p) {
  return p.n_branch == 2 && p.branch[0].w_reg == 0 && p.branch[1].w_poi == 0 && p.dist_mode != NAIS_DIST_LATLON;
}
// The layouts the split backward phases and the fused optimizer take: one branch, or the disentangled two.
inline bool pairs_fused_layout(const NaisParams& p) { return p.n_branch == 1 || pairs_disentangled(p); }
__host__ __device__ inline bool pairs_segmented(const NaisPairs& b) { return b.seg_offsets != nullptr; }
__host__ __device__ inline int64_t pairs_n_cells(const NaisPairs& b) { return pairs_segmented(b) ? b.n_cells : b.B * (int64_t)b.H; }
__host__ __device__ inline int64_t pairs_n_tiles(const NaisPairs& b) {
  if (pairs_segmented(b)) return b.n_tiles;
  const int rpt = pair_rows_per_tile(b.H);
  return (b.B + rpt - 1) / rpt;
}

__device__ __forceinline__ PairTile pair_tile(const NaisPairs& b, int64_t item) {
  PairTile t;
  if (!pairs_segmented(b)) {
    const int rpt = pair_rows_per_tile(b.H);
    t.row0 = item * rpt;
    const int64_t left = b.B - t.row0;
    t.nrows = (int)(left < rpt ? left : rpt);
    t.H = b.H;
    t.hist0 = t.row0 * (int64_t)b.H;
    t.hist_rs = b.H;
    t.cell0 = t.hist0;
  } else {
    const int s = __ldg(b.tile_seg + item);
    t.row0 = __ldg(b.tile_row0 + item);
    const int64_t h0 = __ldg(b.seg_offsets + s), r0 = __ldg(b.row_offsets + s), r1 = __ldg(b.row_offsets + s + 1);
    t.H = (int)(__ldg(b.seg_offsets + s + 1) - h0);
    const int rpt = pair_rows_per_tile(t.H);
    const int64_t left = r1 - t.row0;
    t.nrows = (int)(left < rpt ? left : rpt);
    t.hist0 = h0;
    t.hist_rs = 0;
    t.cell0 = __ldg(b.seg_cell_offsets + s) + (t.row0 - r0) * (int64_t)t.H;
  }
  return t;
}

// |dlat|, |dlon| (degrees) of one cell: the dense layout reads the tensor the reference gathers from latlon_mat (run.py:239-247),
// the segmented layout forms them from the centred fp32 coordinates like the full-rank path (exact to ~1e-8 degrees, DESIGN.md)
__device__ __forceinline__ void pair_latlon(const NaisPairs& b, int64_t cidx, int64_t hidx, int64_t row, float& l0, float& l1) {
  if (b.aux) {
    l0 = __ldg(b.aux + cidx * 2);
    l1 = __ldg(b.aux + cidx * 2 + 1);
  } else {
    l0 = fabsf(__ldg(b.tgt_coords + row * 2) - __ldg(b.hist_coords + hidx * 2));
    l1 = fabsf(__ldg(b.tgt_coords + row * 2 + 1) - __ldg(b.hist_coords + hidx * 2 + 1));
  }
}

// dist_km of one cell (NAIS_DIST_KM): the dense layout reads the tensor the caller built (powerLaw.dist, model.py:497-504), the
// segmented layout forms the haversine distance from the centred fp32 coordinates like the full-rank path (nais_fp32.cu)
__device__ __forceinline__ float coords_km(const NaisPairs& b, float tla, float tlo, float hla, float hlo) {
  const float d2r = 0.017453292519943295f;
  return dist_km_f(tla, tlo, hla, hlo, cosf((b.center_lat + tla) * d2r), cosf((b.center_lat + hla) * d2r));
}
__device__ __forceinline__ float pair_km(const NaisPairs& b, int64_t cidx, int64_t hidx, int64_t row) {
  if (b.aux) return __ldg(b.aux + cidx);
  const float tla = __ldg(b.tgt_coords + row * 2), tlo = __ldg(b.tgt_coords + row * 2 + 1);
  const float hla = __ldg(b.hist_coords + hidx * 2), hlo = __ldg(b.hist_coords + hidx * 2 + 1);
  return coords_km(b, tla, tlo, hla, hlo);
}
// the coefficient of the km logit term, sum_d embed_distance[0, d], in the order of the FP32 kernels (km_coef, nais_fp32.cu)
__device__ __forceinline__ float km_coef0(const NaisParams& p, int D) {
  float c = 0.f;
  for (int d = 0; d < D; ++d) c += __ldg(p.dist_embed + d);
  return c;
}

// ---- software pipelining of a tile's inputs (the two-threads-per-cell tcgen05 pair kernels): Ampere-style cp.async into shared
// memory, issued one work unit ahead; a thread waits for ITS OWN copies with cp_async_wait_all(), other threads' after a barrier.
__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst_smem_addr, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem_addr), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// The warp-cooperative gather of the 32-float segment [s0, s0 + 32) of a warp's 32 history rows (ids it32 / rg32 held one per lane):
// 8 lanes cover one row's 128 bytes, request q of a lane is row (lane / 8) + 4 q, and a lane's column — hence its offset in the
// table row and its 16 bytes in the staged row — is the same in all 8 requests: set up once per kernel.  The whole segment must lie
// in ONE table (w_poi a multiple of 32: every shipped model class; pair_gather_uniform() gates the kernels that use this), so one
// shuffle per request fetches the id and the choice of the id register is warp-uniform.
struct RowGather {
  const float* tbl;  // table base + this lane's column
  int stride;        // floats per table row
  bool use_reg;      // the segment is in the region table (warp-uniform)
  int row0;          // lane / 8
  uint32_t dst;      // shared-memory address of this lane's 16 bytes of staged row `row0`
};
__host__ __device__ inline bool pair_gather_uniform(const NaisBranch& br) { return br.w_poi % 32 == 0; }
__device__ __forceinline__ RowGather row_gather_init(const NaisBranch& br, int s0, int lane, const void* stg, int stg_stride) {
  RowGather G;
  const int part = lane & 7, col = s0 + 4 * part;
  G.use_reg = s0 >= br.w_poi;
  G.tbl = G.use_reg ? br.hist_reg + (col - br.w_poi) : br.hist_poi + col;
  G.stride = G.use_reg ? br.w_reg : br.w_poi;
  G.row0 = lane >> 3;
  G.dst = (uint32_t)__cvta_generic_to_shared(stg) + (uint32_t)(G.row0 * stg_stride + part * 16);
  return G;
}
// address of this lane's 16 bytes of request q (q = 0..7): the table row of cell row0 + 4 q of the warp
__device__ __forceinline__ const float* row_gather_src(const RowGather& G, int it32, int rg32, int q) {
  const int id = __shfl_sync(0xffffffffu, G.use_reg ? rg32 : it32, G.row0 + 4 * q);
  return G.tbl + (size_t)id * G.stride;
}

// cell `cell` (0..127) of a work unit of those kernels (128 cells = chunk `ch` of a tile; a tile with H > 128 has several chunks,
// else one): which row of the tile / history position it is, and where its inputs live
struct PairCell {
  bool valid;
  int r, h;
  int64_t cidx, hidx;
};
__device__ __forceinline__ PairCell pair_cell(const PairTile& T, int ch, int cell) {
  PairCell c;
  if (T.H <= TC) {
    c.r = div_small(cell, T.H);
    c.h = cell - c.r * T.H;
    c.valid = c.r < T.nrows;
  } else {
    c.r = 0;
    c.h = ch * TC + cell;
    c.valid = c.h < T.H;
  }
  c.cidx = c.valid ? T.cell0 + c.r * (int64_t)T.H + c.h : 0;
  c.hidx = c.valid ? T.hist0 + c.r * T.hist_rs + c.h : 0;
  return c;
}
__device__ __forceinline__ int pair_chunks(const PairTile& T) { return T.H <= TC ? 1 : (T.H + TC - 1) / TC; }

}  // namespace nais
