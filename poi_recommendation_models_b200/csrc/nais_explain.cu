// Explanations of pair scores (nais_pairs_explain, include/nais_b200.h): which history items a score is made of.
//
// The pair forward (FP32 or tcgen05, kCells) stores every cell's masked exp E_bh and E_bh * s_bh; this file's selection kernel
// turns them into per-row contributions c_h = sum_b E_bh s_bh / S_b^beta (summed over h they are the row's pre-sigmoid score)
// and keeps the m largest by the ranking key of the full-rank top-k (make_key: value descending, then position ascending).
// One warp per row: the row's history is walked 32 positions at a time, each lane keys one position, and the running top-32
// is kept in registers (warp_sort_desc + warp_fold_top32, nais_common.cuh) — no shared memory, no atomics, deterministic.
#include "nais_common.cuh"
#include "nais_pairs_tile.cuh"

namespace nais {

struct ExplainArgs {
  NaisPairs b;
  int n_branch, m;
  float beta;
  int64_t n_cells;
  const float* cell_e;   // [n_branch, cells]
  const float* cell_es;  // [n_branch, cells]
  const float* row_sum;  // [n_branch, B]: S_b of every row (the forward's row_sum)
  int32_t* out_pos;      // [B, m]
  float* out_contrib;    // [B, m]
  float* out_attn;       // [n_branch, B, m] or NULL
};

constexpr int EXPLAIN_THREADS = 256;

__global__ void __launch_bounds__(EXPLAIN_THREADS) explain_select_kernel(const __grid_constant__ ExplainArgs A) {
  const int64_t row = ((int64_t)blockIdx.x * EXPLAIN_THREADS + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= A.b.B) return;  // (warp-uniform)
  // the row's history: H positions at hist0 .. in the history arrays, cells cell0 .. in the per-cell arrays (NaisPairs)
  int64_t H, hist0, cell0;
  if (!pairs_segmented(A.b)) {
    H = A.b.H;
    hist0 = cell0 = row * H;
  } else {  // segment s with row_offsets[s] <= row < row_offsets[s + 1]
    int lo = 0, hi = A.b.n_seg;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(A.b.row_offsets + mid) <= row) lo = mid;
      else hi = mid;
    }
    hist0 = __ldg(A.b.seg_offsets + lo);
    H = __ldg(A.b.seg_offsets + lo + 1) - hist0;
    cell0 = __ldg(A.b.seg_cell_offsets + lo) + (row - __ldg(A.b.row_offsets + lo)) * H;
  }
  const int64_t tgt = A.b.tgt[row];
  float S[2] = {1.f, 1.f}, den[2] = {1.f, 1.f};
#pragma unroll
  for (int bi = 0; bi < 2; ++bi) {
    if (bi < A.n_branch) {
      S[bi] = A.row_sum[(size_t)bi * A.b.B + row];
      den[bi] = powf(S[bi], A.beta);  // one powf per row and branch, as the forward's score
    }
  }
  unsigned long long top = 0ull;  // lane i: the i-th best key so far (0 = none)
  for (int64_t h0 = 0; h0 < H; h0 += 32) {
    const int64_t h = h0 + lane;
    unsigned long long key = 0ull;
    if (h < H && A.b.hist[hist0 + h] != tgt) {  // a masked cell (history item == target) is never selected
      float c = 0.f;
#pragma unroll
      for (int bi = 0; bi < 2; ++bi)
        if (bi < A.n_branch) c += A.cell_es[(size_t)bi * A.n_cells + cell0 + h] / den[bi];
      key = make_key(c, (int)h);
    }
    const unsigned long long v = warp_sort_desc(key, lane);
    top = h0 == 0 ? v : warp_fold_top32(top, v, lane);
  }
  if (lane < A.m) {
    float c;
    int pos;
    split_key(top, c, pos);  // (-inf, -1) for a lane without a selectable cell
    const size_t o = (size_t)row * A.m + lane;
    A.out_pos[o] = pos;
    A.out_contrib[o] = c;
    if (A.out_attn) {
#pragma unroll
      for (int bi = 0; bi < 2; ++bi)
        if (bi < A.n_branch)
          A.out_attn[((size_t)bi * A.b.B + row) * A.m + lane] = pos >= 0 ? A.cell_e[(size_t)bi * A.n_cells + cell0 + pos] / S[bi] : 0.f;
    }
  }
}

int launch_explain_select(const NaisParams& p, const NaisPairs& b, int m, const float* cell_e, const float* cell_es,
                          const float* row_sum, int32_t* out_pos, float* out_contrib, float* out_attn, cudaStream_t stream) {
  if (b.B == 0) return 0;
  ExplainArgs A;
  A.b = b;
  A.n_branch = p.n_branch;
  A.m = m;
  A.beta = p.beta;
  A.n_cells = pairs_n_cells(b);
  A.cell_e = cell_e;
  A.cell_es = cell_es;
  A.row_sum = row_sum;
  A.out_pos = out_pos;
  A.out_contrib = out_contrib;
  A.out_attn = out_attn;
  const int64_t blocks = (b.B + EXPLAIN_THREADS / 32 - 1) / (EXPLAIN_THREADS / 32);
  explain_select_kernel<<<(unsigned)blocks, EXPLAIN_THREADS, 0, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

}  // namespace nais
