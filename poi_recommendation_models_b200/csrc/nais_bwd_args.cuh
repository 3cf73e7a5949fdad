// Arguments and per-CTA partial layout shared by the FP32 backward (nais_bwd.cu) and the tensor-core backward
// (nais_pairs_tc_bwd.cu): both write the same workspace (dq rows, dp rows, parameter partials) for the same reduce kernels.
#pragma once
#include "nais_common.cuh"

namespace nais {

constexpr int BWD_MAXROWS = 16;  // == PAIR_MAXROWS (nais_pairs_tile.cuh)

struct BwdArgs {
  NaisParams p;
  NaisPairs b;
  int bi;                 // branch
  const float* parts;     // [B] per-branch score of this branch
  const float* row_sum;   // [B]
  const float* dscore;    // [B]
  const unsigned long long* act_mask;  // [B*H] ReLU pattern saved by the tcgen05 forward (hid <= 64), or NULL
  // Embedding-row contributions: per-cell dq rows and per-row dp rows, in cell / row order (contiguous 4*D-byte stores); the
  // sorted-segment reduce that follows gathers them through the sorted source lists.  (r2 tried writing them at their position
  // in key order so the reduce could stream: the scattered 128-byte stores cost the tile kernel +75 us at C3 and bought the
  // reduce only 2 x 17 us.)  NULL = no table needs a gradient: nothing is written.
  float* ws_dq;           // [cells, D]
  float* ws_dp;           // [B, D]
  float* ws_part;         // [grid, part_stride]
  int part_stride;
  int64_t n_items;        // work items (tiles of rows: nais_pairs_tile.cuh)
  int* bad;               // the library's bad-index word (nais_common.cuh)
  float drop_inv;         // 1 / (1 - dropout_p) (tcgen05 dropout backward; a kernel parameter, so no register holds it)
};

// layout of one CTA's parameter partial: w1 [hid][D+lanes] | b1 [hid] | w2 [hid] | dist_w[4] dist_b[2] km[1] pad[1]
__host__ __device__ inline int part_floats(int hid, int D, int lanes) { return hid * (D + lanes) + 2 * hid + 8; }

}  // namespace nais
