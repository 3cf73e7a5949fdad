// Pair forward (model.py:246-297) with the attention-MLP contraction on tcgen05 — the default of nais_pairs_forward
// (NaisParams::pairs_precision = NAIS_PAIRS_AUTO) for one branch with lat/lon or no distance mode, and for the disentangled two
// branches (nais_pairs_tile.cuh) with no distance mode or NAIS_DIST_KM; D in {16, 32, 48, 64} per branch, hid <= 128 (multiple of
// 16); everything else runs the FP32 kernel (nais_fp32.cu).  Train-mode dropout is a compile-time parameter (kDrop): the epilogue
// draws the keep bits of NaisParams::dropout_seed (the FP32 kernels' mask, bit for bit) and saves "active and kept" in act_mask.
// The haversine-km logit term is another (kKm): a += km * sum_d embed_distance[0, d], added once per cell.  Two branches run one
// launch each on a one-branch view of the parameters; the second adds its branch score to `score` (kAcc), so score = s0 + s1 as in
// the FP32 kernel.
//
// A training row has its own history, so unlike full-rank scoring there is no per-user operand to reuse: the GEMM is
//     T[cell, k] = sum_d X[cell, d] * W[k, d],      X[cell, :] = q_cell (.) p_row       (M = 128 cells, N = hid, K = D)
// with the CONSTANT operand W (packed once per CTA into shared memory, hi/lo fp16 planes) and the A operand built per tile by
// the CTA itself: thread = cell gathers its history row with 128-bit loads, forms x in fp32, scales the row by its own
// power of two (one TMEM lane = one cell, so the epilogue un-scales per lane), splits hi/lo and writes the 16-byte k-chunks
// of the canonical K-major SWIZZLE_NONE image (umma.cuh) — consecutive threads write consecutive 16 B, no bank conflicts.
// Three MMA passes (hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM) give fp32-grade products.  Bias, the two distance
// lanes, ReLU, the second layer, exp, mask and the row sums are the epilogue (fp32 CUDA cores, thread = cell = TMEM lane).
// The similarity s = sum_d x_d is summed in fp32 by the building thread.  Four CTAs per SM overlap build / MMA / epilogue.
#include <cstdlib>

#include "nais_common.cuh"
#include "nais_pairs_tile.cuh"
#include "umma.cuh"

namespace nais {
namespace ptc {
using namespace umma;

constexpr int PT = 128;        // threads per CTA = cells per tile = TMEM lanes
constexpr int PMAXROWS = PAIR_MAXROWS;  // rows (targets) sharing one tile when H is small
constexpr int STG_STRIDE = 144;  // bytes per staged row segment: 32 floats + 16 B skew (conflict-free per-thread read-back)

struct Args {
  NaisParams p;
  NaisPairs b;
  float* score;    // [B]
  float* row_sum;  // [B] or NULL
  float* parts;    // [B] or NULL
  unsigned long long* act_mask;  // [cells] ReLU pattern per cell of this branch (hid <= 64) or NULL
  uint32_t tmem_cols;
  int* bad;  // the library's bad-index word (nais_common.cuh)
  uint32_t drop_thresh;  // dropout: dropout_threshold(dropout_p) and 1 / (1 - dropout_p) (kernel parameters: read from the constant bank)
  float drop_inv;
  float* cell_e;   // kCells: [cells] masked exp E of every cell of this branch (nais_pairs_explain), indexed like act_mask
  float* cell_es;  // kCells: [cells] E * similarity
};

__device__ __forceinline__ float pow2_scale(float amax, int target_exp) {
  // power of two s with amax * s in [2^(target_exp-1), 2^target_exp); exponent clamped so 1/s stays a normal float
  if (!(amax > 0.f)) return 1.f;
  int e;
  frexpf(amax, &e);  // amax = f * 2^e, f in [0.5, 1)
  int k = target_exp - e;
  k = k > 40 ? 40 : (k < -40 ? -40 : k);
  return ldexpf(1.f, k);
}

// kCells (instantiated with kDrop = false only): also store every cell's e and e * s for nais_pairs_explain
template <int D, bool kDrop, bool kKm, bool kAcc, bool kCells>
__global__ void __launch_bounds__(PT, (D > 48) ? 3 : 4) pairs_fwd_tc_kernel(const __grid_constant__ Args A) {
  extern __shared__ __align__(128) uint8_t smem[];
  const NaisParams& p = A.p;
  const NaisBranch& br = p.branch[0];
  const int hid = p.hid;
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0, ldw = D + lanes;
  constexpr int KC = D / 8;                // 16-byte k-chunks along K
  constexpr int A_PLANE = KC * PT * 16;    // one fp16 plane of the X tile
  const int w_plane = KC * hid * 16;       // one fp16 plane of W
  uint8_t* sA = smem;                      // [hi | lo][KC][128 rows][16 B]
  uint8_t* sWi = sA + 2 * A_PLANE;         // [hi | lo][KC][hid rows][16 B]
  float* kc = reinterpret_cast<float*>(sWi + 2 * w_plane);  // [4][hid] b1, w2, w1[:, D], w1[:, D+1]
  float* ps = kc + 4 * hid;                // [PMAXROWS][D] target vectors of the rows of this tile
  float* red_e = ps + PMAXROWS * D;        // [PT] masked exp per cell
  float* red_es = red_e + PT;              // [PT] masked exp * similarity
  float* row_e = red_es + PT;              // [PMAXROWS]
  float* row_es = row_e + PMAXROWS;        // [PMAXROWS]
  float* wred = row_es + PMAXROWS;         // [8] per-warp |W| maxima
  uint64_t* bar = reinterpret_cast<uint64_t*>(wred + 8);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  uint8_t* stg_all = reinterpret_cast<uint8_t*>(bar + 2);  // [PT][STG_STRIDE] row staging of the cooperative gather (16-B aligned)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tslot, A.tmem_cols);

  // ---- constant operand: W[:, :D] * wscale as hi/lo fp16 planes, plus the per-hidden-unit constants -------------------------
  float wmax = 0.f;
  for (int i = tid; i < hid * D; i += PT) {
    const int k = i / D, d = i - k * D;
    wmax = fmaxf(wmax, fabsf(__ldg(br.w1 + (size_t)k * ldw + d)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if (lane == 0) wred[warp] = wmax;
  __syncthreads();
  wmax = fmaxf(fmaxf(wred[0], wred[1]), fmaxf(wred[2], wred[3]));
  const float wscale = pow2_scale(wmax, 9);  // |W| * wscale < 512
  const float inv_wscale = 1.f / wscale;
  for (int i = tid; i < hid * KC; i += PT) {
    const int c = i / hid, k = i - c * hid;  // consecutive threads -> consecutive rows -> consecutive 16 B
    __align__(16) __half hi[8], lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split_f16(__ldg(br.w1 + (size_t)k * ldw + c * 8 + e) * wscale, hi[e], lo[e]);
    *reinterpret_cast<uint4*>(sWi + ((size_t)c * hid + k) * 16) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(sWi + w_plane + ((size_t)c * hid + k) * 16) = *reinterpret_cast<const uint4*>(lo);
  }
  for (int k = tid; k < hid; k += PT) {
    kc[k] = __ldg(br.b1 + k);
    kc[hid + k] = __ldg(br.w2 + k);
    kc[2 * hid + k] = lanes ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f;
    kc[3 * hid + k] = lanes ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);  // warp w owns TMEM lanes 32w .. 32w+31
  const bool vec4 = rows_vec4(br, 4);
  float kmc = 0.f;  // kKm: sum_d embed_distance[0, d]
  if constexpr (kKm) kmc = km_coef0(p, D);

  const int64_t n_items = pairs_n_tiles(A.b);
  uint32_t phase = 0;
  for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const PairTile T = pair_tile(A.b, item);
    const int64_t row0 = T.row0;
    const int nrows = T.nrows, H = T.H;
    const int n_chunks = (H <= PT) ? 1 : (H + PT - 1) / PT;
    for (int i = tid; i < nrows * D; i += PT) {
      const int r = i / D, d = i - r * D;
      ps[r * D + d] = (d < br.w_poi) ? __ldg(br.tgt_poi + (size_t)checked_id(A.b.tgt[row0 + r], p.item_num, A.bad) * br.w_poi + d)
                                     : __ldg(br.tgt_reg + (size_t)checked_id(A.b.treg[row0 + r], p.region_num, A.bad) * br.w_reg + (d - br.w_poi));
    }
    if (tid < PMAXROWS) {
      row_e[tid] = 0.f;
      row_es[tid] = 0.f;
    }
    __syncthreads();
    for (int ch = 0; ch < n_chunks; ++ch) {
      int r, h;
      bool valid;
      if (H <= PT) {
        r = tid / H;
        h = tid - r * H;
        valid = r < nrows;
      } else {
        r = 0;
        h = ch * PT + tid;
        valid = h < H;
      }
      const int64_t cidx = valid ? T.cell0 + r * (int64_t)H + h : 0;      // per-cell arrays
      const int64_t hidx = valid ? T.hist0 + r * T.hist_rs + h : 0;       // history arrays
      // ---- build this cell's row of X -------------------------------------------------------------------------------------
      float x[D];
      float ssum = 0.f, amax = 0.f, g0 = 0.f, g1 = 0.f, km = 0.f;
      bool live = false;  // valid and not masked (history item != target)
      int it32 = 0, rg32 = 0;  // POI / region id of this cell (ids fit int32: item_num is int32); row 0 for padding cells
      if (valid) {
        it32 = checked_id(A.b.hist[hidx], p.item_num, A.bad);
        rg32 = br.w_reg ? checked_id(A.b.hreg[hidx], p.region_num, A.bad) : 0;
      }
      if (vec4) {
        // Warp-cooperative gather: consecutive lanes read consecutive 16 B of the SAME table row, so one request covers whole
        // 128-byte lines (4 rows of 32 floats) instead of 32 lines x 16 B — the per-thread pattern kept the kernel waiting on
        // L1 requests in flight.  Rows are staged in this warp's private slice of `stg_all` with a 16-byte skew per row, then
        // each thread reads its own row back conflict-free (only __syncwarp between the two).
        uint8_t* stg = stg_all + (size_t)(warp * 32) * STG_STRIDE;
#pragma unroll
        for (int s0 = 0; s0 < D; s0 += 32) {
          constexpr int full_seg = 32;
          const int segw = (D - s0 < full_seg) ? (D - s0) : full_seg;
          const int P = segw / 4;  // 16-byte parts per row in this segment
          float4 v[full_seg / 4];
#pragma unroll
          for (int q = 0; q < full_seg / 4; ++q) {  // all P loads of this lane are in flight before the first store
            if (q < P) {
              const int idx = lane + 32 * q, c = idx / P, part = idx - c * P;
              const int ci = __shfl_sync(0xffffffffu, it32, c), cr = __shfl_sync(0xffffffffu, rg32, c);
              v[q] = ldg_row4(br.hist_poi + (size_t)ci * br.w_poi, br.hist_reg + (size_t)cr * br.w_reg, br.w_poi, s0 + 4 * part);
            }
          }
#pragma unroll
          for (int q = 0; q < full_seg / 4; ++q) {
            if (q < P) {
              const int idx = lane + 32 * q, c = idx / P, part = idx - c * P;
              *reinterpret_cast<float4*>(stg + (size_t)c * STG_STRIDE + part * 16) = v[q];
            }
          }
          __syncwarp();
#pragma unroll
          for (int j4 = 0; j4 < full_seg / 4; ++j4) {
            if (4 * j4 < segw) {
              const float4 v = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + j4 * 16);
              x[s0 + 4 * j4] = v.x;
              x[s0 + 4 * j4 + 1] = v.y;
              x[s0 + 4 * j4 + 2] = v.z;
              x[s0 + 4 * j4 + 3] = v.w;
            }
          }
          __syncwarp();
        }
      } else if (valid) {
        const float* qp = br.hist_poi + (size_t)it32 * br.w_poi;
        const float* qr = br.hist_reg + (size_t)rg32 * br.w_reg;
#pragma unroll
        for (int d = 0; d < D; ++d) x[d] = (d < br.w_poi) ? __ldg(qp + d) : __ldg(qr + (d - br.w_poi));
      }
      if (valid) {
        const float* pr = ps + r * D;
#pragma unroll
        for (int d = 0; d < D; d += 4) {
          const float4 t = *reinterpret_cast<const float4*>(pr + d);
          x[d] *= t.x;
          x[d + 1] *= t.y;
          x[d + 2] *= t.z;
          x[d + 3] *= t.w;
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          ssum += x[d];
          amax = fmaxf(amax, fabsf(x[d]));
        }
        if (lanes) {
          float l0, l1;
          pair_latlon(A.b, cidx, hidx, row0 + r, l0, l1);
          l0 *= p.dist_scale;
          l1 *= p.dist_scale;
          g0 = sigmoidf_exact(fmaf(l1, __ldg(p.dist_w + 1), fmaf(l0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0))));
          g1 = sigmoidf_exact(fmaf(l1, __ldg(p.dist_w + 3), fmaf(l0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1))));
        }
        if constexpr (kKm) km = pair_km(A.b, cidx, hidx, row0 + r);
        live = A.b.hist[hidx] != A.b.tgt[row0 + r];
      } else {
#pragma unroll
        for (int d = 0; d < D; ++d) x[d] = 0.f;
      }
      const float xscale = pow2_scale(amax, 9);
      const float inv = (1.f / xscale) * inv_wscale;  // both exact powers of two
#pragma unroll
      for (int c = 0; c < KC; ++c) {
        __align__(16) __half hi[8], lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) split_f16(x[c * 8 + e] * xscale, hi[e], lo[e]);
        *reinterpret_cast<uint4*>(sA + ((size_t)c * PT + tid) * 16) = *reinterpret_cast<const uint4*>(hi);
        *reinterpret_cast<uint4*>(sA + A_PLANE + ((size_t)c * PT + tid) * 16) = *reinterpret_cast<const uint4*>(lo);
      }
      fence_proxy_async();  // generic-proxy smem writes -> visible to the MMA's async-proxy reads
      __syncthreads();
      // ---- T = X W^T: hi*hi + hi*lo + lo*hi, one elected thread issues, completion arrives on `bar` ---------------------------
      if (warp == 0) {
        if (elect_one()) {
          tc_fence_after();
          const uint32_t a0 = smem_u32(sA), w0 = smem_u32(sWi);
          const uint32_t idesc = idesc_f16(PT, hid);
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint32_t ab = a0 + (pass == 2 ? A_PLANE : 0), wb = w0 + (pass == 1 ? w_plane : 0);
#pragma unroll
            for (int s = 0; s < D / 16; ++s)
              mma_f16(tmem, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 2 * hid * 16, hid * 16, 128), idesc,
                      (pass | s) != 0);
          }
          mma_commit(bar);
        }
        __syncwarp();
      }
      mbar_wait(bar, phase);
      phase ^= 1u;
      tc_fence_after();
      // ---- epilogue: thread = cell = TMEM lane ------------------------------------------------------------------------------------
      float a = 0.f;
      uint32_t act_lo = 0u, act_hi = 0u;  // ReLU pattern of this cell (hidden units 0..31 / 32..63), saved for the backward
      for (int c0 = 0; c0 < hid; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tlane + c0, v);
        uint32_t keep = 0u;  // kDrop: keep bits of hidden units c0 .. c0 + 15 of this cell (independent of t: hashed while the load runs)
        if constexpr (kDrop) keep = dropout_keep_bits<16>(p.dropout_seed + ((uint64_t)cidx * hid + c0) * DROPOUT_GOLDEN, A.drop_thresh);
        tmem_wait_ld16(v);
        uint32_t bits = 0u;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int k = c0 + i;
          float t = fmaf(__uint_as_float(v[i]), inv, kc[k]);
          if (lanes) t = fmaf(kc[3 * hid + k], g1, fmaf(kc[2 * hid + k], g0, t));
          if constexpr (kDrop) t = ((keep >> i) & 1u) ? t * A.drop_inv : 0.f;  // relu(drop(t)), model.py:71,162
          bits |= (t > 0.f ? 1u : 0u) << i;
          a = fmaf(kc[hid + k], fmaxf(t, 0.f), a);
        }
        if (c0 < 32) act_lo |= bits << c0;
        else if (c0 < 64) act_hi |= bits << (c0 - 32);
      }
      if constexpr (kKm) a += __fmul_rn(km, kmc);  // (the product rounded on its own, as the FP32 kernel adds it)
      if (A.act_mask && valid) A.act_mask[cidx] = ((unsigned long long)act_hi << 32) | act_lo;
      tc_fence_before();  // TMEM reads ordered before the barrier that precedes the next tile's MMAs
      float e = 0.f, es = 0.f;
      if (live) {  // masked cells stay exactly 0 even if exp overflows (reference: exp_A * mask, then * history)
        e = expf(a);
        es = e * ssum;
      }
      red_e[tid] = e;
      red_es[tid] = es;
      if constexpr (kCells) {
        if (valid) {
          A.cell_e[cidx] = e;
          A.cell_es[cidx] = es;
        }
      }
      __syncthreads();
      for (int rr = warp; rr < ((H <= PT) ? nrows : 1); rr += PT / 32) {
        const int c0 = (H <= PT) ? rr * H : 0;
        const int cn = (H <= PT) ? H : min(PT, H - ch * PT);
        float se = 0.f, ses = 0.f;
        for (int c = lane; c < cn; c += 32) {
          se += red_e[c0 + c];
          ses += red_es[c0 + c];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          se += __shfl_xor_sync(0xffffffffu, se, o);
          ses += __shfl_xor_sync(0xffffffffu, ses, o);
        }
        if (lane == 0) {
          row_e[rr] += se;
          row_es[rr] += ses;
        }
      }
      __syncthreads();
    }
    if (tid < nrows) {
      const float S = row_e[tid];
      const float sc = row_es[tid] / powf(S, p.beta);
      A.score[row0 + tid] = kAcc ? A.score[row0 + tid] + sc : sc;
      if (A.row_sum) A.row_sum[row0 + tid] = S;
      if (A.parts) A.parts[row0 + tid] = sc;
    }
    __syncthreads();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, A.tmem_cols);
}

// =====================================================================================================================
// The headline shape (D = hid = 64) with TWO threads per cell (256 threads): warps 0-3 build / drain the first 32 embedding
// columns / hidden units of every cell, warps 4-7 the other 32 (warps w and w + 4 share a TMEM lane quarter).  ncu on the
// 128-thread kernel at C3 (profiles/r2_ncu_pairs_fwd_tc_summary.csv): 168 registers -> 12 warps per SM, issue slots 37 % busy,
// stalled on the L2 gathers; halving the per-thread row (x[32] instead of x[64]) doubles the warps in flight and halves every
// serial phase of a tile.  The halves meet twice per tile: the row's scaling maximum + similarity sum, and the logit.
// =====================================================================================================================
constexpr int PT2 = 256;

// Per-phase clocks of thread 0 (examples/diag_phase_clocks.py builds a private library with -DNAIS_PHASE_CLOCKS; never in the product)
#ifdef NAIS_PHASE_CLOCKS
__device__ unsigned long long g_phase_clk[16];
#define NAIS_PH_INIT long long ph_t = clock64();
#define NAIS_PH(i)                                                               \
  if (tid == 0) {                                                                \
    const long long ph_n = clock64();                                            \
    atomicAdd(&g_phase_clk[i], (unsigned long long)(ph_n - ph_t));               \
    ph_t = ph_n;                                                                 \
  }
#else
#define NAIS_PH_INIT
#define NAIS_PH(i)
#endif

template <bool kDrop, bool kKm, bool kAcc, bool kCells>
__global__ void __launch_bounds__(PT2, 3) pairs_fwd_tc2_kernel(const __grid_constant__ Args A) {
  constexpr int D = 64, HIDC = 64, KC = D / 8, A_PLANE = KC * PT * 16, W_PLANE = KC * HIDC * 16;
  extern __shared__ __align__(128) uint8_t smem[];
  const NaisParams& p = A.p;
  const NaisBranch& br = p.branch[0];
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0, ldw = D + lanes;
  constexpr int STG_BYTES = 8 * 32 * STG_STRIDE;  // 36 864 B: the row staging of eight warps ALIASES the A image (+ 4 KB of padding):
  static_assert(STG_BYTES <= 2 * A_PLANE + 4096, "staging must fit in the A image + pad");  // rows are read back before A is written
  uint8_t* sA = smem;                      // [hi | lo][KC][128 rows][16 B]
  uint8_t* sWi = sA + 2 * A_PLANE + 4096;  // [hi | lo][KC][64 rows][16 B]
  float* kc = reinterpret_cast<float*>(sWi + 2 * W_PLANE);  // [64] x {b1, w2, w1[:, D], w1[:, D+1]}
  float* ps = kc + 4 * HIDC;               // [2][PMAXROWS][D] target vectors of the rows of this tile / of the next tile
  float* red_e = ps + 2 * PMAXROWS * D;    // [PT] masked exp per cell
  float* red_es = red_e + PT;              // [PT] masked exp * similarity
  float* row_e = red_es + PT;              // [PMAXROWS] running sums of a row with more than one chunk
  float* row_es = row_e + PMAXROWS;        // [PMAXROWS]
  float* wred = row_es + PMAXROWS;         // [8] per-warp |W| maxima
  float* xmax = wred + 8;                  // [2][PT] |x| maximum of each half of a cell's row
  float* xsum = xmax + 2 * PT;             // [2][PT] similarity partial of each half
  float* apart = xsum + 2 * PT;            // [2][PT] logit partial of each half
  uint32_t* abits = reinterpret_cast<uint32_t*>(apart + 2 * PT);  // [PT] ReLU pattern of hidden units 32..63 (from half 1)
  // inputs of the NEXT work unit, copied one unit ahead with cp.async (see the loop): ids private to the copying thread
  long long* m_hist = reinterpret_cast<long long*>(abits + PT);  // [PT2] history POI id of this thread's cell
  long long* m_hreg = m_hist + PT2;                              // [PT2] its region id
  long long* m_psid = m_hreg + PT2;                              // [PT2] target POI / region id behind this thread's 16 B of `ps`
  long long* m_tgt = m_psid + PT2;                               // [PMAXROWS] target POI id of each row (live mask)
  float2* m_ll = reinterpret_cast<float2*>(m_tgt + PMAXROWS);    // [PT] |dlat|,|dlon| (kKm: .x = km) of the cell, or the history item's coordinates
  float2* m_tco = m_ll + PT;                                     // [PMAXROWS] target coordinates (segmented layout)
  uint64_t* bar = reinterpret_cast<uint64_t*>(m_tco + PMAXROWS);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  uint8_t* stg_all = sA;                   // [8 warps][32][STG_STRIDE] row staging of the cooperative gather

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int half = warp >> 2, qd = warp & 3, cell = qd * 32 + lane, s0 = 32 * half;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tslot, 64u);
  // ---- constant operand: W[:, :D] * wscale as hi/lo fp16 planes, plus the per-hidden-unit constants -------------------------
  float wmax = 0.f;
  for (int i = tid; i < HIDC * D; i += PT2) {
    const int k = i / D, d = i - k * D;
    wmax = fmaxf(wmax, fabsf(__ldg(br.w1 + (size_t)k * ldw + d)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if (lane == 0) wred[warp] = wmax;
  __syncthreads();
  wmax = fmaxf(fmaxf(fmaxf(wred[0], wred[1]), fmaxf(wred[2], wred[3])), fmaxf(fmaxf(wred[4], wred[5]), fmaxf(wred[6], wred[7])));
  const float wscale = pow2_scale(wmax, 9);  // |W| * wscale < 512
  const float inv_wscale = 1.f / wscale;
  for (int i = tid; i < HIDC * KC; i += PT2) {
    const int c = i / HIDC, k = i - c * HIDC;
    __align__(16) __half hi[8], lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split_f16(__ldg(br.w1 + (size_t)k * ldw + c * 8 + e) * wscale, hi[e], lo[e]);
    *reinterpret_cast<uint4*>(sWi + ((size_t)c * HIDC + k) * 16) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(sWi + W_PLANE + ((size_t)c * HIDC + k) * 16) = *reinterpret_cast<const uint4*>(lo);
  }
  for (int k = tid; k < HIDC; k += PT2)  // one 16-byte load per hidden unit in the epilogue: {b1, w2, w1[:, D], w1[:, D+1]}
    reinterpret_cast<float4*>(kc)[k] = make_float4(__ldg(br.b1 + k), __ldg(br.w2 + k), lanes ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f,
                                                   lanes ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tlane = tmem + ((uint32_t)(qd * 32) << 16);
  uint8_t* stg = stg_all + (size_t)(warp * 32) * STG_STRIDE;
  float kmc = 0.f;  // kKm: sum_d embed_distance[0, d]
  if constexpr (kKm) kmc = km_coef0(p, D);

  // ---- the input pipeline.  ncu + per-phase clocks on the unpipelined kernel (profiles/r2_phase_clocks_before.txt): 41 % of a
  // tile's time was exposed load latency in a dependent chain (target id -> target row; history id -> history row).  Now the
  // inputs of work unit u + 1 are copied while unit u computes, with nothing held in registers:
  //   P1 (after u's inputs are consumed)  ids / lat-lon of u + 1                  -> m_* arrays           (DRAM latency)
  //   P2 (after u's MMAs are complete)    history rows of u + 1 -> `stg` (aliases the A image, free now); target rows -> ps[next]
  // and u + 1 starts with cp.async.wait_all + one barrier.
  const RowGather RG = row_gather_init(br, s0, lane, stg, STG_STRIDE);
  auto issue_ids = [&](const PairTile& Tn, int chn) {
    const PairCell c = pair_cell(Tn, chn, cell);
    if (c.valid) {
      cp_async8(m_hist + tid, A.b.hist + c.hidx);
      if (br.w_reg) cp_async8(m_hreg + tid, A.b.hreg + c.hidx);
      if (lanes && half == 0) cp_async8(m_ll + cell, A.b.aux ? A.b.aux + c.cidx * 2 : A.b.hist_coords + c.hidx * 2);
      if (kKm && half == 0) {  // the dense layout's km, or the history item's coordinates (where the lat/lon lanes stage theirs)
        if (A.b.aux) cp_async4(m_ll + cell, A.b.aux + c.cidx);
        else cp_async8(m_ll + cell, A.b.hist_coords + c.hidx * 2);
      }
    }
    if (tid < Tn.nrows) cp_async8(m_tgt + tid, A.b.tgt + Tn.row0 + tid);
    if ((lanes || kKm) && !A.b.aux && tid >= 32 && tid < 32 + Tn.nrows)
      cp_async8(m_tco + (tid - 32), A.b.tgt_coords + (Tn.row0 + tid - 32) * 2);
    if (chn == 0 && tid * 4 < Tn.nrows * D) {
      const int r = (tid * 4) / D, d = tid * 4 - r * D;
      cp_async8(m_psid + tid, (d < br.w_poi ? A.b.tgt : A.b.treg) + Tn.row0 + r);
    }
  };
  auto issue_rows = [&](const PairTile& Tn, int chn, int pbn) {  // (this thread's own id copies have landed: cp_async_wait_all)
    const PairCell c = pair_cell(Tn, chn, cell);
    int it32 = 0, rg32 = 0;
    if (c.valid) {
      it32 = checked_id(m_hist[tid], p.item_num, A.bad);
      rg32 = br.w_reg ? checked_id(m_hreg[tid], p.region_num, A.bad) : 0;
    }
    // warp-cooperative gather of the 32-float segment [s0, s0 + 32) of this warp's 32 history rows (nais_pairs_tile.cuh RowGather)
#pragma unroll
    for (int q = 0; q < 8; ++q) cp_async16(RG.dst + (uint32_t)(q * 4 * STG_STRIDE), row_gather_src(RG, it32, rg32, q));
    if (chn == 0 && tid * 4 < Tn.nrows * D) {
      const int r = (tid * 4) / D, d = tid * 4 - r * D;
      const float* src = d < br.w_poi ? br.tgt_poi + (size_t)checked_id(m_psid[tid], p.item_num, A.bad) * br.w_poi + d
                                      : br.tgt_reg + (size_t)checked_id(m_psid[tid], p.region_num, A.bad) * br.w_reg + (d - br.w_poi);
      cp_async16(ps + (size_t)pbn * PMAXROWS * D + tid * 4, src);
    }
  };

  const int64_t n_items = pairs_n_tiles(A.b);
  int64_t item = blockIdx.x;  // (the launch gives every CTA at least one tile)
  int ch = 0, pb = 0;
  uint32_t phase = 0;
  NAIS_PH_INIT
  {
    const PairTile T0 = pair_tile(A.b, item);
    issue_ids(T0, 0);
    cp_async_wait_all();
    issue_rows(T0, 0, 0);
  }
  NAIS_PH(0)
  while (true) {
    const PairTile T = pair_tile(A.b, item);
    const int64_t row0 = T.row0;
    const int nrows = T.nrows, H = T.H;
    const int n_chunks = pair_chunks(T);
    const PairCell c = pair_cell(T, ch, cell);
    const bool valid = c.valid;
    const int r = c.r;
    const bool same = ch + 1 < n_chunks;               // the next unit: the next chunk of this tile, or this CTA's next tile
    const int64_t item_n = same ? item : item + gridDim.x;
    const int ch_n = same ? ch + 1 : 0, pb_n = same ? pb : pb ^ 1;
    const bool has_next = item_n < n_items;

    cp_async_wait_all();
    __syncthreads();  // (a) this unit's rows, ids, lat/lon and target vectors are in shared memory
    NAIS_PH(1)
    // ---- this half of the cell's row of X -----------------------------------------------------------------------------------
    float x[32];
    float g0 = 0.f, g1 = 0.f, ssum = 0.f, amax = 0.f, km = 0.f;
    bool live = false;
    if (valid) {
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 t = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + j4 * 16);
        const float4 q = *reinterpret_cast<const float4*>(ps + (size_t)pb * PMAXROWS * D + r * D + s0 + 4 * j4);
        x[4 * j4] = t.x * q.x;
        x[4 * j4 + 1] = t.y * q.y;
        x[4 * j4 + 2] = t.z * q.z;
        x[4 * j4 + 3] = t.w * q.w;
      }
#pragma unroll
      for (int d = 0; d < 32; ++d) {
        ssum += x[d];
        amax = fmaxf(amax, fabsf(x[d]));
      }
      if (lanes) {
        const float2 hl = m_ll[cell];
        float l0 = hl.x, l1 = hl.y;
        if (!A.b.aux) {  // (pair_latlon of the segmented layout)
          const float2 tc = m_tco[r];
          l0 = fabsf(tc.x - hl.x);
          l1 = fabsf(tc.y - hl.y);
        }
        l0 *= p.dist_scale;
        l1 *= p.dist_scale;
        g0 = sigmoidf_exact(fmaf(l1, __ldg(p.dist_w + 1), fmaf(l0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0))));
        g1 = sigmoidf_exact(fmaf(l1, __ldg(p.dist_w + 3), fmaf(l0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1))));
      }
      if (kKm && half == 0) {  // (pair_km: the same dist_km_f call on the same coordinates)
        const float2 hl = m_ll[cell];
        km = hl.x;
        if (!A.b.aux) {
          const float2 tc = m_tco[r];
          km = coords_km(A.b, tc.x, tc.y, hl.x, hl.y);
        }
      }
      live = m_hist[tid] != m_tgt[r];
    } else {
#pragma unroll
      for (int d = 0; d < 32; ++d) x[d] = 0.f;
    }
    xmax[half * PT + cell] = amax;
    xsum[half * PT + cell] = ssum;
    NAIS_PH(2)
    __syncthreads();  // (b) the staged rows and the m_* arrays are consumed (A image / next ids may be written); the halves of a cell meet
    NAIS_PH(3)
    if (has_next) issue_ids(same ? T : pair_tile(A.b, item_n), ch_n);  // P1
    amax = fmaxf(xmax[cell], xmax[PT + cell]);
    ssum = xsum[cell] + xsum[PT + cell];
    const float xscale = pow2_scale(amax, 9);
    const float inv = (1.f / xscale) * inv_wscale;  // both exact powers of two
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      __align__(16) __half hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) split_f16(x[cc * 8 + e] * xscale, hi[e], lo[e]);
      *reinterpret_cast<uint4*>(sA + ((size_t)(s0 / 8 + cc) * PT + cell) * 16) = *reinterpret_cast<const uint4*>(hi);
      *reinterpret_cast<uint4*>(sA + A_PLANE + ((size_t)(s0 / 8 + cc) * PT + cell) * 16) = *reinterpret_cast<const uint4*>(lo);
    }
    fence_proxy_async();  // generic-proxy smem writes -> visible to the MMA's async-proxy reads
    __syncthreads();      // (c)
    NAIS_PH(4)
    // ---- T = X W^T: hi*hi + hi*lo + lo*hi, one elected thread issues, completion arrives on `bar` ---------------------------
    if (warp == 0) {
      if (elect_one()) {
        tc_fence_after();
        const uint32_t a0 = smem_u32(sA), w0 = smem_u32(sWi);
        const uint32_t idesc = idesc_f16(PT, HIDC);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t ab = a0 + (pass == 2 ? A_PLANE : 0), wb = w0 + (pass == 1 ? W_PLANE : 0);
#pragma unroll
          for (int s = 0; s < D / 16; ++s)
            mma_f16(tmem, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 2 * HIDC * 16, HIDC * 16, 128), idesc,
                    (pass | s) != 0);
        }
        mma_commit(bar);
      }
      __syncwarp();
    }
    // kDrop: keep bits of this thread's 32 hidden units s0 .. s0 + 31 (they depend on (seed, cell, k) only: hashed while the MMAs run)
    uint32_t keep = 0u;
    if constexpr (kDrop) keep = dropout_keep_bits<32>(p.dropout_seed + ((uint64_t)c.cidx * HIDC + s0) * DROPOUT_GOLDEN, A.drop_thresh);
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after();
    NAIS_PH(5)
    if (has_next) {  // P2: the A image is free (MMAs complete) -> stage the next unit's rows on it
      cp_async_wait_all();
      issue_rows(same ? T : pair_tile(A.b, item_n), ch_n, pb_n);
    }
    NAIS_PH(6)
    // ---- epilogue: this thread's 32 hidden units of its cell -------------------------------------------------------------------
    float a = 0.f;
    uint32_t bits = 0u;
#pragma unroll
    for (int c0 = 0; c0 < 32; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(tlane + s0 + c0, v);
      tmem_wait_ld16(v);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float4 c4 = reinterpret_cast<const float4*>(kc)[s0 + c0 + i];
        float t = fmaf(__uint_as_float(v[i]), inv, c4.x);
        if (lanes) t = fmaf(c4.w, g1, fmaf(c4.z, g0, t));
        if constexpr (kDrop) t = ((keep >> (c0 + i)) & 1u) ? t * A.drop_inv : 0.f;  // relu(drop(t)): a dropped unit is inactive in the saved pattern
        // t > 0  <=>  the sign bit of (0 - t) is set (IEEE: 0 - (+-0) = +0, so an exact zero counts as inactive like torch's
        // relu backward); shifted in from the right, un-reversed once below: 2 instructions per unit instead of 5
        bits = __funnelshift_l(__float_as_uint(0.f - t), bits, 1);
        a = fmaf(c4.y, fmaxf(t, 0.f), a);
      }
    }
    bits = __brev(bits);
    tc_fence_before();  // TMEM reads ordered before the barrier that precedes the next unit's MMAs
    apart[half * PT + cell] = a;
    if (half == 1) abits[cell] = bits;
    asm volatile("bar.sync %0, 64;" ::"r"(1 + qd) : "memory");
    NAIS_PH(7)
    if (half == 0) {
      a = apart[cell] + apart[PT + cell];
      if constexpr (kKm) a += __fmul_rn(km, kmc);  // the halves meet at the logit; the km term once per cell
      if (A.act_mask && valid) A.act_mask[c.cidx] = ((unsigned long long)abits[cell] << 32) | bits;
      float e = 0.f, es = 0.f;
      if (live) {  // masked cells stay exactly 0 even if exp overflows (reference: exp_A * mask, then * history)
        e = expf(a);
        es = e * ssum;
      }
      red_e[cell] = e;
      red_es[cell] = es;
      if constexpr (kCells) {
        if (valid) {
          A.cell_e[c.cidx] = e;
          A.cell_es[c.cidx] = es;
        }
      }
    }
    __syncthreads();  // (d)
    NAIS_PH(8)
    // ---- per-row sums; the warp that owns a row keeps its running sums and writes the score with the last chunk (no barrier) ----
    for (int rr = warp; rr < ((H <= PT) ? nrows : 1); rr += PT2 / 32) {
      const int c0 = (H <= PT) ? rr * H : 0;
      const int cn = (H <= PT) ? H : min(PT, H - ch * PT);
      float se = 0.f, ses = 0.f;
      for (int cc = lane; cc < cn; cc += 32) {
        se += red_e[c0 + cc];
        ses += red_es[c0 + cc];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        se += __shfl_xor_sync(0xffffffffu, se, o);
        ses += __shfl_xor_sync(0xffffffffu, ses, o);
      }
      if (lane == 0) {
        if (ch > 0) {
          se += row_e[rr];
          ses += row_es[rr];
        }
        if (same) {
          row_e[rr] = se;
          row_es[rr] = ses;
        } else {
          const float sc = ses / powf(se, p.beta);
          A.score[row0 + rr] = kAcc ? A.score[row0 + rr] + sc : sc;
          if (A.row_sum) A.row_sum[row0 + rr] = se;
          if (A.parts) A.parts[row0 + rr] = sc;
        }
      }
    }
    NAIS_PH(9)
    if (!has_next) break;
    item = item_n;
    ch = ch_n;
    pb = pb_n;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64u);
}

template <bool kDrop, bool kKm, bool kAcc, bool kCells>
static int launch2(const Args& A, int64_t n_items, int sms, cudaStream_t stream) {
  constexpr int D = 64, HIDC = 64;
  const size_t smem = 2 * (size_t)(D / 8) * PT * 16 + 2 * (size_t)(D / 8) * HIDC * 16 +
                      4096 + (4 * (size_t)HIDC + 2 * PMAXROWS * D + 2 * PT + 2 * PMAXROWS + 8 + 6 * PT + PT) * 4 +
                      (3 * (size_t)PT2 + PMAXROWS) * 8 + ((size_t)PT + PMAXROWS) * 8 + 16;
  static SmemAttrOnce attr;
  cudaError_t e = attr(pairs_fwd_tc2_kernel<kDrop, kKm, kAcc, kCells>, smem, true);
  if (e != cudaSuccess) return (int)e;
  int per_sm = 3;
  const int by_smem = (int)((227 * 1024) / (smem + 1024));
  per_sm = per_sm < by_smem ? per_sm : by_smem;
  if (per_sm < 1) return NAIS_ERR_SHAPE;
  const int64_t cap = (int64_t)sms * per_sm;
  const int grid = (int)(n_items < cap ? n_items : cap);
  pairs_fwd_tc2_kernel<kDrop, kKm, kAcc, kCells><<<grid, PT2, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

template <int D, bool kDrop, bool kKm, bool kAcc, bool kCells>
static int launch(const Args& A, int hid, int64_t n_items, int sms, cudaStream_t stream) {
  const size_t smem = 2 * (size_t)(D / 8) * PT * 16 + 2 * (size_t)(D / 8) * hid * 16 +
                      (4 * (size_t)hid + PMAXROWS * D + 2 * PT + 2 * PMAXROWS + 8) * 4 + 16 + (size_t)PT * STG_STRIDE;
  cudaError_t e = cudaFuncSetAttribute(pairs_fwd_tc_kernel<D, kDrop, kKm, kAcc, kCells>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(pairs_fwd_tc_kernel<D, kDrop, kKm, kAcc, kCells>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return (int)e;
  // Persistent grid: as many CTAs as can be co-resident — the kernel's register budget (3 per SM for D = 64, else 4), shared
  // memory, and TMEM (tmem_cols of the SM's 512 columns per CTA; a CTA beyond that would simply wait in tcgen05.alloc).
  int per_sm = (D > 48) ? 3 : 4;
  const int by_tmem = (int)(512 / A.tmem_cols), by_smem = (int)((227 * 1024) / (smem + 1024));
  per_sm = per_sm < by_tmem ? per_sm : by_tmem;
  per_sm = per_sm < by_smem ? per_sm : by_smem;
  if (per_sm < 1) return NAIS_ERR_SHAPE;
  const int64_t cap = (int64_t)sms * per_sm;
  const int grid = (int)(n_items < cap ? n_items : cap);
  pairs_fwd_tc_kernel<D, kDrop, kKm, kAcc, kCells><<<grid, PT, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// `two`: two threads per cell (D = hid = 64, a cell's 32-column halves each lie in one table)
template <bool kDrop, bool kKm, bool kAcc, bool kCells = false>
static int launch_shape(const Args& A, int D, bool two, int64_t n_items, int sms, cudaStream_t stream) {
  if (two) return launch2<kDrop, kKm, kAcc, kCells>(A, n_items, sms, stream);
  switch (D) {
    case 16: return launch<16, kDrop, kKm, kAcc, kCells>(A, A.p.hid, n_items, sms, stream);
    case 32: return launch<32, kDrop, kKm, kAcc, kCells>(A, A.p.hid, n_items, sms, stream);
    case 48: return launch<48, kDrop, kKm, kAcc, kCells>(A, A.p.hid, n_items, sms, stream);
    case 64: return launch<64, kDrop, kKm, kAcc, kCells>(A, A.p.hid, n_items, sms, stream);
    default: return NAIS_ERR_SHAPE;
  }
}

}  // namespace ptc

// One branch (lat/lon or no distance mode, dropout or not), or the disentangled two (no distance mode or km, no dropout: the
// disentangled model has none).
bool pairs_tc_supported(const NaisParams& p, const NaisPairs& b) {
  if (b.B < 1) return false;
  const bool two = pairs_disentangled(p);
  if (p.n_branch != 1 && !two) return false;
  if (p.dist_mode == NAIS_DIST_KM && !two) return false;
  if (two && p.dropout_p > 0.f) return false;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const int D = p.branch[bi].w_poi + p.branch[bi].w_reg;
    if (D != 16 && D != 32 && D != 48 && D != 64) return false;
  }
  if (p.hid < 16 || p.hid > 128 || (p.hid & 15)) return false;
  return true;
}

// row_sum / parts are [n_branch, B], act_mask and cell_e / cell_es [n_branch, cells] (each may be NULL); branch bi writes its
// slice.  cell_e and cell_es (nais_pairs_explain) run the kCells kernels; they are never given with dropout.
int launch_pairs_fwd_tc(const NaisParams& p, const NaisPairs& b, float* score, float* row_sum, float* parts,
                        unsigned long long* act_mask, cudaStream_t stream, float* cell_e, float* cell_es) {
  const DeviceInfo di = device_info();
  if (di.major != 10) return NAIS_ERR_ARCH;
  const int sms = di.sms;
  const int64_t n_items = pairs_n_tiles(b);
  if (n_items < 1) return 0;
  const bool km = p.dist_mode == NAIS_DIST_KM;
  const bool cells = cell_e && cell_es;
  if (cells && p.dropout_p > 0.f) return NAIS_ERR_MODE;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    ptc::Args A;
    A.p = p;
    A.p.n_branch = 1;  // the kernels read branch 0: a one-branch view of branch bi
    A.p.branch[0] = p.branch[bi];
    A.b = b;
    A.score = score;
    A.row_sum = row_sum ? row_sum + (size_t)bi * b.B : nullptr;
    A.parts = parts ? parts + (size_t)bi * b.B : nullptr;
    A.act_mask = (p.hid <= 64 && act_mask) ? act_mask + (size_t)bi * pairs_n_cells(b) : nullptr;
    A.bad = bad_index_flag();
    A.drop_thresh = p.dropout_p > 0.f ? dropout_threshold(p.dropout_p) : 0u;
    A.drop_inv = p.dropout_p > 0.f ? 1.f / (1.f - p.dropout_p) : 1.f;
    A.tmem_cols = p.hid <= 32 ? 32u : (p.hid <= 64 ? 64u : 128u);
    A.cell_e = cells ? cell_e + (size_t)bi * pairs_n_cells(b) : nullptr;
    A.cell_es = cells ? cell_es + (size_t)bi * pairs_n_cells(b) : nullptr;
    const NaisBranch& br = p.branch[bi];
    const int D = br.w_poi + br.w_reg;
    const bool two = D == 64 && p.hid == 64 && rows_vec4(br, 4) && pair_gather_uniform(br);
    int rc;
    if (cells) rc = km ? (bi ? ptc::launch_shape<false, true, true, true>(A, D, two, n_items, sms, stream)
                             : ptc::launch_shape<false, true, false, true>(A, D, two, n_items, sms, stream))
                       : (bi ? ptc::launch_shape<false, false, true, true>(A, D, two, n_items, sms, stream)
                             : ptc::launch_shape<false, false, false, true>(A, D, two, n_items, sms, stream));
    else if (p.dropout_p > 0.f) rc = ptc::launch_shape<true, false, false>(A, D, two, n_items, sms, stream);  // (one branch only)
    else if (km) rc = bi ? ptc::launch_shape<false, true, true>(A, D, two, n_items, sms, stream)
                         : ptc::launch_shape<false, true, false>(A, D, two, n_items, sms, stream);
    else rc = bi ? ptc::launch_shape<false, false, true>(A, D, two, n_items, sms, stream)
                 : ptc::launch_shape<false, false, false>(A, D, two, n_items, sms, stream);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace nais

#ifdef NAIS_PHASE_CLOCKS
extern "C" __attribute__((visibility("default"))) int nais_debug_phase_fwd(unsigned long long* host16, int reset) {
  cudaError_t e = cudaMemcpyFromSymbol(host16, nais::ptc::g_phase_clk, sizeof(unsigned long long) * 16);
  if (e == cudaSuccess && reset) {
    unsigned long long z[16] = {};
    e = cudaMemcpyToSymbol(nais::ptc::g_phase_clk, z, sizeof(z));
  }
  return (int)e;
}
#endif
