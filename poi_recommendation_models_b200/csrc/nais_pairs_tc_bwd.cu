// Backward of the pair scorer with all three contractions on tcgen05 — the default of nais_pairs_backward[_adagrad]
// (NaisParams::pairs_precision = NAIS_PAIRS_AUTO) for one branch with lat/lon or no distance mode and for the disentangled two
// branches with no distance mode or NAIS_DIST_KM (one launch per branch, BwdArgs::bi), hidden_size = 64, D in {32, 64}, 16-byte
// aligned table rows; everything else runs the FP32 kernel (nais_bwd.cu).  The km logit term is a compile-time mode (kKm): the
// recomputed logit adds km * sum_d embed_distance[0, d], and each CTA sums da * km over its cells in a fixed order into the partial
// slot of the FP32 kernel (no atomics).  Train-mode dropout (kDrop) draws nothing: with
// m = the forward's saved "active and kept" bit, relu(drop(t)) = m relu(t) / (1-p), so m gives the recomputed logit, the dw2 term
// and dt = m da v / (1-p) — the dropout backward needs act_mask (without it the FP32 kernel runs, which regenerates the mask).
// It writes the SAME workspace as pairs_bwd_kernel (dq rows, dp rows, one parameter partial per CTA), so the deterministic
// param_reduce and the sorted-segment embedding reduce that follow are shared.
//
// Tile = 128 cells (one row's history at H = 128).  Operands are bf16 two-term splits (hi*hi + hi*lo + lo*hi, fp32 accumulation
// in TMEM) with NO scaling anywhere: dW is a contraction over cells accumulated across all tiles of the CTA, so no per-row
// scale could be undone (examples/precision_emulation_backward.py: every gradient within 7e-6 of its tensor maximum, bar 2e-4).
//
//   GEMM1  T[cell,k]  = sum_d X[cell,d] W[k,d]            A = X image (K-major), B = W image (K-major)            -> TMEM cols 0..63
//   epi 1  a, e, da, gw; dt = da v [t > 0] -> DT image; dg -> dist-layer partials; sum_cell da relu(t) -> dv (shuffle halving)
//   GEMM2  dX[cell,d] = sum_k dt[cell,k] W[k,d]           A = DT image (K-major), B = W image read MN-major       -> cols 64..127
//   GEMM3  dW[k,n]   += sum_cell dt[cell,k] Xe[cell,n]    A = DT image, B = X image, BOTH read MN-major (transpose bits;
//          Xe = [X | 1 g0 g1]: the ext chunk yields db1 and the two lane columns of dW)  M = 64 -> cols 128..199, row m in
//          TMEM lane 32*(m/16) + m%16 (tests/umma_probe_mn.cu); accumulated across the tiles of the persistent CTA
//   epi 2  dq = (dX + gw) (.) p -> workspace; (dX + gw) (.) q -> smem scratch -> per-row dp sums
#include <cuda_bf16.h>

#include <cstdlib>

#include "nais_bwd_args.cuh"
#include "nais_pairs_tile.cuh"
#include "umma.cuh"

namespace nais {
namespace ptcb {
using namespace umma;

constexpr int PT = 128;          // threads = cells per tile = TMEM lanes
constexpr int HID = 64;          // hidden_size of this version
constexpr int STG_STRIDE = 144;  // staged row segment: 32 floats + 16 B skew
constexpr int DP_STRIDE = 132;   // cells per d-row of the dp scratch (aliased on the X image)
constexpr uint32_t TMEM_COLS = 256, COL_T = 0, COL_DX = 64, COL_DW = 128;

__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// kind::f16 with bf16 operands, fp32 accumulate; a_mn / b_mn = 1 reads that operand MN-major (transposed)
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// 8 fp32 -> one 16-byte k-chunk per plane.  Two values per conversion (F2FP.BF16.PACK_AB on the ALU pipe; the scalar
// __float2bfloat16_rn is an F2F on the 16-lane conversion unit: 75 of them per thread and work unit were ~20 % of the backward's
// time), hi back to fp32 by a shift / mask: same roundings, same bits as split_bf16.
__device__ __forceinline__ void store_chunk_bf16(uint8_t* hi_plane, uint8_t* lo_plane, size_t off, const float (&v)[8]) {
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);  // .x = low half = v[2e]
    const uint32_t u = *reinterpret_cast<const uint32_t*>(&h2);
    const float ha = __uint_as_float(u << 16), hb = __uint_as_float(u & 0xffff0000u);
    const __nv_bfloat162 l2 = __floats2bfloat162_rn(v[2 * e] - ha, v[2 * e + 1] - hb);
    hi[e] = u;
    lo[e] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  *reinterpret_cast<uint4*>(hi_plane + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(lo_plane + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// Warp-cooperative gather of the 32-float segment [s0, s0+segw) of the 32 history rows of this warp's cells (ids it32 / rg32 held
// per lane) into q[0..segw): whole 128-byte lines per request, staged with a 16-byte skew, read back by the owning lane.
template <int SEGW>
__device__ __forceinline__ void gather_segment(const NaisBranch& br, int it32, int rg32, int s0, uint8_t* stg, int lane, float (&q)[32]) {
  constexpr int P = SEGW / 4;
  float4 v[P];
#pragma unroll
  for (int j = 0; j < P; ++j) {
    const int idx = lane + 32 * j, c = idx / P, part = idx - c * P;
    const int ci = __shfl_sync(0xffffffffu, it32, c), cr = __shfl_sync(0xffffffffu, rg32, c);
    v[j] = ldg_row4(br.hist_poi + (size_t)ci * br.w_poi, br.hist_reg + (size_t)cr * br.w_reg, br.w_poi, s0 + 4 * part);
  }
#pragma unroll
  for (int j = 0; j < P; ++j) {
    const int idx = lane + 32 * j, c = idx / P, part = idx - c * P;
    *reinterpret_cast<float4*>(stg + (size_t)c * STG_STRIDE + part * 16) = v[j];
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < P; ++j) {
    const float4 t = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + j * 16);
    q[4 * j] = t.x;
    q[4 * j + 1] = t.y;
    q[4 * j + 2] = t.z;
    q[4 * j + 3] = t.w;
  }
  __syncwarp();
}

template <int D, bool kDrop, bool kKm>
__global__ void __launch_bounds__(PT, 2) pairs_bwd_tc_kernel(const __grid_constant__ BwdArgs A) {
  static_assert(D == 32 || D == 64, "segments of 32");
  extern __shared__ __align__(128) uint8_t smem[];
  const NaisParams& p = A.p;
  const NaisBranch& br = p.branch[A.bi];
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0, ldw = D + lanes;
  constexpr int XC = D / 8 + 1;                 // k-chunks of the X image: D/8 + the ext chunk [1 g0 g1 0 0 0 0 0]
  constexpr int X_PLANE = XC * PT * 16, W_PLANE = (D / 8) * HID * 16, DT_PLANE = (HID / 8) * PT * 16;
  uint8_t* sX = smem;                           // [hi | lo][XC][128 cells][16 B]      (dp scratch aliases it after GEMM3)
  uint8_t* sW = sX + 2 * X_PLANE;               // [hi | lo][D/8][64 hidden][16 B]
  uint8_t* sDT = sW + 2 * W_PLANE;              // [hi | lo][8][128 cells][16 B]       (row staging aliases it outside GEMM2/3)
  float* kc = reinterpret_cast<float*>(sDT + 2 * DT_PLANE);  // [4][HID] b1, w2, w1[:, D], w1[:, D+1]
  float* ps = kc + 4 * HID;                     // [BWD_MAXROWS][D]
  float* dpacc = ps + BWD_MAXROWS * D;          // [BWD_MAXROWS][D]
  float* rowv = dpacc + BWD_MAXROWS * D;        // [4][BWD_MAXROWS] S, score, G, S^beta
  float* dvs = rowv + 4 * BWD_MAXROWS;          // [4 warps][HID]
  float* red = dvs + 4 * HID;                   // [8][4]
  uint64_t* bar = reinterpret_cast<uint64_t*>(red + 32);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  float* dps = reinterpret_cast<float*>(sX);    // [D][DP_STRIDE]
  static_assert(D * DP_STRIDE * 4 <= 2 * X_PLANE, "dp scratch must fit in the X image");
  static_assert(PT * STG_STRIDE <= 2 * DT_PLANE, "row staging must fit in the DT image");

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tslot, TMEM_COLS);
  for (int i = tid; i < HID * (D / 8); i += PT) {
    const int c = i / HID, k = i - c * HID;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = __ldg(br.w1 + (size_t)k * ldw + c * 8 + e);
    store_chunk_bf16(sW, sW + W_PLANE, ((size_t)c * HID + k) * 16, v);
  }
  for (int k = tid; k < HID; k += PT) {
    kc[k] = __ldg(br.b1 + k);
    kc[HID + k] = __ldg(br.w2 + k);
    kc[2 * HID + k] = lanes ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f;
    kc[3 * HID + k] = lanes ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
  uint8_t* stg = sDT + (size_t)(warp * 32) * STG_STRIDE;

  float pd[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // dist_w[4], dist_b[2] partials of this thread's cells
  float pkm = 0.f, kmc = 0.f;                    // kKm: sum of da * km over this thread's cells; sum_d embed_distance[0, d]
  if constexpr (kKm) kmc = km_coef0(p, D);
  float dv_acc[2] = {0.f, 0.f};                  // dw2 partial of hidden units dv_k0, dv_k0 + 1 over this warp's cells
  const int dv_k0 = 32 * ((lane >> 4) & 1) + 16 * ((lane >> 3) & 1) + 8 * ((lane >> 2) & 1) + 4 * ((lane >> 1) & 1) + 2 * (lane & 1);
  uint32_t phase = 0, dw_started = 0;

  for (int64_t item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    const PairTile T = pair_tile(A.b, item);
    const int64_t row0 = T.row0;
    const int nrows = T.nrows, H = T.H;
    const int n_chunks = (H <= PT) ? 1 : (H + PT - 1) / PT;
    for (int i = tid; i < nrows * D; i += PT) {
      const int r = i / D, d = i - r * D;
      ps[i] = (d < br.w_poi) ? __ldg(br.tgt_poi + (size_t)checked_id(A.b.tgt[row0 + r], p.item_num, A.bad) * br.w_poi + d)
                             : __ldg(br.tgt_reg + (size_t)checked_id(A.b.treg[row0 + r], p.region_num, A.bad) * br.w_reg + (d - br.w_poi));
      dpacc[i] = 0.f;
    }
    if (tid < nrows) {
      const float S = A.row_sum[row0 + tid];
      rowv[tid] = S;
      rowv[BWD_MAXROWS + tid] = A.parts[row0 + tid];
      rowv[2 * BWD_MAXROWS + tid] = A.dscore[row0 + tid];
      rowv[3 * BWD_MAXROWS + tid] = powf(S, p.beta);
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
      const int64_t cidx = valid ? T.cell0 + r * (int64_t)H + h : 0;  // per-cell arrays
      const int64_t hidx = valid ? T.hist0 + r * T.hist_rs + h : 0;   // history arrays
      int it32 = 0, rg32 = 0;
      float l0r = 0.f, l1r = 0.f, km = 0.f;
      bool live = false;
      if (valid) {
        it32 = checked_id(A.b.hist[hidx], p.item_num, A.bad);
        rg32 = br.w_reg ? checked_id(A.b.hreg[hidx], p.region_num, A.bad) : 0;
        if (lanes) pair_latlon(A.b, cidx, hidx, row0 + r, l0r, l1r);
        if constexpr (kKm) km = pair_km(A.b, cidx, hidx, row0 + r);
        live = A.b.hist[hidx] != A.b.tgt[row0 + r];
      }
      float g0 = 0.f, g1 = 0.f;
      if (valid && lanes) {
        const float a0 = l0r * p.dist_scale, a1 = l1r * p.dist_scale;
        g0 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 1), fmaf(a0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0))));
        g1 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 3), fmaf(a0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1))));
      }
      // ---- X image (bf16 hi/lo, unscaled) + similarity -----------------------------------------------------------------------------
      float ssum = 0.f;
      const float* pr = ps + (valid ? r : 0) * D;
#pragma unroll
      for (int s0 = 0; s0 < D; s0 += 32) {
        float q[32];
        gather_segment<32>(br, it32, rg32, s0, stg, lane, q);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            x[e] = valid ? q[c * 8 + e] * pr[s0 + c * 8 + e] : 0.f;
            ssum += x[e];
          }
          store_chunk_bf16(sX, sX + X_PLANE, ((size_t)(s0 / 8 + c) * PT + tid) * 16, x);
        }
      }
      {
        const float ext[8] = {valid ? 1.f : 0.f, g0, g1, 0.f, 0.f, 0.f, 0.f, 0.f};
        store_chunk_bf16(sX, sX + X_PLANE, ((size_t)(D / 8) * PT + tid) * 16, ext);
      }
      fence_proxy_async();
      __syncthreads();  // X image complete; every warp is done with its staging slice (aliased on the DT image)
      // ---- GEMM1: T = X W^T -----------------------------------------------------------------------------------------------------------
      if (warp == 0) {
        if (elect_one()) {
          tc_fence_after();
          const uint32_t x0 = smem_u32(sX), w0 = smem_u32(sW);
          const uint32_t idesc = idesc_bf16(PT, HID, 0, 0);
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint32_t ab = x0 + (pass == 2 ? X_PLANE : 0), wb = w0 + (pass == 1 ? W_PLANE : 0);
#pragma unroll
            for (int s = 0; s < D / 16; ++s)
              mma_f16(tmem + COL_T, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 2 * HID * 16, HID * 16, 128), idesc,
                      (pass | s) != 0);
          }
          mma_commit(bar);
        }
        __syncwarp();
      }
      mbar_wait(bar, phase);
      phase ^= 1u;
      tc_fence_after();
      // ---- epilogue 1: thread = cell = TMEM lane ----------------------------------------------------------------------------------------
      unsigned long long amd = 0ull;  // kDrop: the forward's "active and kept" pattern (a dropped unit counts as t = 0)
      if constexpr (kDrop) amd = valid ? __ldg(A.act_mask + cidx) : 0ull;
      float a = 0.f;
      for (int c0 = 0; c0 < HID; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tlane + COL_T + c0, v);
        tmem_wait_ld16(v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int k = c0 + i;
          float t = __uint_as_float(v[i]) + kc[k];
          if (lanes) t = fmaf(kc[3 * HID + k], g1, fmaf(kc[2 * HID + k], g0, t));
          if constexpr (kDrop) t = ((amd >> k) & 1ull) ? t : 0.f;
          a = fmaf(kc[HID + k], fmaxf(t, 0.f), a);
        }
      }
      if constexpr (kDrop) a *= A.drop_inv;
      if constexpr (kKm) a += __fmul_rn(km, kmc);
      float dav = 0.f, gwv = 0.f;
      if (live) {
        const float S = rowv[r], sc = rowv[BWD_MAXROWS + r], G = rowv[2 * BWD_MAXROWS + r], Sb = rowv[3 * BWD_MAXROWS + r];
        const float e = expf(a);
        const float w = e / Sb;
        dav = G * (w * ssum - p.beta * (e / S) * sc);
        gwv = G * w;
      }
      if constexpr (kKm) pkm = fmaf(dav, km, pkm);  // d logit / d embed_distance[0, d] = km for every d
      if constexpr (kDrop) dav *= A.drop_inv;  // d relu(drop(t)) / dt = m / (1-p)
      // unit step of ReLU: the forward's saved pattern when there is one (its t is accurate to ~2e-7; this kernel's recomputed t,
      // from bf16 two-term splits, only to ~1e-5 — a unit on the kink would flip and move the gradients by this cell's whole term)
      const bool have_mask = kDrop || A.act_mask != nullptr;
      const unsigned long long am = kDrop ? amd : (have_mask && valid) ? __ldg(A.act_mask + cidx) : 0ull;
      float dvv[HID];
      float dg0 = 0.f, dg1 = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < HID; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tlane + COL_T + c0, v);
        tmem_wait_ld16(v);
        float dt[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int k = c0 + i;
          float t = __uint_as_float(v[i]) + kc[k];
          if (lanes) t = fmaf(kc[3 * HID + k], g1, fmaf(kc[2 * HID + k], g0, t));
          if constexpr (kDrop) t = ((am >> k) & 1ull) ? t : 0.f;
          dvv[k] = dav * fmaxf(t, 0.f);
          const bool on = have_mask ? ((am >> k) & 1ull) != 0ull : t > 0.f;
          dt[i] = on ? dav * kc[HID + k] : 0.f;
          dg0 = fmaf(dt[i], kc[2 * HID + k], dg0);
          dg1 = fmaf(dt[i], kc[3 * HID + k], dg1);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float c8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) c8[e] = dt[j * 8 + e];
          store_chunk_bf16(sDT, sDT + DT_PLANE, ((size_t)(c0 / 8 + j) * PT + tid) * 16, c8);
        }
      }
      if (lanes) {  // dist layer: z = Wd (scale * ll) + bd, g = sigmoid(z)
        const float dz0 = dg0 * g0 * (1.f - g0), dz1 = dg1 * g1 * (1.f - g1);
        const float a0 = l0r * p.dist_scale, a1 = l1r * p.dist_scale;
        pd[0] = fmaf(dz0, a0, pd[0]);
        pd[1] = fmaf(dz0, a1, pd[1]);
        pd[2] = fmaf(dz1, a0, pd[2]);
        pd[3] = fmaf(dz1, a1, pd[3]);
        pd[4] += dz0;
        pd[5] += dz1;
      }
      // dw2[k] += sum over this warp's cells of da * relu(t_k): shuffle halving, 62 shuffles for all 64 hidden units
#pragma unroll
      for (int st = 0; st < 5; ++st) {
        const int n = HID >> st, m = 16 >> st;
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < HID / 2; ++i) {
          if (i < n / 2) {
            const float send = up ? dvv[i] : dvv[i + n / 2];
            const float keep = up ? dvv[i + n / 2] : dvv[i];
            dvv[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
          }
        }
      }
      dv_acc[0] += dvv[0];
      dv_acc[1] += dvv[1];
      tc_fence_before();
      fence_proxy_async();
      __syncthreads();  // DT image complete
      // ---- GEMM2: dX = dt W   and   GEMM3: dW += dt^T [X | 1 g0 g1] ---------------------------------------------------------------------
      if (warp == 0) {
        if (elect_one()) {
          tc_fence_after();
          const uint32_t x0 = smem_u32(sX), w0 = smem_u32(sW), t0 = smem_u32(sDT);
          const uint32_t id2 = idesc_bf16(PT, D, 0, 1), id3 = idesc_bf16(HID, D + 8, 1, 1);
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint32_t ab = t0 + (pass == 2 ? DT_PLANE : 0), wb = w0 + (pass == 1 ? W_PLANE : 0);
#pragma unroll
            for (int s = 0; s < HID / 16; ++s)  // K = hidden units 16s..16s+15: DT k-chunks 2s, 2s+1; W image rows 16s.. (+256 B)
              mma_f16(tmem + COL_DX, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 256, 128, HID * 16), id2,
                      (pass | s) != 0);
          }
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint32_t ab = t0 + (pass == 2 ? DT_PLANE : 0), xb = x0 + (pass == 1 ? X_PLANE : 0);
#pragma unroll
            for (int s = 0; s < PT / 16; ++s)  // K = cells 16s..16s+15 of both images (+256 B); mn blocks at the k-chunk stride
              mma_f16(tmem + COL_DW, smem_desc(ab + s * 256, 128, PT * 16), smem_desc(xb + s * 256, 128, PT * 16), id3,
                      (dw_started | pass | s) != 0);
          }
          mma_commit(bar);
        }
        __syncwarp();
      }
      dw_started = 1u;
      mbar_wait(bar, phase);
      phase ^= 1u;
      tc_fence_after();
      // ---- epilogue 2: dq rows to the workspace, dp contributions to the scratch (aliased on the X image) -----------------------------
#pragma unroll
      for (int s0 = 0; s0 < D; s0 += 32) {
        float q[32];
        gather_segment<32>(br, it32, rg32, s0, stg, lane, q);
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(tlane + COL_DX + s0 + c0, v);
          tmem_wait_ld16(v);
          float o[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int d = s0 + c0 + i;
            const float full = __uint_as_float(v[i]) + gwv;
            o[i] = full * pr[d];
            dps[(size_t)d * DP_STRIDE + tid] = valid ? full * q[c0 + i] : 0.f;
          }
          if (valid && A.ws_dq) {
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              *reinterpret_cast<float4*>(A.ws_dq + cidx * D + s0 + c0 + i) = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
          }
        }
      }
      tc_fence_before();
      __syncthreads();
      {
        const int nr = (H <= PT) ? nrows : 1;
        for (int i = tid; i < nr * D; i += PT) {
          const int rr = i / D, d = i - rr * D;
          const int c0 = (H <= PT) ? rr * H : 0;
          const int cn = (H <= PT) ? H : min(PT, H - ch * PT);
          float sacc = 0.f;
          for (int c = 0; c < cn; ++c) sacc += dps[(size_t)d * DP_STRIDE + c0 + c];
          dpacc[rr * D + d] += sacc;
        }
      }
      __syncthreads();  // scratch (X image) and staging (DT image) are free again
    }
    if (A.ws_dp)
      for (int i = tid; i < nrows * D; i += PT) A.ws_dp[(row0 + i / D) * D + (i % D)] = dpacc[i];
    __syncthreads();
  }

  // ---- this CTA's parameter partial: w1 [hid][ldw] | b1 | w2 | dist_w[4] dist_b[2] km pad --------------------------------------------
  float* part = A.ws_part + (size_t)blockIdx.x * A.part_stride;
  tc_fence_after();
  {
    const int m = 16 * warp + (lane & 15);  // the M = 64 accumulator keeps row m in TMEM lane 32*(m/16) + m%16
    for (int c0 = 0; c0 < D + 16; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(tlane + COL_DW + c0, v);
      tmem_wait_ld16(v);
      if (lane < 16) {
        if (c0 < D) {
#pragma unroll
          for (int i = 0; i < 16; ++i) part[(size_t)m * ldw + c0 + i] = __uint_as_float(v[i]);
        } else {  // ext chunk: [sum dt * 1, sum dt * g0, sum dt * g1]
          part[HID * ldw + m] = __uint_as_float(v[0]);
          if (lanes) {
            part[(size_t)m * ldw + D] = __uint_as_float(v[1]);
            part[(size_t)m * ldw + D + 1] = __uint_as_float(v[2]);
          }
        }
      }
    }
  }
  dvs[warp * HID + dv_k0] = dv_acc[0];
  dvs[warp * HID + dv_k0 + 1] = dv_acc[1];
#pragma unroll
  for (int q = 0; q < (kKm ? 7 : 6); ++q) {
    float v = q < 6 ? pd[q] : pkm;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[q * 4 + warp] = v;
  }
  tc_fence_before();
  __syncthreads();
  if (tid < HID) part[HID * ldw + HID + tid] = dvs[tid] + dvs[HID + tid] + dvs[2 * HID + tid] + dvs[3 * HID + tid];
  if (tid < 7)
    part[HID * ldw + 2 * HID + tid] = (tid < 6 || kKm) ? red[tid * 4] + red[tid * 4 + 1] + red[tid * 4 + 2] + red[tid * 4 + 3] : 0.f;
  if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

// =====================================================================================================================
// The headline shape (D = hid = 64) with TWO threads per cell (256 threads, 2 CTAs per SM).
//
// ncu on the 128-thread kernel above at C3 (profiles/r2_ncu_pairs_bwd_tc_summary.csv): 140 M warp instructions, issue slots 24 %
// busy, 8 warps per SM (255 registers x 128 threads x 2 CTAs fills the register file), stalled on the L2 gathers (long
// scoreboard 2.8 per issue) and on TMEM / shared memory (short scoreboard 1.5): a latency-bound kernel with nothing to switch
// to.  Splitting every cell between two threads — warps 0-3 take the first 32 embedding columns / hidden units of a cell, warps
// 4-7 the other 32; warps w and w + 4 share a TMEM lane quarter — halves the per-thread arrays (<= 128 registers), doubles the
// warps in flight and halves the length of each serial phase.  The two halves meet three times per tile: the similarity sum,
// the logit a (needed in full before exp), and the per-row dp reduce.  Same operand images, same MMAs, same workspace outputs.
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

template <bool kDrop, bool kKm>
__global__ void __launch_bounds__(PT2, 2) pairs_bwd_tc2_kernel(const __grid_constant__ BwdArgs A) {
  constexpr int D = 64;
  extern __shared__ __align__(128) uint8_t smem[];
  const NaisParams& p = A.p;
  const NaisBranch& br = p.branch[A.bi];
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0, ldw = D + lanes;
  constexpr int XC = D / 8 + 1;
  constexpr int X_PLANE = XC * PT * 16, W_PLANE = (D / 8) * HID * 16, DT_PLANE = (HID / 8) * PT * 16;
  constexpr int STG_BYTES = 8 * 32 * STG_STRIDE;  // eight warps stage 32 rows each: 36 864 B (the DT image is 32 768 B)
  constexpr int DT_REGION = STG_BYTES > 2 * DT_PLANE ? STG_BYTES : 2 * DT_PLANE;
  uint8_t* sX = smem;                           // [hi | lo][XC][128 cells][16 B]      (dp scratch aliases it after GEMM3)
  uint8_t* sW = sX + 2 * X_PLANE;               // [hi | lo][D/8][64 hidden][16 B]
  uint8_t* sDT = sW + 2 * W_PLANE;              // [hi | lo][8][128 cells][16 B]       (row staging aliases it outside GEMM2/3)
  float* kc = reinterpret_cast<float*>(sDT + DT_REGION);  // [HID] x {b1, w2, w1[:, D], w1[:, D+1]}
  float* ps = kc + 4 * HID;                     // [2][BWD_MAXROWS][D] target vectors of this tile / of the next tile
  float* dpacc = ps + 2 * BWD_MAXROWS * D;      // [BWD_MAXROWS][D] running dp of rows with more than one chunk
  float* rowv = dpacc + BWD_MAXROWS * D;        // [4][BWD_MAXROWS] S, score, G, S^beta
  float* dvs = rowv + 4 * BWD_MAXROWS;          // [4 lane quarters][HID]
  float* red = dvs + 4 * HID;                   // [8][8]
  float* xsum = red + 64;                       // [2][PT] similarity partial of each half
  float* asum = xsum + 2 * PT;                  // [2][PT] logit partial of each half
  // inputs of the NEXT work unit, copied one unit ahead with cp.async (see the loop)
  long long* m_hist = reinterpret_cast<long long*>(asum + 2 * PT);  // [PT] history POI id of each cell      (copied by half 0)
  long long* m_hreg = m_hist + PT;                                  // [PT] its region id                     (half 1)
  unsigned long long* m_mask = reinterpret_cast<unsigned long long*>(m_hreg + PT);  // [PT] ReLU pattern     (half 1)
  long long* m_psid = reinterpret_cast<long long*>(m_mask + PT);    // [PT2] id behind this thread's 16 B of `ps` (private)
  long long* m_tgt = m_psid + PT2;                                  // [BWD_MAXROWS] target POI id of each row (live mask)
  float2* m_ll = reinterpret_cast<float2*>(m_tgt + BWD_MAXROWS);    // [PT] |dlat|,|dlon| (kKm: .x = km) or the history item's coordinates (half 0)
  float2* m_tco = m_ll + PT;                                        // [BWD_MAXROWS] target coordinates (segmented layout)
  float* m_rowv = reinterpret_cast<float*>(m_tco + BWD_MAXROWS);    // [3][BWD_MAXROWS] S, score, dscore of each row
  uint64_t* bar = reinterpret_cast<uint64_t*>(m_rowv + 4 * BWD_MAXROWS);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  float* dps = reinterpret_cast<float*>(sX);    // [D][DP_STRIDE]
  static_assert(D * DP_STRIDE * 4 <= 2 * X_PLANE, "dp scratch must fit in the X image");

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int half = warp >> 2, qd = warp & 3;   // which 32 columns of the cell / which TMEM lane quarter
  const int cell = qd * 32 + lane;             // this thread's cell = TMEM lane
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tslot, TMEM_COLS);
  for (int i = tid; i < HID * (D / 8); i += PT2) {
    const int c = i / HID, k = i - c * HID;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = __ldg(br.w1 + (size_t)k * ldw + c * 8 + e);
    store_chunk_bf16(sW, sW + W_PLANE, ((size_t)c * HID + k) * 16, v);
  }
  for (int k = tid; k < HID; k += PT2)  // one 16-byte load per hidden unit in the epilogue: {b1, w2, w1[:, D], w1[:, D+1]}
    reinterpret_cast<float4*>(kc)[k] = make_float4(__ldg(br.b1 + k), __ldg(br.w2 + k), lanes ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f,
                                                   lanes ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  const uint32_t tlane = tmem + ((uint32_t)(qd * 32) << 16);
  uint8_t* stg = sDT + (size_t)(warp * 32) * STG_STRIDE;
  const int s0 = 32 * half;  // this thread's embedding columns [s0, s0 + 32) and hidden units [s0, s0 + 32)

  // ---- the input pipeline (per-phase clocks of the unpipelined kernel, profiles/r2_phase_clocks_before.txt: 39 % of a tile's
  // time was exposed load latency — target id -> target row, history id -> history row — and another 20 % the second gather).
  // The inputs of work unit u + 1 are copied while unit u computes, with nothing held in registers:
  //   P1 (after u's inputs are consumed)     ids / lat-lon / ReLU mask / row scalars of u + 1       -> m_* arrays
  //   P2 (after u's second gather is staged)  history rows of u + 1 -> `stg` (aliases the DT image, free now); target rows -> ps[next]
  // and u + 1 starts with cp.async.wait_all + one barrier.  The second gather of u's own rows (dp needs them again) is issued
  // into registers BEFORE the wait for GEMM2/3 and staged after it.
  const RowGather RG = row_gather_init(br, s0, lane, stg, STG_STRIDE);
  auto issue_ids = [&](const PairTile& Tn, int chn) {
    const PairCell c = pair_cell(Tn, chn, cell);
    if (c.valid) {
      if (half == 0) {
        cp_async8(m_hist + cell, A.b.hist + c.hidx);
        if (lanes) cp_async8(m_ll + cell, A.b.aux ? A.b.aux + c.cidx * 2 : A.b.hist_coords + c.hidx * 2);
        if (kKm) {  // the dense layout's km, or the history item's coordinates (where the lat/lon lanes stage theirs)
          if (A.b.aux) cp_async4(m_ll + cell, A.b.aux + c.cidx);
          else cp_async8(m_ll + cell, A.b.hist_coords + c.hidx * 2);
        }
      } else {
        if (br.w_reg) cp_async8(m_hreg + cell, A.b.hreg + c.hidx);
        if (A.act_mask) cp_async8(m_mask + cell, A.act_mask + c.cidx);
      }
    }
    if (tid < Tn.nrows) cp_async8(m_tgt + tid, A.b.tgt + Tn.row0 + tid);
    if ((lanes || kKm) && !A.b.aux && tid >= 32 && tid < 32 + Tn.nrows)
      cp_async8(m_tco + (tid - 32), A.b.tgt_coords + (Tn.row0 + tid - 32) * 2);
    if (chn == 0) {
      if (tid >= 64 && tid < 64 + Tn.nrows) {
        const int rr = tid - 64;
        cp_async4(m_rowv + rr, A.row_sum + Tn.row0 + rr);
        cp_async4(m_rowv + BWD_MAXROWS + rr, A.parts + Tn.row0 + rr);
        cp_async4(m_rowv + 2 * BWD_MAXROWS + rr, A.dscore + Tn.row0 + rr);
      }
      if (tid * 4 < Tn.nrows * D) {
        const int r = (tid * 4) / D, d = tid * 4 - r * D;
        cp_async8(m_psid + tid, (d < br.w_poi ? A.b.tgt : A.b.treg) + Tn.row0 + r);
      }
    }
  };
  auto issue_rows = [&](const PairTile& Tn, int chn, int pbn) {  // (after cp_async_wait_all + a barrier: the ids are visible)
    const PairCell c = pair_cell(Tn, chn, cell);
    int it32 = 0, rg32 = 0;
    if (c.valid) {
      it32 = checked_id(m_hist[cell], p.item_num, A.bad);
      rg32 = br.w_reg ? checked_id(m_hreg[cell], p.region_num, A.bad) : 0;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) cp_async16(RG.dst + (uint32_t)(q * 4 * STG_STRIDE), row_gather_src(RG, it32, rg32, q));
    if (chn == 0 && tid * 4 < Tn.nrows * D) {
      const int r = (tid * 4) / D, d = tid * 4 - r * D;
      const float* src = d < br.w_poi ? br.tgt_poi + (size_t)checked_id(m_psid[tid], p.item_num, A.bad) * br.w_poi + d
                                      : br.tgt_reg + (size_t)checked_id(m_psid[tid], p.region_num, A.bad) * br.w_reg + (d - br.w_poi);
      cp_async16(ps + (size_t)pbn * BWD_MAXROWS * D + tid * 4, src);
    }
  };

  float pd[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // dist_w[4], dist_b[2] partials (this thread's hidden units of its cells)
  float pkm = 0.f, kmc = 0.f;                    // kKm: sum of da * km over this thread's cells (half 0); sum_d embed_distance[0, d]
  if constexpr (kKm) kmc = km_coef0(p, D);
  float dv_acc = 0.f;                            // dw2 partial of hidden unit s0 + lane over this warp's cells
  uint32_t phase = 0, dw_started = 0;
  int64_t item = blockIdx.x;  // (the launch gives every CTA at least one tile)
  int ch = 0, pb = 0;
  NAIS_PH_INIT
  {
    const PairTile T0 = pair_tile(A.b, item);
    issue_ids(T0, 0);
    cp_async_wait_all();
    __syncthreads();
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
    const int64_t cidx = c.cidx;
    const bool same = ch + 1 < n_chunks;               // the next unit: the next chunk of this tile, or this CTA's next tile
    const int64_t item_n = same ? item : item + gridDim.x;
    const int ch_n = same ? ch + 1 : 0, pb_n = same ? pb : pb ^ 1;
    const bool has_next = item_n < A.n_items;

    cp_async_wait_all();
    __syncthreads();  // (a) this unit's rows, ids, lat/lon, mask, row scalars and target vectors are in shared memory
    NAIS_PH(1)
    if (ch == 0 && tid < nrows) {
      const float S = m_rowv[tid];
      rowv[tid] = S;
      rowv[BWD_MAXROWS + tid] = m_rowv[BWD_MAXROWS + tid];
      rowv[2 * BWD_MAXROWS + tid] = m_rowv[2 * BWD_MAXROWS + tid];
      rowv[3 * BWD_MAXROWS + tid] = powf(S, p.beta);
    }
    int it32 = 0, rg32 = 0;
    float l0r = 0.f, l1r = 0.f, g0 = 0.f, g1 = 0.f, km = 0.f;
    bool live = false;
    uint32_t am32 = 0u;
    if (valid) {
      const long long hid64 = m_hist[cell];
      it32 = checked_id(hid64, p.item_num, A.bad);
      rg32 = br.w_reg ? checked_id(m_hreg[cell], p.region_num, A.bad) : 0;
      if (lanes) {
        const float2 hl = m_ll[cell];
        l0r = hl.x;
        l1r = hl.y;
        if (!A.b.aux) {  // (pair_latlon of the segmented layout)
          const float2 tc = m_tco[r];
          l0r = fabsf(tc.x - hl.x);
          l1r = fabsf(tc.y - hl.y);
        }
        const float a0 = l0r * p.dist_scale, a1 = l1r * p.dist_scale;
        g0 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 1), fmaf(a0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0))));
        g1 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 3), fmaf(a0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1))));
      }
      if (kKm) {  // both threads of the cell form the same km (pair_km: the same dist_km_f call on the same coordinates)
        const float2 hl = m_ll[cell];
        km = hl.x;
        if (!A.b.aux) {
          const float2 tc = m_tco[r];
          km = coords_km(A.b, tc.x, tc.y, hl.x, hl.y);
        }
      }
      live = hid64 != m_tgt[r];
      if (A.act_mask) am32 = (uint32_t)(m_mask[cell] >> s0);  // this half's 32 hidden units
    }
    // ---- this half of the X image (bf16 hi/lo, unscaled) + similarity partial -------------------------------------------------------
    const float* pr = ps + (size_t)pb * BWD_MAXROWS * D + (valid ? r : 0) * D;
    {
      float ssum = 0.f;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const float4 q0 = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + cc * 32);
        const float4 q1 = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + cc * 32 + 16);
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          x[e] = valid ? qv[e] * pr[s0 + cc * 8 + e] : 0.f;
          ssum += x[e];
        }
        store_chunk_bf16(sX, sX + X_PLANE, ((size_t)(s0 / 8 + cc) * PT + cell) * 16, x);
      }
      xsum[half * PT + cell] = ssum;
      if (half == 0) {
        const float ext[8] = {valid ? 1.f : 0.f, g0, g1, 0.f, 0.f, 0.f, 0.f, 0.f};
        store_chunk_bf16(sX, sX + X_PLANE, ((size_t)(D / 8) * PT + cell) * 16, ext);
      }
    }
    fence_proxy_async();
    NAIS_PH(2)
    __syncthreads();  // (b) X image complete; the staged rows and the m_* arrays are consumed
    NAIS_PH(3)
    // ---- GEMM1: T = X W^T -----------------------------------------------------------------------------------------------------------
    if (warp == 0) {
      if (elect_one()) {
        tc_fence_after();
        const uint32_t x0 = smem_u32(sX), w0 = smem_u32(sW);
        const uint32_t idesc = idesc_bf16(PT, HID, 0, 0);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t ab = x0 + (pass == 2 ? X_PLANE : 0), wb = w0 + (pass == 1 ? W_PLANE : 0);
#pragma unroll
          for (int s = 0; s < D / 16; ++s)
            mma_f16(tmem + COL_T, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 2 * HID * 16, HID * 16, 128), idesc,
                    (pass | s) != 0);
        }
        mma_commit(bar);
      }
      __syncwarp();
    }
    if (has_next) issue_ids(same ? T : pair_tile(A.b, item_n), ch_n);  // P1
    const float ssum = xsum[cell] + xsum[PT + cell];  // (the same sum, in the same order, in both threads of the cell)
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after();
    NAIS_PH(4)
    // ---- epilogue 1: this thread's 32 hidden units of its cell -------------------------------------------------------------------------
    float tv[32];
    {
      float ap = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tlane + COL_T + s0 + c0, v);
        tmem_wait_ld16(v);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float4 c4 = reinterpret_cast<const float4*>(kc)[s0 + c0 + i];
          float t = __uint_as_float(v[i]) + c4.x;
          if (lanes) t = fmaf(c4.w, g1, fmaf(c4.z, g0, t));
          if constexpr (kDrop) t = ((am32 >> (c0 + i)) & 1u) ? t : 0.f;  // the forward's "active and kept" pattern
          tv[c0 + i] = t;
          ap = fmaf(c4.y, fmaxf(t, 0.f), ap);
        }
      }
      asum[half * PT + cell] = kDrop ? ap * A.drop_inv : ap;
    }
    asm volatile("bar.sync %0, 64;" ::"r"(1 + qd) : "memory");  // the two warps of this lane quarter exchange their halves of a
    NAIS_PH(5)
    float a = asum[cell] + asum[PT + cell];
    if constexpr (kKm) a += __fmul_rn(km, kmc);
    float dav = 0.f, gwv = 0.f;
    if (live) {
      const float S = rowv[r], sc = rowv[BWD_MAXROWS + r], G = rowv[2 * BWD_MAXROWS + r], Sb = rowv[3 * BWD_MAXROWS + r];
      const float e = expf(a);
      const float w = e / Sb;
      dav = G * (w * ssum - p.beta * (e / S) * sc);
      gwv = G * w;
    }
    if constexpr (kKm) pkm = half == 0 ? fmaf(dav, km, pkm) : 0.f;
    if constexpr (kDrop) dav *= A.drop_inv;  // d relu(drop(t)) / dt = m / (1-p)
    const bool have_mask = kDrop || A.act_mask != nullptr;
    float dg0 = 0.f, dg1 = 0.f;
#pragma unroll
    for (int c0 = 0; c0 < 32; c0 += 16) {
      float dt[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int k = s0 + c0 + i;
        const float4 c4 = reinterpret_cast<const float4*>(kc)[k];
        const float t = tv[c0 + i];
        const bool on = have_mask ? ((am32 >> (c0 + i)) & 1u) != 0u : t > 0.f;
        tv[c0 + i] = dav * fmaxf(t, 0.f);  // -> dw2 contribution of this cell
        dt[i] = on ? dav * c4.y : 0.f;
        dg0 = fmaf(dt[i], c4.z, dg0);
        dg1 = fmaf(dt[i], c4.w, dg1);
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        float c8[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) c8[e] = dt[j * 8 + e];
        store_chunk_bf16(sDT, sDT + DT_PLANE, ((size_t)((s0 + c0) / 8 + j) * PT + cell) * 16, c8);
      }
    }
    if (lanes) {  // dist layer: z = Wd (scale * ll) + bd, g = sigmoid(z); linear in dg, so the halves' partials simply add up
      const float dz0 = dg0 * g0 * (1.f - g0), dz1 = dg1 * g1 * (1.f - g1);
      const float a0 = l0r * p.dist_scale, a1 = l1r * p.dist_scale;
      pd[0] = fmaf(dz0, a0, pd[0]);
      pd[1] = fmaf(dz0, a1, pd[1]);
      pd[2] = fmaf(dz1, a0, pd[2]);
      pd[3] = fmaf(dz1, a1, pd[3]);
      pd[4] += dz0;
      pd[5] += dz1;
    }
    // dw2[s0 + k] += sum over this warp's 32 cells of da * relu(t_k): shuffle halving, lane l ends with hidden unit s0 + l
#pragma unroll
    for (int st = 0; st < 5; ++st) {
      const int n = 32 >> st, m = 16 >> st;
      const bool up = (lane & m) != 0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (i < n / 2) {
          const float send = up ? tv[i] : tv[i + n / 2];
          const float keep = up ? tv[i + n / 2] : tv[i];
          tv[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
        }
      }
    }
    dv_acc += tv[0];
    tc_fence_before();
    fence_proxy_async();
    __syncthreads();  // (c) DT image complete
    NAIS_PH(6)
    // ---- GEMM2: dX = dt W   and   GEMM3: dW += dt^T [X | 1 g0 g1] ---------------------------------------------------------------------
    if (warp == 0) {
      if (elect_one()) {
        tc_fence_after();
        const uint32_t x0 = smem_u32(sX), w0 = smem_u32(sW), t0 = smem_u32(sDT);
        const uint32_t id2 = idesc_bf16(PT, D, 0, 1), id3 = idesc_bf16(HID, D + 8, 1, 1);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t ab = t0 + (pass == 2 ? DT_PLANE : 0), wb = w0 + (pass == 1 ? W_PLANE : 0);
#pragma unroll
          for (int s = 0; s < HID / 16; ++s)
            mma_f16(tmem + COL_DX, smem_desc(ab + s * 2 * PT * 16, PT * 16, 128), smem_desc(wb + s * 256, 128, HID * 16), id2,
                    (pass | s) != 0);
        }
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t ab = t0 + (pass == 2 ? DT_PLANE : 0), xb = x0 + (pass == 1 ? X_PLANE : 0);
#pragma unroll
          for (int s = 0; s < PT / 16; ++s)
            mma_f16(tmem + COL_DW, smem_desc(ab + s * 256, 128, PT * 16), smem_desc(xb + s * 256, 128, PT * 16), id3,
                    (dw_started | pass | s) != 0);
        }
        mma_commit(bar);
      }
      __syncwarp();
    }
    dw_started = 1u;
    // second gather of this unit's history rows, in flight while the MMAs run (the staging aliases the DT image they read)
    float4 gv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) gv[q] = __ldg(reinterpret_cast<const float4*>(row_gather_src(RG, it32, rg32, q)));
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after();
    NAIS_PH(7)
    // ---- epilogue 2: this half of the dq row to the workspace, dp contributions to the scratch (aliased on the X image) --------------
    {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(RG.dst + (uint32_t)(q * 4 * STG_STRIDE)), "f"(gv[q].x), "f"(gv[q].y),
                     "f"(gv[q].z), "f"(gv[q].w)
                     : "memory");
      __syncwarp();
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tlane + COL_DX + s0 + c0, v);
        float qv[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 t = *reinterpret_cast<const float4*>(stg + (size_t)lane * STG_STRIDE + (c0 + 4 * j) * 4);
          qv[4 * j] = t.x;
          qv[4 * j + 1] = t.y;
          qv[4 * j + 2] = t.z;
          qv[4 * j + 3] = t.w;
        }
        tmem_wait_ld16(v);
        float o[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int d = s0 + c0 + i;
          const float full = __uint_as_float(v[i]) + gwv;
          o[i] = full * pr[d];
          dps[(size_t)d * DP_STRIDE + cell] = valid ? full * qv[i] : 0.f;
        }
        if (valid && A.ws_dq) {
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(A.ws_dq + cidx * D + s0 + c0 + i) = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
        }
      }
    }
    if (has_next) cp_async_wait_all();  // (this thread's id copies of the next unit; visible to the others after the barrier)
    tc_fence_before();
    NAIS_PH(8)
    __syncthreads();  // (d) dp scratch complete; staging read back by every warp; next ids visible
    NAIS_PH(9)
    if (has_next) issue_rows(same ? T : pair_tile(A.b, item_n), ch_n, pb_n);  // P2
    // ---- dp of the rows: four threads per (row, column) sum interleaved cells (bank-conflict free), the first keeps the running sum ----
    {
      const int nr = (H <= PT) ? nrows : 1;
      const int cn = (H <= PT) ? H : min(PT, H - ch * PT);
      for (int i = tid; i < nr * D * 4; i += PT2) {  // (nr * D * 4 is a multiple of 32: whole warps iterate together)
        const int part = i & 3, rd = i >> 2, rr = rd / D, d = rd - rr * D;
        const int c0 = (H <= PT) ? rr * H : 0;
        float sacc = 0.f;
        for (int cc = part; cc < cn; cc += 4) sacc += dps[(size_t)d * DP_STRIDE + c0 + cc];
        sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
        sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
        if (part == 0) {
          if (ch > 0) sacc += dpacc[rd];
          if (same) dpacc[rd] = sacc;
          else if (A.ws_dp) A.ws_dp[(row0 + rr) * D + d] = sacc;
        }
      }
    }
    NAIS_PH(10)
    if (!has_next) break;
    item = item_n;
    ch = ch_n;
    pb = pb_n;
  }

  // ---- this CTA's parameter partial: w1 [hid][ldw] | b1 | w2 | dist_w[4] dist_b[2] km pad --------------------------------------------
  float* part = A.ws_part + (size_t)blockIdx.x * A.part_stride;
  tc_fence_after();
  if (half == 0) {
    const int m = 16 * qd + (lane & 15);  // the M = 64 accumulator keeps row m in TMEM lane 32*(m/16) + m%16
    for (int c0 = 0; c0 < D + 16; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(tlane + COL_DW + c0, v);
      tmem_wait_ld16(v);
      if (lane < 16) {
        if (c0 < D) {
#pragma unroll
          for (int i = 0; i < 16; ++i) part[(size_t)m * ldw + c0 + i] = __uint_as_float(v[i]);
        } else {  // ext chunk: [sum dt * 1, sum dt * g0, sum dt * g1]
          part[HID * ldw + m] = __uint_as_float(v[0]);
          if (lanes) {
            part[(size_t)m * ldw + D] = __uint_as_float(v[1]);
            part[(size_t)m * ldw + D + 1] = __uint_as_float(v[2]);
          }
        }
      }
    }
  }
  dvs[qd * HID + s0 + lane] = dv_acc;
#pragma unroll
  for (int q = 0; q < (kKm ? 7 : 6); ++q) {
    float v = q < 6 ? pd[q] : pkm;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[q * 8 + warp] = v;
  }
  tc_fence_before();
  __syncthreads();
  if (tid < HID) part[HID * ldw + HID + tid] = dvs[tid] + dvs[HID + tid] + dvs[2 * HID + tid] + dvs[3 * HID + tid];
  if (tid < 7) {
    float v = 0.f;
    if (tid < 6 || kKm)
      for (int w = 0; w < 8; ++w) v += red[tid * 8 + w];
    part[HID * ldw + 2 * HID + tid] = v;
  }
  if (warp == 0) tmem_dealloc(tmem, TMEM_COLS);
}

template <bool kDrop, bool kKm>
static int launch2(const BwdArgs& A, int grid, cudaStream_t stream) {
  constexpr int D = 64;
  constexpr size_t dt_region = (8 * 32 * STG_STRIDE > 2 * (HID / 8) * PT * 16) ? 8 * 32 * STG_STRIDE : 2 * (HID / 8) * PT * 16;
  constexpr size_t smem = 2 * (size_t)(D / 8 + 1) * PT * 16 + 2 * (size_t)(D / 8) * HID * 16 + dt_region +
                          (4 * HID + 3 * BWD_MAXROWS * D + 4 * BWD_MAXROWS + 4 * HID + 64 + 4 * PT) * 4 +
                          (3 * (size_t)PT + PT2 + BWD_MAXROWS) * 8 + ((size_t)PT + BWD_MAXROWS) * 8 + 4 * BWD_MAXROWS * 4 + 16;
  static_assert(2 * (smem + 1024) <= 228 * 1024, "two CTAs per SM");
  static SmemAttrOnce attr;
  cudaError_t e = attr(pairs_bwd_tc2_kernel<kDrop, kKm>, smem, true);
  if (e != cudaSuccess) return (int)e;
  pairs_bwd_tc2_kernel<kDrop, kKm><<<grid, PT2, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

template <int D, bool kDrop, bool kKm>
static int launch(const BwdArgs& A, int grid, cudaStream_t stream) {
  constexpr size_t smem = 2 * (size_t)(D / 8 + 1) * PT * 16 + 2 * (size_t)(D / 8) * HID * 16 + 2 * (size_t)(HID / 8) * PT * 16 +
                          (4 * HID + 2 * BWD_MAXROWS * D + 4 * BWD_MAXROWS + 4 * HID + 32) * 4 + 16;
  cudaError_t e = cudaFuncSetAttribute(pairs_bwd_tc_kernel<D, kDrop, kKm>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(pairs_bwd_tc_kernel<D, kDrop, kKm>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return (int)e;
  pairs_bwd_tc_kernel<D, kDrop, kKm><<<grid, PT, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// D = 64: two threads per cell when each 32-column half of a row lies in one table (every shipped model class)
template <bool kDrop, bool kKm>
static int launch_shape(const BwdArgs& A, int D, int grid, cudaStream_t stream) {
  if (D == 32) return launch<32, kDrop, kKm>(A, grid, stream);
  return pair_gather_uniform(A.p.branch[A.bi]) ? launch2<kDrop, kKm>(A, grid, stream) : launch<64, kDrop, kKm>(A, grid, stream);
}

}  // namespace ptcb

// One branch (lat/lon or no distance mode, dropout or not), or the disentangled two (no distance mode or km, no dropout)
bool pairs_tc_bwd_supported(const NaisParams& p, const NaisPairs& b) {
  if (b.B < 1 || p.hid != ptcb::HID) return false;
  const bool two = pairs_disentangled(p);
  if (p.n_branch != 1 && !two) return false;
  if (p.dist_mode == NAIS_DIST_KM && !two) return false;
  if (two && p.dropout_p > 0.f) return false;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const NaisBranch& br = p.branch[bi];
    const int D = br.w_poi + br.w_reg;
    if (D != 32 && D != 64) return false;
    if (!rows_vec4(br, 4)) return false;
  }
  return device_info().major == 10;
}

// grid <= 2 CTAs per SM (256 TMEM columns each); every CTA owns at least one tile (the caller passes min(n_items, grid)).  With
// dropout A.act_mask must be the forward's pattern (PairsBwd::finish runs the FP32 kernel instead when it is NULL).
int launch_pairs_bwd_tc(const BwdArgs& A, int D, int grid, cudaStream_t stream) {
  if (A.p.dropout_p > 0.f) return A.act_mask ? ptcb::launch_shape<true, false>(A, D, grid, stream) : NAIS_ERR_NULL;
  if (A.p.dist_mode == NAIS_DIST_KM) return ptcb::launch_shape<false, true>(A, D, grid, stream);
  return ptcb::launch_shape<false, false>(A, D, grid, stream);
}

}  // namespace nais

#ifdef NAIS_PHASE_CLOCKS
extern "C" __attribute__((visibility("default"))) int nais_debug_phase_bwd(unsigned long long* host16, int reset) {
  cudaError_t e = cudaMemcpyFromSymbol(host16, nais::ptcb::g_phase_clk, sizeof(unsigned long long) * 16);
  if (e == cudaSuccess && reset) {
    unsigned long long z[16] = {};
    e = cudaMemcpyToSymbol(nais::ptcb::g_phase_clk, z, sizeof(z));
  }
  return (int)e;
}
#endif
