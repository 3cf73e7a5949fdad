// Backward of the pair scorer (FP32): recompute-based, atomics-free.
//
//   pairs_bwd_kernel   per 128-cell tile: recompute t = W x + ..., logits, softmax weights -> da, dt;
//                      dW += dt^T x (register-resident across the tiles of a persistent CTA), dX = dt W,
//                      per-cell dq = (dX + G w) (.) p  -> workspace, per-row dp = sum_h (dX + G w) (.) q -> workspace
//   param_reduce       deterministic sum of the per-CTA parameter partials
//   segment_reduce     embedding-row gradients: contributions sorted by row id (cub radix sort), one warp per run of
//                      equal keys sums its rows and writes the table row once — no atomics, bitwise reproducible.
//
// Math (SURVEY.md §7 'Backward'):  dscore/da_h = w_h s_h - beta (E_h/S) score ;  dt_k = da v_k [t_k > 0]
#include <cub/device/device_radix_sort.cuh>
#include <mutex>

#include "nais_bwd_args.cuh"
#include "nais_common.cuh"
#include "nais_pairs_tile.cuh"

namespace nais {



// nais_pairs_tc_bwd.cu: same workspace outputs as pairs_bwd_kernel
bool pairs_tc_bwd_supported(const NaisParams& p, const NaisPairs& b);
int launch_pairs_bwd_tc(const BwdArgs& A, int D, int grid, cudaStream_t stream);

template <int NKB, int DB>
__global__ void __launch_bounds__(NT, (NKB * DB <= 1) ? 2 : 1) pairs_bwd_kernel(const __grid_constant__ BwdArgs A) {
  extern __shared__ __align__(16) float smem[];
  const NaisParams& p = A.p;
  const NaisBranch& br = p.branch[A.bi];
  const int D = br.w_poi + br.w_reg, hid = p.hid;
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0;
  const int ldw = D + lanes;
  constexpr int HP = NKB * KB;

  float* As = smem;                          // [D][TCP] x, later dp contributions
  float* DTs = As + (size_t)D * TCP;         // [HP][TCP] dt
  float* Wt = DTs + (size_t)HP * TCP;        // [D][KB]   W^T k-block
  float* kc = Wt + (size_t)D * KB;           // [NKB][4][KB]
  float* g = kc + NKB * 4 * KB;              // [2][TC] lanes (or km in g[0])
  float* llc = g + 2 * TC;                   // [2][TC] raw |dlat|,|dlon| (LATLON) for dWd
  float* sp = llc + 2 * TC;                  // [2][TC]
  float* gw = sp + 2 * TC;                   // [TC] G * w
  float* dac = gw + TC;                      // [TC] da
  float* dvp = dac + TC;                     // [16][HP] dv partials
  float* ps = dvp + 16 * HP;                 // [BWD_MAXROWS][D]
  float* dpacc = ps + BWD_MAXROWS * D;       // [BWD_MAXROWS][D]
  float* rowv = dpacc + BWD_MAXROWS * D;     // [4][BWD_MAXROWS] S, score, G, S^beta
  float* red = rowv + 4 * BWD_MAXROWS;       // [8][NT/32] final block reduce scratch
  int* citem = reinterpret_cast<int*>(red + 8 * (NT / 32));  // [TC] history item id per cell
  int* creg = citem + TC;                                   // [TC]
  int* crow = creg + TC;                                    // [TC] row slot per cell (-1 invalid)
  long long* cgl = reinterpret_cast<long long*>(crow + TC);  // [TC] global cell index (dropout mask, dq positions)
  int* cmask = reinterpret_cast<int*>(cgl + TC);             // [TC] history item != target
  const uint32_t dthresh = p.dropout_p > 0.f ? dropout_threshold(p.dropout_p) : 0u;
  const float dinv = p.dropout_p > 0.f ? 1.f / (1.f - p.dropout_p) : 1.f;

  const int tid = threadIdx.x, cell = tid & (TC - 1), half = tid >> 7;
  const int tk = tid & 15, tj = tid >> 4;
  const bool vec4 = rows_vec4(br, D >> 1);  // 128-bit embedding-row gathers
  const bool w1_vec2 = (reinterpret_cast<uintptr_t>(br.w1) & 7u) == 0;  // ldw = D + lanes is even: rows of W are 8-byte aligned

  // persistent accumulators
  float acc3[NKB * DB][4][4];
#pragma unroll
  for (int s = 0; s < NKB * DB; ++s)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc3[s][i][j] = 0.f;
  float pb = 0.f, pv = 0.f, pl0 = 0.f, pl1 = 0.f;  // thread k < HP: db1, dw2, dW[:,D], dW[:,D+1]
  float pd[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // thread = cell: dist_w[4], dist_b[2], km

  float km_c = 0.f;
  if (p.dist_mode == NAIS_DIST_KM) {
    for (int d = 0; d < D; ++d) km_c += __ldg(p.dist_embed + d);
  }
  // constants for all k-blocks
  for (int i = tid; i < NKB * KB; i += NT) {
    const int kbi = i / KB, kk = i - kbi * KB, k = i;
    const bool ok = k < hid;
    float* c = kc + kbi * 4 * KB;
    c[kk] = ok ? __ldg(br.b1 + k) : 0.f;
    c[KB + kk] = ok ? __ldg(br.w2 + k) : 0.f;
    c[2 * KB + kk] = (ok && lanes) ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f;
    c[3 * KB + kk] = (ok && lanes) ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f;
  }
  int resident = -1;

  for (int64_t item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    const PairTile T = pair_tile(A.b, item);
    const int64_t row0 = T.row0;
    const int nrows = T.nrows, H = T.H;
    const int n_chunks = (H <= TC) ? 1 : (H + TC - 1) / TC;
    __syncthreads();
    for (int i = tid; i < nrows * D; i += NT) {
      int r = i / D, d = i - r * D;
      ps[r * D + d] = (d < br.w_poi) ? __ldg(br.tgt_poi + (size_t)checked_id(A.b.tgt[row0 + r], p.item_num, A.bad) * br.w_poi + d)
                                     : __ldg(br.tgt_reg + (size_t)checked_id(A.b.treg[row0 + r], p.region_num, A.bad) * br.w_reg + (d - br.w_poi));
      dpacc[r * D + d] = 0.f;
    }
    if (tid < nrows) {
      const float S_row = A.row_sum[row0 + tid];
      rowv[tid] = S_row;
      rowv[3 * BWD_MAXROWS + tid] = powf(S_row, p.beta);  // once per row instead of once per (cell, hidden-lane)
      rowv[BWD_MAXROWS + tid] = A.parts[row0 + tid];
      rowv[2 * BWD_MAXROWS + tid] = A.dscore[row0 + tid];
    }
    for (int ch = 0; ch < n_chunks; ++ch) {
      __syncthreads();
      int r, h;
      bool valid;
      if (H <= TC) {
        r = cell / H;
        h = cell - r * H;
        valid = r < nrows;
      } else {
        r = 0;
        h = ch * TC + cell;
        valid = h < H;
      }
      const int64_t cidx = valid ? T.cell0 + r * (int64_t)H + h : 0;  // per-cell arrays
      const int64_t hidx = valid ? T.hist0 + r * T.hist_rs + h : 0;   // history arrays
      // ---- build x, similarity, lanes -------------------------------------------------------------------------
      {
        const int d0 = half ? (D >> 1) : 0, d1 = half ? D : (D >> 1);
        float ssum = 0.f;
        int64_t it = 0, rg = 0;
        if (valid) {
          it = checked_id(A.b.hist[hidx], p.item_num, A.bad);
          rg = br.w_reg ? checked_id(A.b.hreg[hidx], p.region_num, A.bad) : 0;
          const float* qp = br.hist_poi + (size_t)it * br.w_poi;
          const float* qr = br.hist_reg + (size_t)rg * br.w_reg;
          if (vec4) {  // 128-bit row loads (same products, same summation order as the scalar walk and as the forward)
            const float* pr = ps + r * D;
#pragma unroll 4
            for (int d = d0; d < d1; d += 4) {
              const float4 q = ldg_row4(qp, qr, br.w_poi, d);
              const float4 t = *reinterpret_cast<const float4*>(pr + d);
              const float x0 = q.x * t.x, x1 = q.y * t.y, x2 = q.z * t.z, x3 = q.w * t.w;
              As[d * TCP + cell] = x0;
              As[(d + 1) * TCP + cell] = x1;
              As[(d + 2) * TCP + cell] = x2;
              As[(d + 3) * TCP + cell] = x3;
              ssum += x0;
              ssum += x1;
              ssum += x2;
              ssum += x3;
            }
          } else {
            for (int d = d0; d < d1; ++d) {
              float q = (d < br.w_poi) ? __ldg(qp + d) : __ldg(qr + d - br.w_poi);
              float x = q * ps[r * D + d];
              As[d * TCP + cell] = x;
              ssum += x;
            }
          }
        } else {
          for (int d = d0; d < d1; ++d) As[d * TCP + cell] = 0.f;
        }
        sp[half * TC + cell] = ssum;
        if (half == 0) {
          float g0 = 0.f, g1 = 0.f, l0 = 0.f, l1 = 0.f;
          if (valid && lanes) {
            pair_latlon(A.b, cidx, hidx, row0 + r, l0, l1);
            const float a0 = l0 * p.dist_scale, a1 = l1 * p.dist_scale;
            g0 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 1), fmaf(a0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0))));
            g1 = sigmoidf_exact(fmaf(a1, __ldg(p.dist_w + 3), fmaf(a0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1))));
          } else if (valid && p.dist_mode == NAIS_DIST_KM) {
            l0 = pair_km(A.b, cidx, hidx, row0 + r);
            g0 = l0 * km_c;
          }
          g[cell] = g0;
          g[TC + cell] = g1;
          llc[cell] = l0;
          llc[TC + cell] = l1;
          citem[cell] = (int)it;
          creg[cell] = (int)rg;
          crow[cell] = valid ? r : -1;
          cgl[cell] = cidx;
          cmask[cell] = valid && A.b.hist[hidx] != A.b.tgt[row0 + r];  // history item != target (model.py:299-302)
        }
      }
      __syncthreads();
      // ---- GEMM1: t[cell][k] for all k-blocks, kept in registers ----------------------------------------------
      float t[NKB][8][4];
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        if (resident != kb) {
          __syncthreads();
          for (int i = tid; i < D * KB; i += NT) {
            const int d = i / KB, kk = i - d * KB;  // consecutive threads -> consecutive smem words (no bank conflicts)
            int k = kb * KB + kk;
            Wt[d * KB + kk] = (k < hid) ? __ldg(br.w1 + (size_t)k * ldw + d) : 0.f;
          }
          resident = kb;
          __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) t[kb][i][c] = 0.f;
        const float* ap = As + tj * 8;
        const float* bp = Wt + tk * 4;
#pragma unroll 4
        for (int d = 0; d < D; ++d) {
          float4 a0 = *reinterpret_cast<const float4*>(ap + d * TCP);
          float4 a1 = *reinterpret_cast<const float4*>(ap + d * TCP + 4);
          float4 b = *reinterpret_cast<const float4*>(bp + d * KB);
          const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
          const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) t[kb][i][c] = fmaf(av[i], bv[c], t[kb][i][c]);
        }
      }
      // bias + lanes, relu, logits
      float a_part[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) a_part[i] = 0.f;
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        const float* c = kc + kb * 4 * KB + tk * 4;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float g0 = lanes ? g[tj * 8 + i] : 0.f, g1 = lanes ? g[TC + tj * 8 + i] : 0.f;
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            float v = t[kb][i][cc] + c[cc];
            if (lanes) v = fmaf(c[3 * KB + cc], g1, fmaf(c[2 * KB + cc], g0, v));
            if (dthresh) {
              const uint64_t idx = (uint64_t)cgl[tj * 8 + i] * (uint64_t)hid + (uint64_t)(kb * KB + tk * 4 + cc);
              v = dropout_bits(p.dropout_seed, idx) >= dthresh ? v * dinv : 0.f;
            }
            v = fmaxf(v, 0.f);
            t[kb][i][cc] = v;  // relu(t)
            a_part[i] = fmaf(c[KB + cc], v, a_part[i]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float v = a_part[i];
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        a_part[i] = v;
      }
      // da per cell (all 16 tk-lanes compute the same value), dt -> DTs, dv partials
      float da[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = tj * 8 + i;
        const int rr = crow[c];
        float dav = 0.f, gwv = 0.f;
        if (rr >= 0) {
          float a = a_part[i];
          if (p.dist_mode == NAIS_DIST_KM) a += g[c];
          const bool m = cmask[c] != 0;
          if (m) {
            const float S = rowv[rr], sc = rowv[BWD_MAXROWS + rr], G = rowv[2 * BWD_MAXROWS + rr];
            const float e = expf(a);
            const float w = e / rowv[3 * BWD_MAXROWS + rr];
            const float s = sp[c] + sp[TC + c];
            dav = G * (w * s - p.beta * (e / S) * sc);
            gwv = G * w;
          }
        }
        da[i] = dav;
        if (tk == 0) {
          dac[c] = dav;
          gw[c] = gwv;
        }
      }
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        const float* c = kc + kb * 4 * KB + tk * 4;
        float dvl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            const float hval = t[kb][i][cc];
            dvl[cc] = fmaf(da[i], hval, dvl[cc]);
            DTs[(kb * KB + tk * 4 + cc) * TCP + tj * 8 + i] = (hval > 0.f) ? da[i] * c[KB + cc] * dinv : 0.f;
          }
        }
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) dvp[tj * HP + kb * KB + tk * 4 + cc] = dvl[cc];
      }
      __syncthreads();
      // ---- small reductions over cells: db1, dw2, lane columns (thread k), dist layer (thread cell) -------------
      if (tid < HP) {
        float sb = 0.f, s0 = 0.f, s1 = 0.f, sv = 0.f;
        for (int c = 0; c < TC; ++c) {
          const float dtv = DTs[tid * TCP + c];
          sb += dtv;
          if (lanes) {
            s0 = fmaf(dtv, g[c], s0);
            s1 = fmaf(dtv, g[TC + c], s1);
          }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) sv += dvp[j * HP + tid];
        pb += sb;
        pv += sv;
        pl0 += s0;
        pl1 += s1;
      } else if (tid >= TC && tid < 2 * TC) {
        const int c = tid - TC;
        if (lanes) {
          float dg0 = 0.f, dg1 = 0.f;
          for (int k = 0; k < hid; ++k) {
            const float dtv = DTs[k * TCP + c];
            const float* cst = kc + (k / KB) * 4 * KB + (k % KB);
            dg0 = fmaf(dtv, cst[2 * KB], dg0);
            dg1 = fmaf(dtv, cst[3 * KB], dg1);
          }
          const float g0 = g[c], g1 = g[TC + c];
          const float dz0 = dg0 * g0 * (1.f - g0), dz1 = dg1 * g1 * (1.f - g1);
          const float a0 = llc[c] * p.dist_scale, a1 = llc[TC + c] * p.dist_scale;
          pd[0] = fmaf(dz0, a0, pd[0]);
          pd[1] = fmaf(dz0, a1, pd[1]);
          pd[2] = fmaf(dz1, a0, pd[2]);
          pd[3] = fmaf(dz1, a1, pd[3]);
          pd[4] += dz0;
          pd[5] += dz1;
        } else if (p.dist_mode == NAIS_DIST_KM) {
          pd[6] = fmaf(dac[c], llc[c], pd[6]);
        }
      }
      // ---- GEMM3: dW[k][d] += sum_c dt[k][c] x[d][c] ---------------------------------------------------------------
      {
        const int k0 = tid & 15, dd0 = tid >> 4;
#pragma unroll
        for (int s = 0; s < NKB * DB; ++s) {
          const int kb3 = s / DB, db3 = s % DB;
          const float* ar[4];
          const float* brow[4];
          bool dok[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) ar[i] = DTs + (size_t)(kb3 * KB + k0 + 16 * i) * TCP;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int d = db3 * 64 + dd0 + 16 * j;
            dok[j] = d < D;
            brow[j] = As + (size_t)(dok[j] ? d : 0) * TCP;
          }
          for (int c = 0; c < TC; c += 4) {
            float4 av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = *reinterpret_cast<const float4*>(ar[i] + c);
#pragma unroll
            for (int j = 0; j < 4; ++j) bv[j] = *reinterpret_cast<const float4*>(brow[j] + c);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float v = acc3[s][i][j];
                v = fmaf(av[i].x, bv[j].x, v);
                v = fmaf(av[i].y, bv[j].y, v);
                v = fmaf(av[i].z, bv[j].z, v);
                v = fmaf(av[i].w, bv[j].w, v);
                acc3[s][i][j] = v;
              }
          }
        }
      }
      __syncthreads();  // As (x) no longer needed: it becomes the dp-contribution scratch
      // ---- GEMM2: dX[cell][d] = sum_k dt[cell][k] W[k][d]; finalize dq (global) and dp contributions (smem) ------
#pragma unroll 1
      for (int db = 0; db < DB; ++db) {
        const int d0 = db * 64 + tk * 4;
        const bool dact = d0 < D;
        float dx[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) dx[i][c] = 0.f;
        if (dact) {
          const float* ap = DTs + tj * 8;
          const float* wp = br.w1 + d0;
#pragma unroll 2
          for (int k = 0; k < hid; ++k) {
            float4 a0 = *reinterpret_cast<const float4*>(ap + k * TCP);
            float4 a1 = *reinterpret_cast<const float4*>(ap + k * TCP + 4);
            const float* wr = wp + (size_t)k * ldw;
            float bv[4];
            if (w1_vec2) {  // two 64-bit loads instead of four 32-bit ones (this loop issues most of the kernel's L1 requests)
              const float2 w01 = __ldg(reinterpret_cast<const float2*>(wr)), w23 = __ldg(reinterpret_cast<const float2*>(wr + 2));
              bv[0] = w01.x, bv[1] = w01.y, bv[2] = w23.x, bv[3] = w23.y;
            } else {
              bv[0] = __ldg(wr), bv[1] = __ldg(wr + 1), bv[2] = __ldg(wr + 2), bv[3] = __ldg(wr + 3);
            }
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int c = 0; c < 4; ++c) dx[i][c] = fmaf(av[i], bv[c], dx[i][c]);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int c = tj * 8 + i;
            const int rr = crow[c];
            float o[4] = {0.f, 0.f, 0.f, 0.f}, dpv[4] = {0.f, 0.f, 0.f, 0.f};
            if (rr >= 0) {
              const float gwv = gw[c];
              const int it = citem[c], rg = creg[c];
              float qv[4];
              if (vec4) {
                const float4 q4 = ldg_row4(br.hist_poi + (size_t)it * br.w_poi, br.hist_reg + (size_t)rg * br.w_reg, br.w_poi, d0);
                qv[0] = q4.x, qv[1] = q4.y, qv[2] = q4.z, qv[3] = q4.w;
              } else {
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                  const int d = d0 + cc;
                  qv[cc] = (d < br.w_poi) ? __ldg(br.hist_poi + (size_t)it * br.w_poi + d)
                                          : __ldg(br.hist_reg + (size_t)rg * br.w_reg + (d - br.w_poi));
                }
              }
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) {
                const int d = d0 + cc;
                const float full = dx[i][cc] + gwv;
                o[cc] = full * ps[rr * D + d];
                dpv[cc] = full * qv[cc];
              }
              if (A.ws_dq) *reinterpret_cast<float4*>(A.ws_dq + cgl[c] * D + d0) = make_float4(o[0], o[1], o[2], o[3]);
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) As[(size_t)(d0 + cc) * TCP + c] = dpv[cc];
          }
        }
      }
      __syncthreads();
      // ---- dp[row][d] += sum over the row's cells -----------------------------------------------------------------
      {
        const int nr = (H <= TC) ? nrows : 1;
        for (int i = tid; i < nr * D; i += NT) {
          const int rr = i / D, d = i - rr * D;
          const int c0 = (H <= TC) ? rr * H : 0;
          const int cn = (H <= TC) ? H : min(TC, H - ch * TC);
          float sacc = 0.f;
          for (int c = 0; c < cn; ++c) sacc += As[(size_t)d * TCP + c0 + c];
          dpacc[rr * D + d] += sacc;
        }
      }
    }
    __syncthreads();
    if (A.ws_dp)
      for (int i = tid; i < nrows * D; i += NT) A.ws_dp[(row0 + i / D) * D + (i % D)] = dpacc[i];
  }

  // ---- flush this CTA's parameter partials --------------------------------------------------------------------------
  float* part = A.ws_part + (size_t)blockIdx.x * A.part_stride;
  {
    const int k0 = tid & 15, dd0 = tid >> 4;
#pragma unroll
    for (int s = 0; s < NKB * DB; ++s) {
      const int kb3 = s / DB, db3 = s % DB;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = kb3 * KB + k0 + 16 * i, d = db3 * 64 + dd0 + 16 * j;
          if (k < hid && d < D) part[(size_t)k * ldw + d] = acc3[s][i][j];
        }
    }
  }
  if (tid < HP && tid < hid) {
    if (lanes) {
      part[(size_t)tid * ldw + D] = pl0;
      part[(size_t)tid * ldw + D + 1] = pl1;
    }
    part[hid * ldw + tid] = pb;
    part[hid * ldw + hid + tid] = pv;
  }
  // dist-layer partials: block reduce of pd[] held by threads TC..2TC-1
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    float v = pd[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) red[q * (NT / 32) + (tid >> 5)] = v;
  }
  __syncthreads();
  if (tid < 7) {
    float v = 0.f;
    for (int w = 0; w < NT / 32; ++w) v += red[tid * (NT / 32) + w];
    part[hid * ldw + 2 * hid + tid] = v;
  }
}

// out[i] = sum over CTAs of part[cta][i], then scatter into the gradient tensors.
__global__ void param_reduce_kernel(const float* __restrict__ parts, int n_parts, int stride, int hid, int D, int lanes,
                                    float* w1, float* b1, float* w2, float* dist_w, float* dist_b, float* dist_embed,
                                    int dist_D, int accumulate_dist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int ldw = D + lanes, n = hid * ldw + 2 * hid + 7;
  if (i >= n) return;
  float s = 0.f;
  for (int c = 0; c < n_parts; ++c) s += parts[(size_t)c * stride + i];
  if (i < hid * ldw) {
    if (w1) w1[i] = s;
  } else if (i < hid * ldw + hid) {
    if (b1) b1[i - hid * ldw] = s;
  } else if (i < hid * ldw + 2 * hid) {
    if (w2) w2[i - hid * ldw - hid] = s;
  } else {
    const int q = i - hid * ldw - 2 * hid;
    if (q < 4) {
      if (dist_w) dist_w[q] = s;
    } else if (q < 6) {
      if (dist_b) dist_b[q - 4] = s;
    } else if (dist_embed) {
      // d/d embed_distance[0, d] = sum_cells da * km for every d (model.py:497-501); both branches add up
      for (int d = 0; d < dist_D; ++d) dist_embed[d] = accumulate_dist ? dist_embed[d] + s : s;
    }
  }
}

// Keys of the three embedding-row reductions.  src encodes where a contribution row comes from: cell index (dq) or B*H + row (dp).
// An id outside its table gets the key `n_rows` (one past the last row): it sorts behind every real row and the segment
// reduce drops it, so no table / optimizer row is written for it (the kernels that read it raised the bad-index word).
__device__ __forceinline__ int key_of(int64_t id, int n_rows) { return (uint64_t)id < (uint64_t)n_rows ? (int)id : n_rows; }
__global__ void make_keys_kernel(NaisPairs b, int item_num, int region_num, int* k_hist, uint32_t* v_hist, int* k_tgt,
                                 uint32_t* v_tgt, int* k_reg, uint32_t* v_reg) {
  const int64_t n_cells = pairs_n_cells(b);
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n_cells) {
    int64_t hidx = i;  // dense: cell index == history index
    if (pairs_segmented(b)) {
      // cell i belongs to the segment s with seg_cell_offsets[s] <= i < seg_cell_offsets[s+1]; its history item is (i - base) % H_s
      int lo = 0, hi = b.n_seg;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(b.seg_cell_offsets + mid) <= i) lo = mid;
        else hi = mid;
      }
      const int64_t h0 = __ldg(b.seg_offsets + lo), H = __ldg(b.seg_offsets + lo + 1) - h0;
      hidx = h0 + (i - __ldg(b.seg_cell_offsets + lo)) % H;
    }
    if (k_hist) {
      k_hist[i] = key_of(b.hist[hidx], item_num);
      v_hist[i] = (uint32_t)i;
    }
    if (k_reg) {
      k_reg[i] = key_of(b.hreg[hidx], region_num);
      v_reg[i] = (uint32_t)i;
    }
  }
  if (i < b.B) {
    if (k_tgt) {
      k_tgt[i] = key_of(b.tgt[i], item_num);
      v_tgt[i] = (uint32_t)i;
    }
    if (k_reg) {
      k_reg[n_cells + i] = key_of(b.treg[i], region_num);
      v_reg[n_cells + i] = (uint32_t)(n_cells + i);
    }
  }
}

// Embedding-row gradients: out[key, 0:w] = sum of the contribution rows of every sorted entry with that key.  Entry i's row is
// rows + src[i] * stride (src == NULL: entry i's row is row i — nais_rows_adagrad's key-ordered lists).  Two deterministic
// passes, no atomics:
//   pass 1  one warp per chunk of SEG_CHUNK consecutive entries accumulates runs of equal keys in order; a run that lies
//           strictly inside its chunk is complete and is written to the table row directly, the (at most two) runs that touch
//           a chunk boundary go to partial slots [2*chunk] (first run) / [2*chunk+1] (last run) together with a flag saying
//           whether the run STARTS in this chunk;
//   pass 2  one warp per starting partial adds the following chunks' continuing first-run partials, in chunk order.
constexpr int SEG_CHUNK = 64;

// Where a finished row gradient goes: into the dense gradient table (param == nullptr), or straight into a row-sparse
// Adagrad step on the parameter row (run.py:225,254 with weight_decay = lr_decay = 0, where untouched rows do not move):
//   sum += g*g ; param -= lr * g / (sqrt(sum) + eps)          (torch.optim.Adagrad's update, one row, written once)
struct SegOut {
  float* out;
  float* param;
  float* sum;
  float lr, eps;
  const int32_t* remap;  // out row of table row `key` = remap[key] (row-compacted gradient buffers, NaisGrads::remap_*); NULL: key
};
__device__ __forceinline__ size_t seg_row_of(const SegOut& o, int key) { return (o.remap && !o.param) ? (size_t)__ldg(o.remap + key) : (size_t)key; }
__device__ __forceinline__ void seg_store(const SegOut& o, size_t idx, float g) {
  if (o.param) {
    const float s2 = fmaf(g, g, o.sum[idx]);
    o.sum[idx] = s2;
    o.param[idx] -= o.lr * g / (sqrtf(s2) + o.eps);
  } else {
    o.out[idx] = g;
  }
}

// Where the contribution rows of a reduction live: source s < n_cells is cell s's dq row, s >= n_cells is row (s - n_cells)'s
// dp row; `off` selects the table's column range inside the D-wide row.
struct SegRows {
  const float* dq;
  const float* dp;
  int64_t n_cells;
  int D, off;
};
__device__ __forceinline__ const float* seg_row_ptr(const SegRows& R, const uint32_t* __restrict__ src, int64_t i) {
  if (!src) return R.dq + (size_t)i * R.D + R.off;  // key-ordered list: entry i's row is row i
  const uint32_t s = src[i];
  return (s < R.n_cells ? R.dq + (size_t)s * R.D : R.dp + (size_t)(s - R.n_cells) * R.D) + R.off;
}

// Pass 1 reads the rows of its chunk (a chunk is SEG_CHUNK * w * 4 contiguous bytes).  r2 profile of the first version (one
// shuffle + compare + branch + four predicated loads / adds per entry): 50 warp instructions per entry, issue-bound at 1.8 TB/s.
// Now: the chunk's 64 keys sit two per lane, ONE pair of ballots marks where runs start, and each run is a branch-free
// accumulation of its rows (SEG_ILP loads in flight, added in entry order: same sums, bit for bit) — ~4 instructions per entry.
// NQ = ceil(w / 32) floats per lane (w <= 128).
constexpr int SEG_ILP = 8;
template <int NQ, bool kOpt, int ILP>
__global__ void segment_reduce_pass1_kernel(const int* __restrict__ keys, const uint32_t* __restrict__ src, int64_t n, SegRows R, int w,
                                            int n_rows, SegOut out, int* __restrict__ part_key, int* __restrict__ part_start,
                                            float* __restrict__ part_rows) {
  const int64_t chunk = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t start = chunk * SEG_CHUNK;
  if (start >= n) return;
  const int64_t end = min(n, start + SEG_CHUNK);
  const int cnt = (int)(end - start);
  if (lane < 2) part_key[2 * chunk + lane] = -1;
  const int k0 = lane < cnt ? keys[start + lane] : -1, k1 = 32 + lane < cnt ? keys[start + 32 + lane] : -1;
  // where this lane's two entries' rows live (handed around by shuffles below)
  const float* r0p = lane < cnt ? seg_row_ptr(R, src, start + lane) : nullptr;
  const float* r1p = 32 + lane < cnt ? seg_row_ptr(R, src, start + 32 + lane) : nullptr;
  const int key_before = start > 0 ? keys[start - 1] : -1, key_after = end < n ? keys[end] : -1;
  // bit j of `starts` = entry j begins a run (entry 0 always does)
  const int p0 = __shfl_up_sync(0xffffffffu, k0, 1), last0 = __shfl_sync(0xffffffffu, k0, 31), p1 = __shfl_up_sync(0xffffffffu, k1, 1);
  const unsigned m0 = __ballot_sync(0xffffffffu, lane < cnt && (lane == 0 || k0 != p0));
  const unsigned m1 = __ballot_sync(0xffffffffu, 32 + lane < cnt && k1 != (lane == 0 ? last0 : p1));
  const unsigned long long starts = (unsigned long long)m0 | ((unsigned long long)m1 << 32);
  bool col[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) col[q] = lane + 32 * q < w;
  float acc[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) acc[q] = 0.f;
  int key = __shfl_sync(0xffffffffu, k0, 0), run_a = 0;  // the open run: its key and first entry
  auto flush = [&](int b) {                               // the open run ends before entry b
    if ((unsigned)key >= (unsigned)n_rows) return;        // ids outside [0, n_rows) (make_keys_kernel's n_rows) are dropped
    const bool left = run_a == 0 && key == key_before, right = b == cnt && key == key_after;
    if (!left && !right) {
#pragma unroll
      for (int q = 0; q < NQ; ++q)
        if (col[q]) seg_store(out, seg_row_of(out, key) * w + lane + 32 * q, acc[q]);
    } else {
      const int64_t slot = 2 * chunk + (run_a == 0 ? 0 : 1);
      if (lane == 0) {
        part_key[slot] = key;
        part_start[slot] = left ? 0 : 1;
      }
#pragma unroll
      for (int q = 0; q < NQ; ++q)
        if (col[q]) part_rows[(size_t)slot * w + lane + 32 * q] = acc[q];
    }
  };
  // rows are fetched ILP entries at a time whatever the run structure is (unique keys = runs of one entry must not turn
  // into a chain of dependent load -> store round trips); the run bookkeeping is a bit test per entry
  for (int j0 = 0; j0 < cnt; j0 += ILP) {
    float r[ILP][NQ];
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      const int j = j0 + u;  // (j0 is a multiple of ILP, which divides 32: a batch never straddles the two key registers)
      const unsigned long long pj = __shfl_sync(0xffffffffu, (unsigned long long)(j0 < 32 ? r0p : r1p), j & 31);
      const float* row = reinterpret_cast<const float*>(pj);
#pragma unroll
      for (int q = 0; q < NQ; ++q) r[u][q] = (j < cnt && col[q]) ? __ldcs(row + lane + 32 * q) : 0.f;
    }
    // Fused Adagrad: a finished run's update reads its `sum` and `param` rows before it writes them, so a flush per run is a
    // chain of dependent load -> store round trips (ncu launch list of one-user steps: 85 us for ONE 64-entry chunk of unique
    // keys, the target list — the longest kernel of the step).  The runs that end inside this batch are collected (keys are
    // warp-uniform) and updated together after it: all their loads first, then the same arithmetic, then the stores.
    int fkey[ILP];
    float facc[ILP][NQ];
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      const int j = j0 + u;
      fkey[u] = -1;
      if (j < cnt) {
        if (j > 0 && ((starts >> j) & 1ull)) {
          if (kOpt && (unsigned)key < (unsigned)n_rows && !(run_a == 0 && key == key_before)) {
            fkey[u] = key;
#pragma unroll
            for (int q = 0; q < NQ; ++q) facc[u][q] = acc[q];
          } else {
            flush(j);
          }
          run_a = j;
          key = j < 32 ? __shfl_sync(0xffffffffu, k0, j) : __shfl_sync(0xffffffffu, k1, j - 32);
#pragma unroll
          for (int q = 0; q < NQ; ++q) acc[q] = 0.f;
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) acc[q] += r[u][q];
      }
    }
    if constexpr (kOpt) {
      float fs[ILP][NQ], fp[ILP][NQ];
#pragma unroll
      for (int u = 0; u < ILP; ++u)
        if (fkey[u] >= 0) {
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            if (col[q]) {
              const size_t idx = (size_t)fkey[u] * w + lane + 32 * q;
              fs[u][q] = out.sum[idx];
              fp[u][q] = out.param[idx];
            }
        }
#pragma unroll
      for (int u = 0; u < ILP; ++u)
        if (fkey[u] >= 0) {
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            if (col[q]) {  // (seg_store's arithmetic)
              const size_t idx = (size_t)fkey[u] * w + lane + 32 * q;
              const float g = facc[u][q];
              const float s2 = fmaf(g, g, fs[u][q]);
              out.sum[idx] = s2;
              out.param[idx] = fp[u][q] - out.lr * g / (sqrtf(s2) + out.eps);
            }
        }
    }
  }
  flush(cnt);
}

// Pass 2: one warp per partial that STARTS a run; the chunks that continue it are found 32 at a time (one ballot, no chain of
// dependent loads: a hot row spanning hundreds of chunks used to be one warp walking them one by one) and their partial rows
// are added in chunk order.
template <int NQ>
__global__ void segment_reduce_pass2_kernel(const int* __restrict__ part_key, const int* __restrict__ part_start,
                                            const float* __restrict__ part_rows, int64_t n_chunks, int w, SegOut out) {
  const int64_t slot = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (slot >= 2 * n_chunks) return;
  const int key = part_key[slot];
  if (key < 0 || !part_start[slot]) return;
  bool col[NQ];
  float acc[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    col[q] = lane + 32 * q < w;
    acc[q] = col[q] ? part_rows[(size_t)slot * w + lane + 32 * q] : 0.f;
  }
  for (int64_t c0 = (slot >> 1) + 1; c0 < n_chunks; c0 += 32) {
    const int64_t c = c0 + lane;
    const bool cont = c < n_chunks && part_key[2 * c] == key && !part_start[2 * c];
    const unsigned m = __ballot_sync(0xffffffffu, cont);
    const int len = (m == 0xffffffffu) ? 32 : __ffs((int)~m) - 1;  // contiguous prefix of continuing chunks
    for (int j0 = 0; j0 < len; j0 += SEG_ILP) {
      float r[SEG_ILP][NQ];
#pragma unroll
      for (int u = 0; u < SEG_ILP; ++u)
#pragma unroll
        for (int q = 0; q < NQ; ++q) r[u][q] = (j0 + u < len && col[q]) ? part_rows[(size_t)(2 * (c0 + j0 + u)) * w + lane + 32 * q] : 0.f;
#pragma unroll
      for (int u = 0; u < SEG_ILP; ++u)
        if (j0 + u < len) {
#pragma unroll
          for (int q = 0; q < NQ; ++q) acc[q] += r[u][q];
        }
    }
    if (len < 32) break;
  }
#pragma unroll
  for (int q = 0; q < NQ; ++q)
    if (col[q]) seg_store(out, seg_row_of(out, key) * w + lane + 32 * q, acc[q]);
}

// Both passes over n key-ordered rows (keys ascending, rows[i] belongs to keys[i]).  pk / pst / pr: partial slots for
// 2 * ceil(n / SEG_CHUNK) boundary runs (keys, start flags, rows of width w).
static void launch_segment_reduce(const int* keys, const uint32_t* src, int64_t n, const SegRows& rows, int w, int n_rows, const SegOut& out,
                                  int* pk, int* pst, float* pr, cudaStream_t stream) {
  const int64_t nch = (n + SEG_CHUNK - 1) / SEG_CHUNK;
  const unsigned g1 = (unsigned)((nch * 32 + 255) / 256), g2 = (unsigned)((2 * nch * 32 + 255) / 256);
  // kOpt: the fused-Adagrad kernel with the batched row updates, for SMALL lists (the one-user steps: a few chunks, latency-bound;
  // narrow rows then also keep 16 rows in flight per warp).  Large lists hide a warp's load -> store chains behind the other
  // warps and are faster with the leaner kernel (88 vs 56 registers; measured on a C3-sized fused step: 0.86 vs 0.76 ms).
  const bool defer = out.param != nullptr && n <= 65536;
  if (w <= 32) {
    if (defer) segment_reduce_pass1_kernel<1, true, 2 * SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    else segment_reduce_pass1_kernel<1, false, SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    segment_reduce_pass2_kernel<1><<<g2, 256, 0, stream>>>(pk, pst, pr, nch, w, out);
  } else if (w <= 64) {
    if (defer) segment_reduce_pass1_kernel<2, true, SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    else segment_reduce_pass1_kernel<2, false, SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    segment_reduce_pass2_kernel<2><<<g2, 256, 0, stream>>>(pk, pst, pr, nch, w, out);
  } else {
    if (defer) segment_reduce_pass1_kernel<4, true, SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    else segment_reduce_pass1_kernel<4, false, SEG_ILP><<<g1, 256, 0, stream>>>(keys, src, n, rows, w, n_rows, out, pk, pst, pr);
    segment_reduce_pass2_kernel<4><<<g2, 256, 0, stream>>>(pk, pst, pr, nch, w, out);
  }
  NAIS_COUNT_LAUNCH(2);
}

// nais_pairs_train_step (include/nais_b200.h): sigmoid + BCELoss forward and backward on the [B] scores, one CTA, a fixed
// reduction tree (deterministic loss).  x = 1 / (1 + exp(-s)); loss_b = -(y * max(log x, -100) + (1 - y) * max(log(1 - x), -100));
// dL/ds = w * (x - y) / max((1 - x) * x, 1e-12) * ((1 - x) * x)   — torch's binary_cross_entropy_backward x sigmoid_backward.
__global__ void __launch_bounds__(1024, 1) bce_dscore_kernel(const float* __restrict__ score, const float* __restrict__ label,
                                                              const float* __restrict__ row_weight, int64_t B, float* __restrict__ dscore,
                                                              float* __restrict__ loss) {
  __shared__ float red[32];
  const float wmean = 1.f / (float)B;
  float acc = 0.f;
  for (int64_t b = threadIdx.x; b < B; b += blockDim.x) {
    const float s = score[b], y = label[b], w = row_weight ? row_weight[b] : wmean;
    const float x = 1.f / (1.f + expf(-s));
    const float l = -(y * fmaxf(logf(x), -100.f) + (1.f - y) * fmaxf(logf(1.f - x), -100.f));
    acc = fmaf(w, l, acc);
    const float v = (1.f - x) * x;
    dscore[b] = (w * (x - y) / fmaxf(v, 1e-12f)) * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (threadIdx.x == 0) *loss = v;
  }
}
int launch_bce_dscore(const float* score, const float* label, const float* row_weight, int64_t B, float* dscore, float* loss,
                      cudaStream_t stream) {
  bce_dscore_kernel<<<1, 1024, 0, stream>>>(score, label, row_weight, B, dscore, loss);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// nais_pairs_train_step_bpr (include/nais_b200.h): the BPR loss -log sigmoid(s+ - s-) on rows in groups of G = 1 + num_neg
// (positive first), one CTA, the fixed reduction tree of bce_dscore_kernel (deterministic loss).  d = s[gG] - s[gG + j];
// loss = sum_g w_g sum_j softplus(-d) with softplus(-d) = max(-d, 0) + log1p(exp(-|d|)) (finite for any |d|); its derivative
// sigma(-d) in the form of torch's log_sigmoid backward: z = exp(-|d|), z / (1 + z) for d >= 0, 1 - z / (1 + z) for d < 0.
// dscore[negative j] = w_g sigma(-d_j); dscore[positive] = -sum_j w_g sigma(-d_j), summed over j ascending.
__global__ void __launch_bounds__(1024, 1) bpr_dscore_kernel(const float* __restrict__ score, const float* __restrict__ group_weight,
                                                              int64_t n_groups, int num_neg, float* __restrict__ dscore,
                                                              float* __restrict__ loss) {
  __shared__ float red[32];
  const int G = num_neg + 1;
  const float wmean = 1.f / (float)(n_groups * num_neg);
  float acc = 0.f;
  for (int64_t g = threadIdx.x; g < n_groups; g += blockDim.x) {
    const float* s = score + g * G;
    float* ds = dscore + g * G;
    const float sp = s[0], w = group_weight ? group_weight[g] : wmean;
    float dpos = 0.f;
    for (int j = 1; j < G; ++j) {
      const float d = sp - s[j];
      const float z = expf(-fabsf(d));
      acc = fmaf(w, fmaxf(-d, 0.f) + log1pf(z), acc);
      const float q = z / (1.f + z);
      const float gj = w * (d >= 0.f ? q : 1.f - q);
      ds[j] = gj;
      dpos -= gj;
    }
    ds[0] = dpos;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (threadIdx.x == 0) *loss = v;
  }
}
int launch_bpr_dscore(const float* score, const float* group_weight, int64_t B, int num_neg, float* dscore, float* loss,
                      cudaStream_t stream) {
  bpr_dscore_kernel<<<1, 1024, 0, stream>>>(score, group_weight, B / (num_neg + 1), num_neg, dscore, loss);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// dense Adagrad of up to 5 small tensors in one launch (torch.optim.Adagrad, weight_decay = lr_decay = 0)
struct DenseAdagradArgs {
  float* param[5];
  float* sum[5];
  const float* grad[5];
  int n[5];
  float lr, eps;
};
__global__ void dense_adagrad_kernel(const DenseAdagradArgs A) {
  const int t = blockIdx.y;
  if (!A.param[t]) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n[t]; i += gridDim.x * blockDim.x) {
    const float g = A.grad[t][i];
    const float s2 = fmaf(g, g, A.sum[t][i]);
    A.sum[t][i] = s2;
    A.param[t][i] += -A.lr * (g / (sqrtf(s2) + A.eps));
  }
}
int launch_dense_adagrad(float* const* param, float* const* sum, const float* const* grad, const int* n, float lr, float eps,
                         cudaStream_t stream) {
  DenseAdagradArgs A;
  int nmax = 1;
  for (int t = 0; t < 5; ++t) {
    const bool on = param[t] && sum[t] && grad[t] && n[t] > 0;
    A.param[t] = on ? param[t] : nullptr;
    A.sum[t] = sum[t];
    A.grad[t] = grad[t];
    A.n[t] = n[t];
    if (on && n[t] > nmax) nmax = n[t];
  }
  A.lr = lr;
  A.eps = eps;
  dim3 grid((nmax + 255) / 256 < 64 ? (nmax + 255) / 256 : 64, 5);
  dense_adagrad_kernel<<<grid, 256, 0, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// nais_rows_adagrad (include/nais_b200.h): key-ordered (id, gradient row) lists -> one row-sparse Adagrad step per distinct id
size_t rows_adagrad_workspace_bytes(int64_t n, int w) {
  const int64_t nch = (n + SEG_CHUNK - 1) / SEG_CHUNK;
  return 2 * ((size_t)2 * nch * 4 + 256) + (size_t)2 * nch * w * 4 + 256;
}
int launch_rows_adagrad(const int32_t* keys, const float* rows, int64_t n, int w, int n_rows, float* grad_out, float* param, float* sum,
                        float lr, float eps, void* ws, size_t ws_bytes, cudaStream_t stream) {
  if (n == 0) return 0;
  if (ws_bytes < rows_adagrad_workspace_bytes(n, w)) return NAIS_ERR_WORKSPACE;
  const int64_t nch = (n + SEG_CHUNK - 1) / SEG_CHUNK;
  char* base = reinterpret_cast<char*>(ws);
  const size_t kb = ((size_t)2 * nch * 4 + 255) / 256 * 256;
  SegOut o;
  o.out = grad_out;
  o.param = sum ? param : nullptr;
  o.sum = sum;
  o.lr = lr;
  o.eps = eps;
  o.remap = nullptr;
  SegRows R;
  R.dq = rows;
  R.dp = nullptr;
  R.n_cells = n;
  R.D = w;
  R.off = 0;
  launch_segment_reduce(keys, nullptr, n, R, w, n_rows, o, reinterpret_cast<int*>(base), reinterpret_cast<int*>(base + kb),
                        reinterpret_cast<float*>(base + 2 * kb), stream);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

static int bwd_grid() { return 148 * 2; }

// lists: 0 = history ids (B*H entries), 1 = target ids (B), 2 = region ids of both (B*H + B)
static BwdLayout bwd_layout(const NaisParams& p, const NaisPairs& b) {
  const int64_t B = b.B;
  BwdLayout L;
  int D = 0, w_poi = 0, w_reg = 0;
  for (int i = 0; i < p.n_branch; ++i) {
    const NaisBranch& br = p.branch[i];
    D = D > br.w_poi + br.w_reg ? D : br.w_poi + br.w_reg;
    w_poi = w_poi > br.w_poi ? w_poi : br.w_poi;
    w_reg = w_reg > br.w_reg ? w_reg : br.w_reg;
  }
  const int lanes = p.dist_mode == NAIS_DIST_LATLON ? 2 : 0;
  const int64_t n_cells = pairs_n_cells(b), n_max = n_cells + B;
  const int64_t n_of[3] = {n_cells, B, n_max};
  size_t o = 0;
  L.dq = o;
  o += align_up((size_t)n_cells * D * 4);
  L.dp = o;
  o += align_up((size_t)B * D * 4);
  L.grid = bwd_grid();
  L.stride = part_floats(p.hid, D, lanes);
  L.part = o;
  o += align_up((size_t)L.grid * L.stride * 4);
  for (int i = 0; i < 3; ++i) {
    const size_t bytes = align_up((size_t)n_of[i] * 4);
    L.kin[i] = o, o += bytes;
    L.vin[i] = o, o += bytes;
    L.kout[i] = o, o += bytes;
    L.vout[i] = o, o += bytes;
  }
  size_t cb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cb, (const int*)nullptr, (int*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, (int)(n_max > 0x7fffffff ? 0x7fffffff : n_max));
  L.cub_bytes = cb;
  const int wmax = w_poi > w_reg ? w_poi : w_reg;
  for (int i = 0; i < 3; ++i) {  // the three lists are sorted and reduced concurrently (side streams): private scratch each
    const int64_t nch = (n_of[i] + SEG_CHUNK - 1) / SEG_CHUNK;
    L.cub[i] = o;
    o += align_up(cb);
    L.pkey[i] = o;
    o += align_up((size_t)2 * nch * 4);
    L.pstart[i] = o;
    o += align_up((size_t)2 * nch * 4);
    L.prows[i] = o;
    o += align_up((size_t)2 * nch * wmax * 4);
  }
  L.total = o;
  return L;
}

size_t pairs_bwd_workspace_bytes(const NaisParams& p, const NaisPairs& b) { return bwd_layout(p, b).total; }

// The three id lists (history POIs, target POIs, regions) are independent until the gradient tables are written: their radix
// sorts and their segment reduces are latency-bound launches that underfill the GPU one at a time (ncu launch list,
// profiles/r2_launches_train_c3.csv: 29 us to sort 8 192 target ids, 27 us to reduce them), so lists 1 and 2 run on two side
// streams forked from / joined to the caller's stream with events.  One pool per device, created on first use; the mutex is
// held while a PairsBwd step ENQUEUES its work (cudaStreamWaitEvent binds to the record that precedes it at call time).  Every event
// a step waits for is recorded in that step, except `sorted0`, which `finish` waits for after an earlier `sort` released the mutex
// (one host thread per GPU, include/nais_b200.h).
struct SideStreams {
  cudaStream_t s[3] = {nullptr, nullptr, nullptr};  // [0], [1]: lists 1, 2; [2]: list 0's sort when PairsBwd::sort forks it, then param_reduce
  cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr}, sorted0 = nullptr, pjoin = nullptr;  // pjoin: param_reduce (+ dense Adagrad) on s[2]
  bool ok = false;
};
static std::mutex g_side_mu;
static SideStreams* side_streams() {
  static SideStreams pool[64];
  std::lock_guard<std::mutex> side_lock(g_side_mu);
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStreams& S = pool[dev];
  if (!S.ok) {
    bool good = cudaEventCreateWithFlags(&S.fork, cudaEventDisableTiming) == cudaSuccess &&
                cudaEventCreateWithFlags(&S.sorted0, cudaEventDisableTiming) == cudaSuccess &&
                cudaEventCreateWithFlags(&S.pjoin, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 3 && good; ++i) good = cudaStreamCreateWithFlags(&S.s[i], cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 2 && good; ++i) good = cudaEventCreateWithFlags(&S.join[i], cudaEventDisableTiming) == cudaSuccess;
    if (!good) return nullptr;
    S.ok = true;
  }
  return &S;
}

template <int NKB, int DB>
static int launch_bwd_tile(const BwdArgs& A, int D, int grid, cudaStream_t stream) {
  constexpr int HP = NKB * KB;
  const size_t fl = (size_t)D * TCP + (size_t)HP * TCP + (size_t)D * KB + NKB * 4 * KB + 8 * TC + 16 * HP +
                    2 * (size_t)BWD_MAXROWS * D + 4 * BWD_MAXROWS + 8 * (NT / 32);
  const size_t smem = fl * 4 + 3 * TC * 4 + TC * 8 + TC * 4 + 8;
  cudaError_t e = cudaFuncSetAttribute(pairs_bwd_kernel<NKB, DB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  pairs_bwd_kernel<NKB, DB><<<grid, NT, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

// `split` and the fused optimizer take pairs_fused_layout (disentangled: each id list belongs to one branch, so a row-sparse step
// per list IS the dense step); branch 0 sorts lists 0 / 1, branch 1 list 2.
int PairsBwd::open(const NaisParams& p_, const NaisPairs& b_, const NaisGrads& g_, const NaisAdagrad* opt_, const float* score_parts_,
                   const float* row_sum_, const unsigned long long* act_mask_, const float* dscore_, void* ws, size_t ws_bytes, bool split) {
  p = p_, b = b_, g = g_, opt = opt_, base = reinterpret_cast<char*>(ws);
  score_parts = score_parts_, row_sum = row_sum_, act_mask = act_mask_, dscore = dscore_;
  if (pairs_n_cells(b) + b.B >= 0x7fffffffLL) return NAIS_ERR_SHAPE;
  if ((split || opt) && !pairs_fused_layout(p)) return NAIS_ERR_MODE;
  L = bwd_layout(p, b);
  if (ws_bytes < L.total) return NAIS_ERR_WORKSPACE;
  side = side_streams();
  if (!side) return (int)cudaErrorUnknown;
  n_of[0] = pairs_n_cells(b), n_of[1] = b.B, n_of[2] = n_of[0] + b.B;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const NaisBranch& br = p.branch[bi];
    if (br.w_poi + br.w_reg > 128 || p.hid > 128) return NAIS_ERR_SHAPE;  // backward tiles: D, hid <= 128 in this version
    if (pairs_n_tiles(b) < 1) return 0;
    if (p.pairs_precision == NAIS_PAIRS_TC && !pairs_tc_bwd_supported(p, b)) return NAIS_ERR_SHAPE;
    // the tcgen05 dropout backward takes the mask from the forward's act_mask (it regenerates nothing); a call that only sorts
    // (no dscore) runs no tile kernel
    if (p.pairs_precision == NAIS_PAIRS_TC && p.dropout_p > 0.f && !act_mask && dscore) return NAIS_ERR_NULL;
    // a table is processed if it has a gradient destination or a fused-optimizer state
    want[bi][0] = br.w_poi > 0 && (g.hist_poi[bi] || (opt && opt->sum_hist_poi[bi]));
    want[bi][1] = br.w_poi > 0 && (g.tgt_poi[bi] || (opt && opt->sum_tgt_poi[bi]));
    want[bi][2] = br.w_reg > 0 && (g.reg[bi] || (opt && opt->sum_reg[bi]));
  }
  n_branch = p.n_branch;
  return 0;
}

// The ids do not depend on the gradients; stable radix sort: equal ids keep cell order.
void PairsBwd::sort(int bi, cudaStream_t stream, bool fork_long) const {
  const bool* w = want[bi];
  if (!w[0] && !w[1] && !w[2]) return;
  std::lock_guard<std::mutex> side_lock(g_side_mu);
  const int64_t n_thr = n_of[0] > b.B ? n_of[0] : b.B;
  make_keys_kernel<<<(unsigned)((n_thr + 255) / 256), 256, 0, stream>>>(b, p.item_num, p.region_num, w[0] ? I(L.kin[0]) : nullptr,
                                                                        U(L.vin[0]), w[1] ? I(L.kin[1]) : nullptr, U(L.vin[1]),
                                                                        w[2] ? I(L.kin[2]) : nullptr, U(L.vin[2]));
  NAIS_COUNT_LAUNCH(1);
  cudaEventRecord(side->fork, stream);
  for (int t = 2; t >= 0; --t) {  // (the caller's stream last: the side streams are busy while it sorts the long list)
    if (!w[t]) continue;
    cudaStream_t sort_stream = t ? side->s[t - 1] : (fork_long ? side->s[2] : stream);
    if (sort_stream != stream) cudaStreamWaitEvent(sort_stream, side->fork, 0);
    const int n_rows = t == 2 ? p.region_num : p.item_num;
    int bits = 1;  // keys are 0 .. n_rows (n_rows = the "drop" key of an out-of-range id)
    while ((1ll << bits) <= n_rows && bits < 31) ++bits;
    size_t cb = L.cub_bytes;
    cub::DeviceRadixSort::SortPairs(base + L.cub[t], cb, I(L.kin[t]), I(L.kout[t]), U(L.vin[t]), U(L.vout[t]), (int)n_of[t], 0, bits,
                                    sort_stream);
    if (fork_long && t == 0) cudaEventRecord(side->sorted0, side->s[2]);
  }
}

int PairsBwd::join_sorts(cudaStream_t stream) const {
  std::lock_guard<std::mutex> side_lock(g_side_mu);
  for (int bi = 0; bi < n_branch; ++bi)
    for (int t = 0; t < 3; ++t) {
      if (!want[bi][t]) continue;
      cudaEvent_t ev = t ? side->join[t - 1] : side->sorted0;
      cudaEventRecord(ev, t ? side->s[t - 1] : side->s[2]);
      cudaStreamWaitEvent(stream, ev, 0);
    }
  return (int)cudaGetLastError();
}

// `dense`: this branch's DenseAdagradLaunch (or NULL), enqueued behind its param_reduce — branch 1's holds embed_distance, whose
// gradient is complete only after branch 1's param_reduce (both branches read it).
int PairsBwd::finish(int bi, cudaStream_t stream, bool wait_sorted0, const DenseAdagradLaunch* dense) const {
  const bool* w = want[bi];
  const NaisBranch& br = p.branch[bi];
  const int D = br.w_poi + br.w_reg, lanes = p.dist_mode == NAIS_DIST_LATLON ? 2 : 0;
  std::lock_guard<std::mutex> side_lock(g_side_mu);
  // ---- the tile kernel ----------------------------------------------------------------------------------------------------
  BwdArgs A;
  A.p = p;
  A.b = b;
  A.bi = bi;
  A.parts = score_parts + (size_t)bi * b.B;
  A.row_sum = row_sum + (size_t)bi * b.B;
  A.dscore = dscore;
  A.act_mask = (p.hid <= 64 && act_mask) ? act_mask + (size_t)bi * n_of[0] : nullptr;  // [n_branch, cells]: this branch's pattern
  A.ws_dq = (w[0] || w[2]) ? reinterpret_cast<float*>(base + L.dq) : nullptr;
  A.ws_dp = (w[1] || w[2]) ? reinterpret_cast<float*>(base + L.dp) : nullptr;
  A.ws_part = reinterpret_cast<float*>(base + L.part);
  A.part_stride = L.stride;
  A.n_items = pairs_n_tiles(b);
  int grid = (int)(A.n_items < L.grid ? A.n_items : L.grid);
  int rc;
  const int nkb = p.hid <= 64 ? 1 : 2, db = D <= 64 ? 1 : 2;
  A.bad = bad_index_flag();
  A.drop_inv = p.dropout_p > 0.f ? 1.f / (1.f - p.dropout_p) : 1.f;
  const bool tc_ok = pairs_tc_bwd_supported(p, b) && (p.dropout_p <= 0.f || A.act_mask);  // (else the FP32 kernel regenerates the mask)
  if (p.pairs_precision != NAIS_PAIRS_FP32 && tc_ok) rc = launch_pairs_bwd_tc(A, D, grid, stream);  // tcgen05 (bf16 two-term splits)
  else if (nkb == 1 && db == 1) rc = launch_bwd_tile<1, 1>(A, D, grid, stream);
  else if (nkb == 1) rc = launch_bwd_tile<1, 2>(A, D, grid, stream);
  else if (db == 1) rc = launch_bwd_tile<2, 1>(A, D, grid, stream);
  else rc = launch_bwd_tile<2, 2>(A, D, grid, stream);
  auto join_lists = [&] {  // `stream` waits for the side streams of lists 1 / 2
    for (int t = 1; t < 3; ++t)
      if (w[t]) {
        cudaEventRecord(side->join[t - 1], side->s[t - 1]);
        cudaStreamWaitEvent(stream, side->join[t - 1], 0);
      }
  };
  if (rc) {  // (launch failure: rejoin the side streams before the caller may release the workspace)
    join_lists();
    return rc;
  }
  // ---- embedding rows: gather the contribution rows in key order --------------------------------------------------------------
  auto dest = [&](float* grad, const float* param, float* sum, const int32_t* remap) {
    SegOut o;
    o.out = grad;
    o.param = (opt && sum) ? const_cast<float*>(param) : nullptr;
    o.sum = sum;
    o.lr = opt ? opt->lr : 0.f;
    o.eps = opt ? opt->eps : 0.f;
    o.remap = remap;
    return o;
  };
  auto seg = [&](int t, int off, int width, int n_rows, SegOut out) {  // list t runs on: 0 -> the caller's stream, 1 / 2 -> side streams
    SegRows R;
    R.dq = t == 1 ? A.ws_dp : A.ws_dq;  // the target list's sources are plain row indices into dp
    R.dp = A.ws_dp;
    R.n_cells = t == 1 ? n_of[1] : n_of[0];
    R.D = D;
    R.off = off;
    launch_segment_reduce(I(L.kout[t]), U(L.vout[t]), n_of[t], R, width, n_rows, out, I(L.pkey[t]), I(L.pstart[t]),
                          reinterpret_cast<float*>(base + L.prows[t]), t == 0 ? stream : side->s[t - 1]);
  };
  // fork again: the side streams (still ordered after their own sorts) wait for the tile kernel, reduce their list, and join
  cudaEventRecord(side->fork, stream);
  for (int t = 1; t < 3; ++t)
    if (w[t]) cudaStreamWaitEvent(side->s[t - 1], side->fork, 0);
  // the per-CTA parameter partials -> w1 / b1 / w2 / distance-layer gradients (and the dense Adagrad step behind them) on the
  // third side stream, idle since the long list's sort: next to the three lists' reduces instead of in front of one of them
  cudaStream_t pstream = side->s[2];
  cudaStreamWaitEvent(pstream, side->fork, 0);
  const int n = p.hid * (D + lanes) + 2 * p.hid + 7;
  param_reduce_kernel<<<(n + 255) / 256, 256, 0, pstream>>>(
      A.ws_part, grid, L.stride, p.hid, D, lanes, g.w1[bi], g.b1[bi], g.w2[bi], bi == 0 ? g.dist_w : nullptr,
      bi == 0 ? g.dist_b : nullptr, p.dist_mode == NAIS_DIST_KM ? g.dist_embed : nullptr, D, bi > 0);
  NAIS_COUNT_LAUNCH(1);
  // the one-call training step's dense Adagrad of these tensors needs nothing else: right behind them, next to the table reduces
  const int dense_rc = dense ? launch_dense_adagrad(dense->param, dense->sum, dense->grad, dense->n, dense->lr, dense->eps, pstream) : 0;
  cudaEventRecord(side->pjoin, pstream);
  if (wait_sorted0 && w[0]) cudaStreamWaitEvent(stream, side->sorted0, 0);  // the long list was sorted on a side stream
  if (w[0]) seg(0, 0, br.w_poi, p.item_num, dest(g.hist_poi[bi], br.hist_poi, opt ? opt->sum_hist_poi[bi] : nullptr, g.remap_hist_poi[bi]));
  if (w[1]) seg(1, 0, br.w_poi, p.item_num, dest(g.tgt_poi[bi], br.tgt_poi, opt ? opt->sum_tgt_poi[bi] : nullptr, g.remap_tgt_poi[bi]));
  // (history-side and target-side region rows are one table in every variant: hist_reg == tgt_reg)
  if (w[2]) seg(2, br.w_poi, br.w_reg, p.region_num, dest(g.reg[bi], br.hist_reg, opt ? opt->sum_reg[bi] : nullptr, g.remap_reg[bi]));
  join_lists();
  cudaStreamWaitEvent(stream, side->pjoin, 0);
  cudaError_t e = cudaGetLastError();
  return e != cudaSuccess ? (int)e : dense_rc;
}

}  // namespace nais
