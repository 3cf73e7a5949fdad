// FP32 (CUDA-core FFMA) NAIS kernels: the numerically exact path.
//
//   tile_logits      shared tile-GEMM: for 128 cells, a_c = sum_k v_k relu(sum_d W[k,d] x_c[d] + b_k + wd.g_c)
//   pairs_fwd        explicit (history row, target) pairs      (model.py:246-297 and siblings)
//   fullrank_fp32    user x catalogue-range scoring + fused block top-k (validation.py:84-127)
//   topk_merge       merge of per-split / per-shard top-k lists
//
// The B x H x (D+2) pair tensor of the reference (model.py:266-269) only ever exists as one 128-cell tile in
// shared memory.
#include "nais_common.cuh"
#include "nais_pairs_tile.cuh"

namespace nais {

// ---------------------------------------------------------------------------------------------------------------------
// Shared-memory carve-up common to the tile kernels
// ---------------------------------------------------------------------------------------------------------------------
struct TileSmem {
  float* As;  // [D][TCP]  x = q (.) p per cell, d-major
  float* Wt;  // [D][KB]   attn_layer1.weight^T, current k-block (x part only)
  float* kc;  // [4][KB]   b1, w2, w1[:,D], w1[:,D+1] of the current k-block
  float* g;   // [2][TC]   distance lanes per cell (LATLON) / logit bias in g[0] (KM)
  float* sp;  // [2][TC]   similarity partial sums of the two d-halves
  float* a;   // [TC]      logits out
  long long* cg;  // [TC]  global cell index (pair*H + h) of each cell, for the dropout mask (pair kernels)
};
__host__ __device__ inline size_t tile_smem_floats(int D) { return (size_t)D * TCP + (size_t)D * KB + 4 * KB + 5 * TC + 2 * TC; }
__device__ inline float* carve_tile(float* base, int D, TileSmem& s) {
  s.As = base;
  base += (size_t)D * TCP;
  s.Wt = base;
  base += (size_t)D * KB;
  s.kc = base;
  base += 4 * KB;
  s.g = base;
  base += 2 * TC;
  s.sp = base;
  base += 2 * TC;
  s.a = base;
  base += TC;
  s.cg = reinterpret_cast<long long*>(base);  // 8-byte aligned: every preceding block is an even number of floats
  base += 2 * TC;
  return base;
}

// Load k-block kb of branch br: Wt[d][kk] = w1[kb*KB+kk][d], constants; zero padding beyond hid.
__device__ inline void load_wblock(const NaisBranch& br, int hid, int D, int lanes, int kb, const TileSmem& s) {
  const int ldw = D + lanes;
  for (int i = threadIdx.x; i < D * KB; i += blockDim.x) {
    const int d = i / KB, kk = i - d * KB;  // consecutive threads -> consecutive smem words (no bank conflicts)
    int k = kb * KB + kk;
    s.Wt[d * KB + kk] = (k < hid) ? __ldg(br.w1 + (size_t)k * ldw + d) : 0.f;
  }
  for (int kk = threadIdx.x; kk < KB; kk += blockDim.x) {
    int k = kb * KB + kk;
    bool ok = k < hid;
    s.kc[kk] = ok ? __ldg(br.b1 + k) : 0.f;
    s.kc[KB + kk] = ok ? __ldg(br.w2 + k) : 0.f;
    s.kc[2 * KB + kk] = (ok && lanes) ? __ldg(br.w1 + (size_t)k * ldw + D) : 0.f;
    s.kc[3 * KB + kk] = (ok && lanes) ? __ldg(br.w1 + (size_t)k * ldw + D + 1) : 0.f;
  }
}

struct DropCtx {
  uint32_t thresh;  // 0 = dropout off
  float inv_keep;
  uint64_t seed;
  int hid;
};

// One k-block of the tile GEMM + MLP epilogue.  Thread (tj = tid/16, tk = tid%16) owns cells tj*8..+7 and hidden
// units tk*4..+3 of the block; a_part[i] accumulates sum_k v_k relu(t_k) over this thread's hidden units.
__device__ __forceinline__ void tile_kblock(const TileSmem& s, int D, bool lanes, float (&a_part)[8], const DropCtx& dc, int kb) {
  const int tk = threadIdx.x & 15, tj = threadIdx.x >> 4;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[i][c] = 0.f;
  const float* ap = s.As + tj * 8;
  const float* bp = s.Wt + tk * 4;
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
      for (int c = 0; c < 4; ++c) acc[i][c] = fmaf(av[i], bv[c], acc[i][c]);
  }
  const float4 bb = *reinterpret_cast<const float4*>(s.kc + tk * 4);
  const float4 vv = *reinterpret_cast<const float4*>(s.kc + KB + tk * 4);
  const float4 w0 = *reinterpret_cast<const float4*>(s.kc + 2 * KB + tk * 4);
  const float4 w1 = *reinterpret_cast<const float4*>(s.kc + 3 * KB + tk * 4);
  const float bbv[4] = {bb.x, bb.y, bb.z, bb.w}, vvv[4] = {vv.x, vv.y, vv.z, vv.w};
  const float w0v[4] = {w0.x, w0.y, w0.z, w0.w}, w1v[4] = {w1.x, w1.y, w1.z, w1.w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float g0 = 0.f, g1 = 0.f;
    if (lanes) {
      g0 = s.g[tj * 8 + i];
      g1 = s.g[TC + tj * 8 + i];
    }
    float r = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float t = acc[i][c] + bbv[c];
      if (lanes) t = fmaf(w1v[c], g1, fmaf(w0v[c], g0, t));
      if (dc.thresh) {  // relu(drop(W x + b)), model.py:71,162
        const uint64_t idx = (uint64_t)s.cg[tj * 8 + i] * (uint64_t)dc.hid + (uint64_t)(kb * KB + tk * 4 + c);
        t = dropout_bits(dc.seed, idx) >= dc.thresh ? t * dc.inv_keep : 0.f;
      }
      r = fmaf(vvv[c], fmaxf(t, 0.f), r);
    }
    a_part[i] += r;
  }
}

// Whole MLP for the tile currently in s.As / s.g: writes s.a[cell].  `resident_kb` says which (branch,kb) block is
// already in s.Wt (updated).  All threads must call; ends with a __syncthreads().
__device__ inline void tile_logits(const NaisBranch& br, int br_idx, int hid, int D, int lanes, const TileSmem& s,
                                   int& resident, const DropCtx& dc) {
  const int n_kb = (hid + KB - 1) / KB;
  float a_part[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a_part[i] = 0.f;
  for (int kb = 0; kb < n_kb; ++kb) {
    const int want = br_idx * 1024 + kb;
    if (resident != want) {
      __syncthreads();  // previous users of Wt are done
      load_wblock(br, hid, D, lanes, kb, s);
      resident = want;
      __syncthreads();
    }
    tile_kblock(s, D, lanes != 0, a_part, dc, kb);
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
  if ((threadIdx.x & 15) == 0) {
    const int tj = threadIdx.x >> 4;
#pragma unroll
    for (int i = 0; i < 8; ++i) s.a[tj * 8 + i] = a_part[i];
  }
  __syncthreads();
}

__device__ __forceinline__ void dist_lanes(const NaisParams& p, float dlat, float dlon, float& g0, float& g1) {
  const float l0 = dlat * p.dist_scale, l1 = dlon * p.dist_scale;
  const float z0 = fmaf(l1, __ldg(p.dist_w + 1), fmaf(l0, __ldg(p.dist_w + 0), __ldg(p.dist_b + 0)));
  const float z1 = fmaf(l1, __ldg(p.dist_w + 3), fmaf(l0, __ldg(p.dist_w + 2), __ldg(p.dist_b + 1)));
  g0 = sigmoidf_exact(z0);
  g1 = sigmoidf_exact(z1);
}

__device__ __forceinline__ float km_coef(const NaisParams& p, int D, float km) {
  // sum_d embed_distance[bucket, d]   (model.py:497-501; the reference only has bucket 0)
  int b = 0;
  if (p.dist_buckets > 1) b = min((int)floorf(km / p.dist_bucket_km), p.dist_buckets - 1);
  float c = 0.f;
  for (int d = 0; d < D; ++d) c += __ldg(p.dist_embed + (size_t)b * D + d);
  return c;
}

// ---------------------------------------------------------------------------------------------------------------------
// Explicit pairs: forward
// ---------------------------------------------------------------------------------------------------------------------
struct PairsFwdArgs {
  NaisParams p;
  NaisPairs b;
  float* score;    // [B]
  float* row_sum;  // [n_branch,B] or NULL
  float* parts;    // [n_branch,B] per-branch score or NULL
  int* bad;        // the library's bad-index word (nais_common.cuh)
  float* cell_e;   // kCells: [n_branch, cells] masked exp E of every cell (nais_pairs_explain), indexed like act_mask
  float* cell_es;  // kCells: [n_branch, cells] E * similarity
};

constexpr int MAXROWS = PAIR_MAXROWS;  // rows (targets) sharing one 128-cell tile when H is small

// kCells: also store every cell's e and e * s (the per-history-item terms of the score) for nais_pairs_explain
template <bool kCells>
__global__ void __launch_bounds__(NT, 2) pairs_fwd_kernel(const __grid_constant__ PairsFwdArgs A) {
  extern __shared__ __align__(16) float smem[];
  const NaisParams& p = A.p;
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0;
  int Dmax = 0;
  for (int i = 0; i < p.n_branch; ++i) Dmax = max(Dmax, p.branch[i].w_poi + p.branch[i].w_reg);
  TileSmem s;
  float* rest = carve_tile(smem, Dmax, s);
  float* ps = rest;                        // [MAXROWS][Dmax] target vectors of the rows in this tile
  float* red_e = ps + MAXROWS * Dmax;      // [TC] masked exp per cell
  float* red_es = red_e + TC;              // [TC] masked exp * similarity
  float* row_e = red_es + TC;              // [MAXROWS] running sum E
  float* row_es = row_e + MAXROWS;         // [MAXROWS] running sum E*s
  __shared__ float km_c;

  const int tid = threadIdx.x, cell = tid & (TC - 1), half = tid >> 7;
  int resident = -1;
  DropCtx dc{0u, 1.f, p.dropout_seed, p.hid};
  if (p.dropout_p > 0.f) {
    dc.thresh = dropout_threshold(p.dropout_p);
    dc.inv_keep = 1.f / (1.f - p.dropout_p);
  }
  // persistent over work items (groups of rows): the W^T block stays resident in shared memory across items
  const int64_t n_items = pairs_n_tiles(A.b);
  for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
  const PairTile T = pair_tile(A.b, item);
  const int64_t row0 = T.row0;
  const int nrows = T.nrows, H = T.H;
  const int n_chunks = (H <= TC) ? 1 : (H + TC - 1) / TC;
  float my_total = 0.f;  // thread r (< nrows) accumulates the final score of row r over branches

  for (int bi = 0; bi < p.n_branch; ++bi) {
    const NaisBranch& br = p.branch[bi];
    const int D = br.w_poi + br.w_reg;
    const bool vec4 = rows_vec4(br, D >> 1) && (Dmax & 3) == 0;
    if (p.dist_mode == NAIS_DIST_KM && p.dist_buckets == 1) {
      if (tid == 0) km_c = km_coef(p, D, 0.f);
    }
    __syncthreads();
    // target vectors
    for (int i = tid; i < nrows * D; i += NT) {
      int r = i / D, d = i - r * D;
      ps[r * Dmax + d] = (d < br.w_poi) ? __ldg(br.tgt_poi + (size_t)checked_id(A.b.tgt[row0 + r], p.item_num, A.bad) * br.w_poi + d)
                                        : __ldg(br.tgt_reg + (size_t)checked_id(A.b.treg[row0 + r], p.region_num, A.bad) * br.w_reg + (d - br.w_poi));
    }
    if (tid < MAXROWS) {
      row_e[tid] = 0.f;
      row_es[tid] = 0.f;
    }
    __syncthreads();
    for (int ch = 0; ch < n_chunks; ++ch) {
      // cell -> (row, h)
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
      // build x = q (.) p for this thread's d-half, similarity partial, distance lanes
      {
        const int d0 = half ? (D >> 1) : 0, d1 = half ? D : (D >> 1);
        float ssum = 0.f;
        if (valid) {
          const int item = checked_id(A.b.hist[hidx], p.item_num, A.bad);
          const int reg = br.w_reg ? checked_id(A.b.hreg[hidx], p.region_num, A.bad) : 0;
          const float* qp = br.hist_poi + (size_t)item * br.w_poi;
          const float* qr = br.hist_reg + (size_t)reg * br.w_reg;
          if (vec4) {  // 128-bit row loads: 4x fewer L1 requests than the scalar walk, same products in the same order
            const float* pr = ps + r * Dmax;
#pragma unroll 4
            for (int d = d0; d < d1; d += 4) {
              const float4 q = ldg_row4(qp, qr, br.w_poi, d);
              const float4 t = *reinterpret_cast<const float4*>(pr + d);
              const float x0 = q.x * t.x, x1 = q.y * t.y, x2 = q.z * t.z, x3 = q.w * t.w;
              s.As[d * TCP + cell] = x0;
              s.As[(d + 1) * TCP + cell] = x1;
              s.As[(d + 2) * TCP + cell] = x2;
              s.As[(d + 3) * TCP + cell] = x3;
              ssum += x0;
              ssum += x1;
              ssum += x2;
              ssum += x3;
            }
          } else {
            for (int d = d0; d < d1; ++d) {
              float q = (d < br.w_poi) ? __ldg(qp + d) : __ldg(qr + d - br.w_poi);
              float x = q * ps[r * Dmax + d];
              s.As[d * TCP + cell] = x;
              ssum += x;
            }
          }
        } else {
          for (int d = d0; d < d1; ++d) s.As[d * TCP + cell] = 0.f;
        }
        s.sp[half * TC + cell] = ssum;
        if (half == 0) {
          s.cg[cell] = cidx;
          float g0 = 0.f, g1 = 0.f;
          if (valid && p.dist_mode == NAIS_DIST_LATLON) {
            float l0, l1;
            pair_latlon(A.b, cidx, hidx, row0 + r, l0, l1);
            dist_lanes(p, l0, l1, g0, g1);
          } else if (valid && p.dist_mode == NAIS_DIST_KM) {
            const float km = pair_km(A.b, cidx, hidx, row0 + r);
            g0 = km * (p.dist_buckets == 1 ? km_c : km_coef(p, D, km));
          }
          s.g[cell] = g0;
          s.g[TC + cell] = g1;
        }
      }
      __syncthreads();
      tile_logits(br, bi, p.hid, D, lanes, s, resident, dc);
      if (tid < TC) {
        float e = 0.f, es = 0.f;
        if (valid) {
          float a = s.a[cell];
          if (p.dist_mode == NAIS_DIST_KM) a += s.g[cell];
          const bool m = A.b.hist[hidx] != A.b.tgt[row0 + r];
          e = m ? expf(a) : 0.f;
          es = e * (s.sp[cell] + s.sp[TC + cell]);
          if (!m) es = 0.f;  // exp overflow * 0 must stay 0, like the reference's exp_A * mask then * history
        }
        red_e[cell] = e;
        red_es[cell] = es;
        if constexpr (kCells) {
          if (valid) {
            const size_t ci = (size_t)bi * pairs_n_cells(A.b) + cidx;
            A.cell_e[ci] = e;
            A.cell_es[ci] = es;
          }
        }
      }
      __syncthreads();
      // row reductions: warp w handles rows w, w+8, ...
      {
        const int w = tid >> 5, lane = tid & 31;
        for (int rr = w; rr < ((H <= TC) ? nrows : 1); rr += NT / 32) {
          const int c0 = (H <= TC) ? rr * H : 0;
          const int cn = (H <= TC) ? H : min(TC, H - ch * TC);
          float e = 0.f, es = 0.f;
          for (int c = lane; c < cn; c += 32) {
            e += red_e[c0 + c];
            es += red_es[c0 + c];
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            e += __shfl_xor_sync(0xffffffffu, e, o);
            es += __shfl_xor_sync(0xffffffffu, es, o);
          }
          if (lane == 0) {
            row_e[rr] += e;
            row_es[rr] += es;
          }
        }
      }
      __syncthreads();
    }
    if (tid < nrows) {
      const float S = row_e[tid];
      const float sc = row_es[tid] / powf(S, p.beta);
      my_total += sc;
      if (A.row_sum) A.row_sum[(size_t)bi * A.b.B + row0 + tid] = S;
      if (A.parts) A.parts[(size_t)bi * A.b.B + row0 + tid] = sc;
    }
    __syncthreads();
  }
  if (tid < nrows) A.score[row0 + tid] = my_total;
  __syncthreads();
  }  // items
}

// ---------------------------------------------------------------------------------------------------------------------
// Full-rank scoring + fused block top-k (FP32)
// ---------------------------------------------------------------------------------------------------------------------
struct FullrankArgs {
  NaisParams p;
  NaisCatalog cat;
  NaisUsers users;
  int64_t poi_begin, poi_end;
  int k;
  int exclude;
  int n_splits;
  unsigned long long* part_keys;  // [n_users, n_splits, k] (n_splits > 1)
  float* out_score;               // [n_users, k]           (n_splits == 1)
  int32_t* out_id;
  float* all_scores;  // optional [n_users, poi_end - poi_begin]
  int stage_p;        // 1: candidate vectors staged in smem (embed_size <= 128); 0: re-read from the tables (L1/L2) per history item
  int hc;             // history rows staged per chunk (HC, smaller when shared memory is tight)
  GeoMixArgs geo;     // kGeo: rank by the power-law mix (nais_fullrank_topk_geo_planned)
};

// kGeo: every cell also adds its power-law term ln a + b ln max(0.01, d_km) to log G (in history order, as
// nais_powerlaw_logscore), and the candidate is ranked by geo_mixed(score, log G, M_u) instead of its score.
template <bool kGeo>
__global__ void __launch_bounds__(NT, 2) fullrank_fp32_kernel(const __grid_constant__ FullrankArgs A) {
  extern __shared__ __align__(16) float smem[];
  const NaisParams& p = A.p;
  const int lanes = (p.dist_mode == NAIS_DIST_LATLON) ? 2 : 0;
  const bool km_mode = p.dist_mode == NAIS_DIST_KM, geo = lanes || km_mode;
  __shared__ float km_coef_s[64];  // sum_d embed_distance[bucket, d] (model.py:497-501)
  if (km_mode) {
    for (int b = threadIdx.x; b < min(p.dist_buckets, 64); b += blockDim.x) {
      float c = 0.f;
      const int Dk = p.branch[0].w_poi + p.branch[0].w_reg;
      for (int d = 0; d < Dk; ++d) c += __ldg(p.dist_embed + (size_t)b * Dk + d);
      km_coef_s[b] = c;
    }
  }
  int Dmax = 0;
  for (int i = 0; i < p.n_branch; ++i) Dmax = max(Dmax, p.branch[i].w_poi + p.branch[i].w_reg);
  TileSmem s;
  float* rest = carve_tile(smem, Dmax, s);
  const int HCr = A.hc;
  float* Ps = rest;                                 // [Dmax][TCP] candidate vectors, d-major (only if A.stage_p)
  float* Qs = Ps + (A.stage_p ? (size_t)Dmax * TCP : 0);  // [HCr][Dmax]  history vectors of the current chunk
  int* hid_s = reinterpret_cast<int*>(Qs + HCr * Dmax);  // [HCr] history item ids
  float* hco = reinterpret_cast<float*>(hid_s + HCr);    // [HCr][2] history coords
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(hco + 2 * HCr);  // [2*KCAP]

  const int u = blockIdx.x, split = blockIdx.y;
  const int64_t h_begin = A.users.offsets[u];
  const int H = (int)(A.users.offsets[u + 1] - h_begin);
  const int64_t range = A.poi_end - A.poi_begin;
  const int n_tiles = (int)((range + TC - 1) / TC);
  const int tid = threadIdx.x, cell = tid & (TC - 1), half = tid >> 7;
  int resident = -1;

  for (int i = tid; i < 2 * KCAP; i += NT) keys[i] = 0ull;
  __syncthreads();

  for (int tile = split; tile < n_tiles; tile += A.n_splits) {
    const int64_t j = A.poi_begin + (int64_t)tile * TC + cell;  // global POI id of this thread's cell
    const bool jvalid = j < A.poi_end;
    const int64_t jl = j - A.cat.row_base;
    float cla = 0.f, clo = 0.f, ccos = 1.f;
    if (jvalid && (geo || kGeo)) {
      cla = __ldg(A.cat.coords + jl * 2);
      clo = __ldg(A.cat.coords + jl * 2 + 1);
      if (km_mode || kGeo) ccos = cosf((A.cat.center_lat + cla) * 0.017453292519943295f);
    }
    float score = 0.f, logg = 0.f;
    bool excluded = false;
    for (int bi = 0; bi < p.n_branch; ++bi) {
      const NaisBranch& br = p.branch[bi];
      const int D = br.w_poi + br.w_reg;
      // candidate tile, d-major
      __syncthreads();
      const float* pp = jvalid ? br.tgt_poi + (size_t)j * br.w_poi : nullptr;
      const float* pr = (jvalid && br.w_reg) ? br.tgt_reg + (size_t)__ldg(A.cat.region + jl) * br.w_reg : nullptr;
      if (A.stage_p) {
        const int d0 = half ? (D >> 1) : 0, d1 = half ? D : (D >> 1);
        if (jvalid) {
          for (int d = d0; d < d1; ++d)
            Ps[d * TCP + cell] = (d < br.w_poi) ? __ldg(pp + d) : __ldg(pr + d - br.w_poi);
        } else {
          for (int d = d0; d < d1; ++d) Ps[d * TCP + cell] = 0.f;
        }
      }
      float sumE = 0.f, sumES = 0.f;
      for (int h0 = 0; h0 < H; h0 += HCr) {
        const int hn = min(HCr, H - h0);
        __syncthreads();
        for (int i = tid; i < hn * D; i += NT) {
          int hh = i / D, d = i - hh * D;
          const int64_t e = h_begin + h0 + hh;
          Qs[hh * Dmax + d] = (d < br.w_poi)
                                  ? __ldg(br.hist_poi + (size_t)__ldg(A.users.items + e) * br.w_poi + d)
                                  : __ldg(br.hist_reg + (size_t)__ldg(A.users.region + e) * br.w_reg + (d - br.w_poi));
        }
        if (tid < hn) {
          const int64_t e = h_begin + h0 + tid;
          hid_s[tid] = __ldg(A.users.items + e);
          if (geo || kGeo) {
            hco[2 * tid] = __ldg(A.users.coords + 2 * e);
            hco[2 * tid + 1] = __ldg(A.users.coords + 2 * e + 1);
          }
        }
        __syncthreads();
        for (int hh = 0; hh < hn; ++hh) {
          {
            const int d0 = half ? (D >> 1) : 0, d1 = half ? D : (D >> 1);
            const float* q = Qs + hh * Dmax;
            float ssum = 0.f;
            if (A.stage_p) {
              for (int d = d0; d < d1; ++d) {
                float x = Ps[d * TCP + cell] * q[d];
                s.As[d * TCP + cell] = x;
                ssum += x;
              }
            } else {  // embed_size > 128: no room for the candidate tile, re-read the table rows (L1/L2 resident)
              for (int d = d0; d < d1; ++d) {
                const float pv = !jvalid ? 0.f : ((d < br.w_poi) ? __ldg(pp + d) : __ldg(pr + d - br.w_poi));
                float x = pv * q[d];
                s.As[d * TCP + cell] = x;
                ssum += x;
              }
            }
            s.sp[half * TC + cell] = ssum;
            if (half == 0 && lanes) {
              float g0, g1;
              dist_lanes(p, fabsf(cla - hco[2 * hh]), fabsf(clo - hco[2 * hh + 1]), g0, g1);
              s.g[cell] = g0;
              s.g[TC + cell] = g1;
            }
          }
          __syncthreads();
          tile_logits(br, bi, p.hid, D, lanes, s, resident, DropCtx{0u, 1.f, 0ull, 0});
          if (tid < TC) {
            const bool m = (int64_t)hid_s[hh] != j;
            if constexpr (kGeo) {
              if (bi == 0) {  // every cell, the h = j one included; once per candidate, not per branch
                const float hla = hco[2 * hh], hlo = hco[2 * hh + 1];
                const float km = dist_km_f(cla, clo, hla, hlo, ccos, cosf((A.cat.center_lat + hla) * 0.017453292519943295f));
                logg += powerlaw_log_term(km, A.geo.ln_a, A.geo.b);
              }
            }
            if (m) {
              float a = s.a[cell];
              if (km_mode) {  // logit += dist_km * sum_d embed_distance[bucket] (haversine from centred coordinates)
                const float hla = hco[2 * hh], hlo = hco[2 * hh + 1];
                const float km = dist_km_f(cla, clo, hla, hlo, ccos, cosf((A.cat.center_lat + hla) * 0.017453292519943295f));
                int bkt = 0;
                if (p.dist_buckets > 1) bkt = min(min((int)floorf(km / p.dist_bucket_km), p.dist_buckets - 1), 63);
                a = fmaf(km, km_coef_s[bkt], a);
              }
              const float e = expf(a);
              sumE += e;
              sumES = fmaf(e, s.sp[cell] + s.sp[TC + cell], sumES);
            } else {
              excluded = true;
            }
          }
          // next iteration's As writes are ordered after this read of s.a/s.sp by the barrier inside tile_logits
          // of the NEXT call only for Wt; As/sp/g are rewritten immediately -> barrier here.
          __syncthreads();
        }
      }
      if (tid < TC) score += sumES / powf(sumE, p.beta);
    }
    if (tid < TC) {
      if constexpr (kGeo) score = geo_mixed(score, logg, __ldg(A.geo.user_logmax + u), A.geo.alpha);
      if (A.all_scores && jvalid) A.all_scores[(size_t)u * range + (j - A.poi_begin)] = score;
      const bool keep = jvalid && !(A.exclude && excluded);
      keys[KCAP + cell] = keep ? make_key(score, (int)j) : 0ull;
    }
    __syncthreads();
    bitonic_sort_desc(keys, 2 * KCAP);
  }
  // emit
  if (A.n_splits == 1) {
    for (int i = tid; i < A.k; i += NT) {
      float sc;
      int id;
      split_key(keys[i], sc, id);
      A.out_score[(size_t)u * A.k + i] = sc;
      A.out_id[(size_t)u * A.k + i] = id;
    }
  } else {
    for (int i = tid; i < A.k; i += NT) A.part_keys[((size_t)u * A.n_splits + split) * A.k + i] = keys[i];
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Top-k merge: n_lists lists of k per user -> k
// ---------------------------------------------------------------------------------------------------------------------
__global__ void topk_merge_kernel(const unsigned long long* in_keys, const float* in_score, const int32_t* in_id,
                                  int n_lists, int k, int n_pow2, float* out_score, int32_t* out_id) {
  extern __shared__ __align__(16) unsigned long long mkeys[];
  const int u = blockIdx.x, n = n_lists * k;
  for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
    unsigned long long key = 0ull;
    if (i < n) {
      if (in_keys) {
        key = in_keys[(size_t)u * n + i];
      } else {
        const int id = in_id[(size_t)u * n + i];
        if (id >= 0) key = make_key(in_score[(size_t)u * n + i], id);
      }
    }
    mkeys[i] = key;
  }
  __syncthreads();
  bitonic_sort_desc(mkeys, n_pow2);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    float sc;
    int id;
    split_key(mkeys[i], sc, id);
    out_score[(size_t)u * k + i] = sc;
    out_id[(size_t)u * k + i] = id;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Host launchers (called from nais_capi.cu)
// ---------------------------------------------------------------------------------------------------------------------
static int max_D(const NaisParams& p) {
  int D = 0;
  for (int i = 0; i < p.n_branch; ++i) D = D > p.branch[i].w_poi + p.branch[i].w_reg ? D : p.branch[i].w_poi + p.branch[i].w_reg;
  return D;
}

int launch_pairs_fwd(const NaisParams& p, const NaisPairs& b, float* score, float* row_sum, float* parts,
                     cudaStream_t stream, float* cell_e, float* cell_es) {
  if (b.B == 0) return 0;
  PairsFwdArgs A;
  A.p = p;
  A.b = b;
  A.score = score;
  A.row_sum = row_sum;
  A.parts = parts;
  A.bad = bad_index_flag();
  A.cell_e = cell_e;
  A.cell_es = cell_es;
  const bool cells = cell_e && cell_es;
  const int D = max_D(p);
  const size_t smem = (tile_smem_floats(D) + (size_t)MAXROWS * D + 2 * TC + 2 * MAXROWS) * sizeof(float);
  if (smem > 227 * 1024) return NAIS_ERR_SHAPE;
  cudaError_t e = cells ? cudaFuncSetAttribute(pairs_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                        : cudaFuncSetAttribute(pairs_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int64_t grid = pairs_n_tiles(b);
  if (grid < 1) return 0;
  if (grid > 148 * 4) grid = 148 * 4;
  if (cells) pairs_fwd_kernel<true><<<(unsigned)grid, NT, smem, stream>>>(A);
  else pairs_fwd_kernel<false><<<(unsigned)grid, NT, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

size_t fullrank_fp32_smem(const NaisParams& p, int& stage_p, int& hc) {
  const int D = max_D(p);
  stage_p = D <= 128;
  hc = D <= 128 ? HC : 8;
  return (tile_smem_floats(D) + (stage_p ? (size_t)D * TCP : 0) + (size_t)hc * D + 3 * hc) * sizeof(float) +
         2 * KCAP * sizeof(unsigned long long) + 16;
}

int choose_splits(int n_users, int64_t range) {
  const int n_tiles = (int)((range + TC - 1) / TC);
  int s = (148 * 2 * 4 + n_users - 1) / (n_users > 0 ? n_users : 1);
  if (s > 32) s = 32;
  if (s > n_tiles) s = n_tiles;
  if (s < 1) s = 1;
  return s;
}

int launch_topk_merge(const unsigned long long* in_keys, const float* in_score, const int32_t* in_id, int n_users,
                      int n_lists, int k, float* out_score, int32_t* out_id, cudaStream_t stream) {
  if (n_users == 0) return 0;
  int n = n_lists * k, n2 = 1;
  while (n2 < n) n2 <<= 1;
  if (n2 > 4096) return NAIS_ERR_SHAPE;
  const int threads = n2 >= 512 ? 512 : (n2 < 64 ? 64 : n2);
  topk_merge_kernel<<<n_users, threads, n2 * sizeof(unsigned long long), stream>>>(in_keys, in_score, in_id, n_lists, k, n2,
                                                                                  out_score, out_id);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}


// Keys -> keys (and / or final score, id) merge of blocks of `lpb` lists; grid (users, blocks): users on grid.x (no 65 535
// limit).  List l of user u starts at in + u * user_stride + l * list_stride (8-byte words).
__global__ void topk_merge_keys_kernel(const unsigned long long* __restrict__ in, long long user_stride, long long list_stride,
                                       int n_lists, int k, int lpb, int n2, unsigned long long* out_keys, int final_level,
                                       float* out_score, int32_t* out_id) {
  extern __shared__ __align__(16) unsigned long long mk[];
  const int u = blockIdx.x, b = blockIdx.y;
  const int l0 = b * lpb, l1 = min(n_lists, l0 + lpb);
  const int n = (l1 - l0) * k;
  const unsigned long long* src = in + (size_t)u * user_stride;
  for (int i = threadIdx.x; i < n2; i += blockDim.x) {
    unsigned long long v = 0ull;
    if (i < n) {
      const int l = i / k;
      v = src[(size_t)(l0 + l) * list_stride + (i - l * k)];
    }
    mk[i] = v;
  }
  __syncthreads();
  bitonic_sort_desc(mk, n2);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    if (out_keys) out_keys[((size_t)u * gridDim.y + b) * k + i] = mk[i];
    if (final_level && out_score) {
      float sc;
      int id;
      split_key(mk[i], sc, id);
      out_score[(size_t)u * k + i] = sc;
      out_id[(size_t)u * k + i] = id;
    }
  }
}

// Hierarchical merge of n_lists key lists per user: a level merges blocks of lpb = min(256, 8192 / k) lists; intermediate
// levels write to `scratch` one after the other (merge_scratch_lists(n_lists, k) lists per user in total; NULL is fine when
// one level suffices).  The last level writes out_keys and / or score + id.
int merge_scratch_lists(int n_lists, int k) {
  int lpb = 8192 / k;
  lpb = lpb > 256 ? 256 : (lpb < 2 ? 2 : lpb);
  int total = 0;
  while (n_lists > lpb) {
    n_lists = (n_lists + lpb - 1) / lpb;
    total += n_lists;
  }
  return total;
}
int launch_topk_merge_keys_multi(const unsigned long long* keys, unsigned long long* scratch, int64_t user_stride, int64_t list_stride,
                                 int n_users, int n_lists, int k, unsigned long long* out_keys, float* out_score, int32_t* out_id,
                                 cudaStream_t stream) {
  if (n_users == 0) return 0;
  cudaError_t e = cudaFuncSetAttribute(topk_merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * 8);
  if (e != cudaSuccess) return (int)e;
  const unsigned long long* src = keys;
  unsigned long long* dst = scratch;
  while (true) {
    int lpb = 8192 / k;
    if (lpb > 256) lpb = 256;
    if (lpb < 2) lpb = 2;
    if (lpb > n_lists) lpb = n_lists;
    const int blocks = (n_lists + lpb - 1) / lpb;
    int n2 = 1;
    while (n2 < lpb * k) n2 <<= 1;
    if (n2 > 8192) return NAIS_ERR_SHAPE;
    const bool last = blocks == 1;
    if (!last && !dst) return NAIS_ERR_WORKSPACE;
    dim3 grid(n_users, blocks);
    const int threads = n2 >= 1024 ? 512 : (n2 < 64 ? 64 : n2 / 2);
    topk_merge_keys_kernel<<<grid, threads, (size_t)n2 * 8, stream>>>(src, user_stride, list_stride, n_lists, k, lpb, n2,
                                                                      last ? out_keys : dst, last ? 1 : 0, out_score, out_id);
    NAIS_COUNT_LAUNCH(1);
    e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    if (last) return 0;
    // next level: [u][blocks][k] contiguous in dst; its output goes behind it
    n_lists = blocks;
    user_stride = (int64_t)blocks * k;
    list_stride = k;
    src = dst;
    dst = dst + (size_t)n_users * blocks * k;
  }
}

int launch_fullrank_fp32(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin,
                         int64_t poi_end, int k, int exclude, float* out_score, int32_t* out_id, float* all_scores,
                         void* ws, size_t ws_bytes, cudaStream_t stream, const GeoMixArgs* geo) {
  if (users.n_users == 0 || poi_end <= poi_begin) return 0;
  FullrankArgs A;
  A.geo = geo ? *geo : GeoMixArgs{};
  A.p = p;
  A.cat = cat;
  A.users = users;
  A.poi_begin = poi_begin;
  A.poi_end = poi_end;
  A.k = k;
  A.exclude = exclude;
  A.n_splits = choose_splits(users.n_users, poi_end - poi_begin);
  A.out_score = out_score;
  A.out_id = out_id;
  A.all_scores = all_scores;
  A.part_keys = reinterpret_cast<unsigned long long*>(ws);
  if (A.n_splits > 1 && ws_bytes < (size_t)users.n_users * A.n_splits * k * sizeof(unsigned long long)) return NAIS_ERR_WORKSPACE;
  const size_t smem = fullrank_fp32_smem(p, A.stage_p, A.hc);
  if (smem > 227 * 1024) return NAIS_ERR_SHAPE;
  void (*kern)(const FullrankArgs) = geo ? fullrank_fp32_kernel<true> : fullrank_fp32_kernel<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  dim3 grid(users.n_users, A.n_splits);
  kern<<<grid, NT, smem, stream>>>(A);
  NAIS_COUNT_LAUNCH(1);
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if (A.n_splits > 1) return launch_topk_merge(A.part_keys, nullptr, nullptr, users.n_users, A.n_splits, k, out_score, out_id, stream);
  return 0;
}

}  // namespace nais
