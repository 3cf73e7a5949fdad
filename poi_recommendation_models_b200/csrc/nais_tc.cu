// Tensor-core (tcgen05 / TMEM) full-rank scorer for sm_100a.
//
// Per user u and candidate j the attention logits need t[k] = sum_d W[k,d] q_h[d] p_j[d] for every history item h and
// hidden unit k: a GEMM  T[j, (h,k)] = P[j,:] . B_u[(h,k),:]^T  with  B_u[(h,k), d] = c_k W[k,d] q_h[d]  built ONCE per
// user (pack kernel) and reused against the whole catalogue.  M = 128 candidates (one TMEM lane = one candidate = one
// epilogue thread), N = 2 history items x (hid + 2) rows, K = D + 16:
//
//   * the two distance lanes and the bias are folded into an extra K-step: A_ext[j, 2*hs+c] = g_c(h_hs, j) (written by
//     the epilogue warps, 3 steps ahead), A_ext[j,4] = 1;  B_ext[(hs,k), 2*hs+c] = c_k W[k,D+c], B_ext[.,4] = c_k b_k;
//   * ReLU + second layer in ONE FADD per accumulator element: with c_k = |v_k|/2 and t'_k = c_k t_k,
//         sum_k v_k relu(t_k) = sum_k sgn_k t'_k + sum_k sgn_k |t'_k| = L + sum_{k in pos}|t'_k| - sum_{k in neg}|t'_k|
//     L is linear, so it is one more row of B ("L row"); hidden units are permuted positive-v first;
//   * the similarity s_hj = <q_h, p_j> is another row of B ("S row");
//   * fp32-grade products from fp16 tensor cores: every operand is split x = hi + lo (two fp16 planes, power-of-two
//     pre-scaling), D += A_hi B_hi + A_hi B_lo + A_lo B_hi  (NAIS_PREC_TC_SPLIT).  NAIS_PREC_TC_FAST keeps the three
//     passes only for the S/L rows (an N=16 MMA at a column offset) and runs the main rows single-pass.
//     NAIS_PREC_TC_MIX keeps A_hi B_hi in fp16 and issues the two correction products as e5m2 MMAs
//     (kind::f8f6f4, K = 32 per instruction, same issue time as an fp16 K = 16 MMA): D += A_hi B_hi + e5m2(A_hi) e5m2(B_lo)
//     + e5m2(A_lo) e5m2(B_hi).  e5m2 has fp16's exponent range, so the byte planes need no extra scaling; the corrections
//     are ~2^-12 of the product, so their 3-bit significands leave ~3e-5 per term (1e-5 conditioned, tests/ and
//     examples/precision_emulation.py).  The ext K-step carries its own hi/lo split inside its 16 K slots (one MMA).
//     9 MMA issue slots per step instead of 15.
//
// Warp roles (576 threads, 1 CTA/SM, persistent over work items = (user, 3 candidate tiles)):
//   warps 0-15 epilogue, two groups of 8 alternating steps: lane quarter = warp%4, history slot = (warp/4)%2;
//              produce A_ext, TMEM -> registers, beta-softmax state
//   warp 16    MMA issuer (one elected lane) + TMEM allocation
//   warp 17    bulk-copy producer (one elected lane): A tiles per item, B chunks through a ring of stages
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include <type_traits>

#include "nais_common.cuh"
#include "umma.cuh"

namespace nais {

using namespace umma;

namespace tc {

constexpr int TM = 128;
constexpr int NBUF = 3;          // TMEM accumulator buffers == A_ext buffers == look-ahead of the g producer
constexpr int ACC_STRIDE = 160;  // TMEM columns per accumulator buffer
constexpr int TPC = 3;           // candidate tiles per work item
constexpr int EPI_WARPS = 16;    // two groups of 8 alternate steps
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int ARRIVE_WARPS = 8;  // warps that arrive per step on e_full / acc_empty (one group)
constexpr int THREADS = (EPI_WARPS + 2) * 32;
constexpr int MAX_STAGES = 4;
constexpr int SORTN = 512;
constexpr int HMETA = 512;      // history items whose id/coords are staged in smem per item (longer ones: __ldg)

struct Geo {
  int D, hid, lanes, split;
  int pair;      // CTA pairs (cta_group::2, the headline shape only): a stage holds this CTA's HALF of a B chunk (rows [rank * nrow/2, +nrow/2))
  int km;        // NAIS_DIST_KM: logit += haversine_km(h, j) * sum_d embed_distance[0, d] in the (run-time-shape) epilogue
  int mix;       // NAIS_PREC_TC_MIX: lo section of A tiles / B chunks = e5m2(hi) | e5m2(lo) byte planes, two ext k-chunks
  int kx;        // D / 8 x k-chunks
  int hsplit;    // chunks per history item: 1, or 2 for hid = 256 — a chunk then holds ONE HALF (128) of the item's hidden units
                 // (`hid` below is the per-chunk count); the two halves of a cell are consecutive chunks = the two epilogue groups
  int hch;       // history items per chunk / MMA step: 2 (hid <= 64) or 1 (hid 96, 128: a cell's hidden columns are split
                 // between the two warps of a lane quarter and their partial sums exchanged through shared memory)
  int aux0;      // first S/L row = hch * hid
  int nrow;      // rows of a B chunk (hch*hid + 2*hch S/L rows, padded; at least aux0 + 16 for the N = 16 aux MMA)
  int tpc;       // candidate tiles per item (3, or 2 when the A tiles of D > 64 would not fit)
  int stages;    // B ring depth
  int kp;        // K-parts per B chunk: 1 (D <= 64: a stage = the whole chunk) or D/32 (a stage = 4 x k-chunks of both
                 // planes; the last part also carries the ext k-chunk)
  int kc_part;   // x k-chunks per part
  int part_bytes, part_last_bytes, stage_bytes;
  int a_plane, a_tile;          // bytes
  int b_hi, b_lo, b_chunk;      // bytes (whole chunk, all parts)
  int smem_bytes;
};

__host__ __device__ inline int pad16(int x) { return (x + 15) / 16 * 16; }

__host__ inline bool make_geo(const NaisParams& p, int precision, Geo& g) {
  if (p.n_branch != 1) return false;
  const NaisBranch& br = p.branch[0];
  g.D = br.w_poi + br.w_reg;
  g.hsplit = p.hid == 256 ? 2 : 1;
  g.hid = p.hid / g.hsplit;
  g.lanes = p.dist_mode == NAIS_DIST_LATLON ? 2 : 0;
  g.split = precision == NAIS_PREC_TC_SPLIT;
  g.mix = precision == NAIS_PREC_TC_MIX;
  g.pair = 0;
  g.km = p.dist_mode == NAIS_DIST_KM ? 1 : 0;
  if (g.km && p.dist_buckets != 1) return false;
  if (precision == NAIS_PREC_TC_AUTO) {  // MIX geometry where an e5m2 K-step exists, else SPLIT (same image sizes)
    g.mix = g.D % 32 == 0;
    g.split = !g.mix;
  }
  if (g.mix && g.D % 32) return false;  // an e5m2 MMA covers K = 32
  if (g.D % 16 || g.D < 16 || g.D > 256 || (g.D > 64 && g.D % 32) || g.hid % 16 || g.hid < 16 || g.hid > 128) return false;
  g.hch = g.hid <= 64 ? 2 : 1;
  if (g.hch == 1 && g.hid % 32) return false;
  g.kx = g.D / 8;
  g.aux0 = g.hch * g.hid;
  g.nrow = pad16(g.aux0 + 2 * g.hch);
  if (g.nrow < g.aux0 + 16) g.nrow = g.aux0 + 16;
  if (g.nrow > ACC_STRIDE) return false;
  g.a_plane = g.kx * TM * 16;
  g.a_tile = 2 * g.a_plane;
  // split: hi and lo planes of kx + 1 k-chunks.  mix: hi plane of kx + 2 k-chunks (two ext chunks), lo section = two byte
  // planes of kx/2 k-chunks (16 e5m2 per 16 B).  Same totals.  fast: lo = a 16-row image of the S/L rows.
  g.b_hi = (g.kx + 1 + g.mix) * g.nrow * 16;
  g.b_lo = g.split ? g.b_hi : (g.mix ? g.kx * g.nrow * 16 : (g.kx + 1) * 16 * 16);
  g.b_chunk = g.b_hi + g.b_lo;
  if (g.D <= 64) {
    g.kp = 1;
    g.kc_part = g.kx;
    g.part_bytes = g.part_last_bytes = g.stage_bytes = g.b_chunk;
    g.stages = (g.split || g.mix) ? 2 : 3;
  } else {
    g.kp = g.D / 32;
    g.kc_part = 4;
    const int lo4 = (g.split || g.mix) ? 4 * g.nrow * 16 : 4 * 16 * 16;
    const int lo5 = g.split ? 5 * g.nrow * 16 : (g.mix ? lo4 : 5 * 16 * 16);
    g.part_bytes = 4 * g.nrow * 16 + lo4;
    g.part_last_bytes = g.stage_bytes = (5 + g.mix) * g.nrow * 16 + lo5;
    g.stages = 3;
  }
  // smem: A tiles | B stages | A_ext (hi,lo) x NBUF | zero  (item-end `comb` partials alias A_ext+zero) | keys | hist meta |
  //       partner exchange | barriers
  g.tpc = g.kp == 1 ? TPC : (g.D > 128 ? 1 : 2);  // compile-time constant per kernel instantiation (kSinglePart / kFix == 4)
  g.smem_bytes = g.tpc * g.a_tile + g.stages * g.stage_bytes + NBUF * 2 * TM * 16 + 4096 + SORTN * 8 + 3 * HMETA * 4 + 6 * TM * 4 + 256 + 128 +
                 (g.kp == 1 ? 9 * TPC * TM * 4 : 0) +  // D <= 64 has room for a private `comb`; D > 64 aliases it on A_ext + zero
                 (g.km ? HMETA * 4 : 0);               // cos(latitude) of the staged history items
  return g.smem_bytes <= 227 * 1024;
}

// device-side scalars written by tc_scales_kernel
struct Scales {
  float sA, sS, sB, sAe, sBe, inv_sigma, inv_s;
  int npos;
  float omega0, omega1, omegab;
  float rho;     // maxP * maxB * sqrt(hid * D): scale of the logit sum that the e5m2 corrections' ~3e-5 per-term error multiplies
  int use_mix;   // NAIS_PREC_TC_AUTO: rho <= kMixRhoMax -> the MIX kernels run, else the SPLIT kernels (the others exit at once)
};
// Emulated (examples/precision_emulation.py) conditioned error of MIX: ~1e-5 up to rho ~ 100, 2.3e-5 at 250, 4.7e-5 at 490,
// 1.3e-4 at 1170 (embedding std 1.0 with 4x weights).  MEASURED worst case (tests/test_gpu_gate.py, attention weights scaled
// through the switch, histories of 16..128 items, every candidate of the catalogue): 4.3e-5 at rho = 120, 8.7e-5 at rho = 236 (a
// 16-item history) — so the r1 threshold of 256 left no margin to the 1e-4 bar; 128 keeps a factor 2.
constexpr float kMixRhoMax = 128.f;
// ... and the similarity S_hj carries the same ~3e-5 per-term error into the score directly; it averages out over the
// history but not for a handful of items (emulated worst case over 2000 candidates: H = 64: 1.7e-5, 16: 2.8e-5, 6: 7e-5,
// 2: 1e-3), so under NAIS_PREC_TC_AUTO users with a shorter history than this take the SPLIT pass (they are cheap anyway).
constexpr int kMixMinHist = 16;
// NAIS_PREC_TC_AUTO runs a MIX pass (gate 1) and a SPLIT pass (gate 0) over the same user batch; each user belongs to one.
__device__ __forceinline__ bool user_in_pass(int gate, int use_mix, int H) {
  return gate < 0 || ((use_mix && H >= kMixMinHist) ? 1 : 0) == gate;
}
// workspace header: [0,64) maxes (uint bits) | [64,128) Scales | perm[256] int | ck[256] float | u[256] float
constexpr int HDR_BYTES = 4096;
constexpr int HDR_PERM = 128, HDR_CK = HDR_PERM + 256 * 4, HDR_U = HDR_CK + 256 * 4;
static_assert(HDR_U + 256 * 4 <= HDR_BYTES, "header");

__global__ void absmax_kernel(const float* __restrict__ x, size_t n, unsigned* out) {
  float m = 0.f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));  // non-negative floats order like their bit patterns
}

__device__ __forceinline__ float pow2floor(float x) { return exp2f(floorf(log2f(x))); }

// One CTA: permutation (positive v first), c_k, u_d, omegas, power-of-two scales.
__global__ void scales_kernel(NaisParams p, unsigned char* hdr) {
  const NaisBranch& br = p.branch[0];
  const int D = br.w_poi + br.w_reg, hid = p.hid;
  const int lanes = p.dist_mode == NAIS_DIST_LATLON ? 2 : 0, ldw = D + lanes;
  const unsigned* mx = reinterpret_cast<const unsigned*>(hdr);
  Scales* sc = reinterpret_cast<Scales*>(hdr + 64);
  int* perm = reinterpret_cast<int*>(hdr + HDR_PERM);
  float* ck = reinterpret_cast<float*>(hdr + HDR_CK);
  float* u = reinterpret_cast<float*>(hdr + HDR_U);
  __shared__ float red[8];
  __shared__ int s_npos;
  if (threadIdx.x == 0) {
    int n = 0;
    for (int k = 0; k < hid; ++k)
      if (br.w2[k] >= 0.f) perm[n++] = k;
    s_npos = n;
    for (int k = 0; k < hid; ++k)
      if (!(br.w2[k] >= 0.f)) perm[n++] = k;
    for (int i = 0; i < 8; ++i) red[i] = 0.f;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < hid; k += blockDim.x) ck[k] = 0.5f * fabsf(br.w2[k]);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float a = 0.f;
    for (int k = 0; k < hid; ++k) a += 0.5f * br.w2[k] * br.w1[(size_t)k * ldw + d];
    u[d] = a;
  }
  __syncthreads();
  // maxima of the MLP-derived operand factors
  float mcw = 0.f, mbe = 0.f;
  for (int i = threadIdx.x; i < hid * D; i += blockDim.x) {
    int k = i / D, d = i - k * D;
    mcw = fmaxf(mcw, fabsf(ck[k] * br.w1[(size_t)k * ldw + d]));
  }
  for (int d = threadIdx.x; d < D; d += blockDim.x) mcw = fmaxf(mcw, fabsf(u[d]));
  for (int k = threadIdx.x; k < hid; k += blockDim.x) {
    mbe = fmaxf(mbe, fabsf(ck[k] * br.b1[k]));
    if (lanes) {
      mbe = fmaxf(mbe, fabsf(ck[k] * br.w1[(size_t)k * ldw + D]));
      mbe = fmaxf(mbe, fabsf(ck[k] * br.w1[(size_t)k * ldw + D + 1]));
    }
  }
  atomicMax(reinterpret_cast<unsigned*>(&red[0]), __float_as_uint(mcw));
  atomicMax(reinterpret_cast<unsigned*>(&red[1]), __float_as_uint(mbe));
  __syncthreads();
  if (threadIdx.x == 0) {
    float o0 = 0.f, o1 = 0.f, ob = 0.f;
    for (int k = 0; k < hid; ++k) {
      const float hv = 0.5f * br.w2[k];
      ob += hv * br.b1[k];
      if (lanes) {
        o0 += hv * br.w1[(size_t)k * ldw + D];
        o1 += hv * br.w1[(size_t)k * ldw + D + 1];
      }
    }
    const float tiny = 1e-30f;
    const float maxP = fmaxf(fmaxf(__uint_as_float(mx[0]), __uint_as_float(mx[1])), tiny);
    const float maxQ = fmaxf(fmaxf(__uint_as_float(mx[2]), __uint_as_float(mx[3])), tiny);
    const float maxB = fmaxf(maxQ * red[0], tiny);
    const float maxBe = fmaxf(fmaxf(red[1], fmaxf(fabsf(o0), fmaxf(fabsf(o1), fabsf(ob)))), tiny);
    float sA = pow2floor(512.f / maxP), sS = pow2floor(512.f / maxQ), sB = pow2floor(512.f / maxB);
    const float sAe = 256.f;
    // ext products must carry the same scale sigma = sA*sB = sAe*sBe and stay inside fp16
    float sBe = sA * sB / sAe;
    while (maxBe * sBe > 16384.f) {
      sB *= 0.5f;
      sBe *= 0.5f;
    }
    sc->sA = sA;
    sc->sS = sS;
    sc->sB = sB;
    sc->sAe = sAe;
    sc->sBe = sBe;
    sc->inv_sigma = 1.f / (sA * sB);
    sc->inv_s = 1.f / (sA * sS);
    sc->npos = s_npos;
    sc->omega0 = o0;
    sc->omega1 = o1;
    sc->omegab = ob;
    sc->rho = maxP * maxB * sqrtf((float)(hid * D));
    sc->use_mix = sc->rho <= kMixRhoMax ? 1 : 0;
  }
}

// 8 fp16 -> 8 e5m2 bytes (round to nearest even; e5m2 shares fp16's exponent range, so no rescaling)
__device__ __forceinline__ uint2 pack_e5m2(const __half* h) {
  unsigned char b[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) b[e] = (unsigned char)__nv_cvt_halfraw_to_fp8(static_cast<__half_raw>(h[e]), __NV_SATFINITE, __NV_E5M2);
  uint2 r;
  r.x = b[0] | (b[1] << 8) | (b[2] << 16) | ((unsigned)b[3] << 24);
  r.y = b[4] | (b[5] << 8) | (b[6] << 16) | ((unsigned)b[7] << 24);
  return r;
}

// Candidate tiles: image [tile][plane hi|lo][k-chunk][row][8 x fp16] of p_j * sA.  One thread = (row, k-chunk).
__global__ void pack_candidates_kernel(NaisParams p, NaisCatalog cat, int64_t poi_begin, int64_t poi_end, Geo g,
                                       const unsigned char* hdr, unsigned char* Pimg) {
  const NaisBranch& br = p.branch[0];
  const Scales* sc = reinterpret_cast<const Scales*>(hdr + 64);
  const float sA = sc->sA;
  const int tile = blockIdx.x;
  for (int i = threadIdx.x; i < TM * g.kx; i += blockDim.x) {
    const int c = i / TM, r = i - c * TM;
    const int64_t j = poi_begin + (int64_t)tile * TM + r;
    __half hi[8], lo[8];
    if (j < poi_end) {
      const int64_t jl = j - cat.row_base;
      for (int e = 0; e < 8; ++e) {
        const int d = c * 8 + e;
        const float v = (d < br.w_poi) ? __ldg(br.tgt_poi + (size_t)j * br.w_poi + d)
                                       : __ldg(br.tgt_reg + (size_t)__ldg(cat.region + jl) * br.w_reg + (d - br.w_poi));
        split_f16(v * sA, hi[e], lo[e]);
      }
    } else {
      for (int e = 0; e < 8; ++e) hi[e] = lo[e] = __float2half(0.f);
    }
    unsigned char* base = Pimg + (size_t)tile * g.a_tile + ((size_t)c * TM + r) * 16;
    *reinterpret_cast<uint4*>(base) = *reinterpret_cast<uint4*>(hi);
    if (g.mix) {  // byte planes e5m2(hi) | e5m2(lo): 16 K elements per 16 B, this thread owns half a row of one k-chunk
      unsigned char* b8 = Pimg + (size_t)tile * g.a_tile + g.a_plane + ((size_t)(c >> 1) * TM + r) * 16 + (c & 1) * 8;
      *reinterpret_cast<uint2*>(b8) = pack_e5m2(hi);
      *reinterpret_cast<uint2*>(b8 + g.a_plane / 2) = pack_e5m2(lo);
    } else {
      *reinterpret_cast<uint4*>(base + g.a_plane) = *reinterpret_cast<uint4*>(lo);
    }
  }
}

// first chunk slot of user u: users get ceil(H/hch) consecutive slots (hch = 2: (offsets[u] + u) / 2 never overlaps)
__device__ __forceinline__ int64_t chunk_base(const int64_t* offsets, int u, int hch, int hsplit = 1) {
  return hch == 2 ? (offsets[u] + u) >> 1 : offsets[u] * hsplit;
}

// User operand: grid (user, chunk slot) — users ride grid.x, which has no 65 535 limit.  One thread = (row n, k-chunk c) -> 8 fp16 (hi) + 8 fp16 (lo).
// NAIS_PREC_TC_AUTO (two_pass): every user is packed in the image format of the pass that scores it — `g` (MIX geometry) for
// the users of pass 1, `gs` (SPLIT geometry, same image sizes) for those of pass 0 — and pass_flags[pass] is raised so a pass
// without users exits at once.  Otherwise everybody takes `g`.
__global__ void pack_users_kernel(NaisParams p, NaisUsers users, Geo g_mix, Geo g_split, int two_pass, const unsigned char* hdr,
                                  unsigned char* Bimg, int64_t max_chunks, int* pass_flags, int* bad) {
  const NaisBranch& br = p.branch[0];
  const Scales* sc = reinterpret_cast<const Scales*>(hdr + 64);
  const int* perm = reinterpret_cast<const int*>(hdr + HDR_PERM);
  const float* ck = reinterpret_cast<const float*>(hdr + HDR_CK);
  const float* uu = reinterpret_cast<const float*>(hdr + HDR_U);
  const int u = blockIdx.x;
  const int64_t hb = users.offsets[u];
  const int H = (int)(users.offsets[u + 1] - hb);
  int pass = 1;
  if (two_pass) {
    pass = user_in_pass(1, sc->use_mix, H) ? 1 : 0;
    if (threadIdx.x == 0 && blockIdx.y == 0) pass_flags[pass] = 1;  // (benign race: every writer stores 1)
  }
  const Geo& g = pass ? g_mix : g_split;
  const int hch = g.hch, aux0 = g.aux0, hsplit = g.hsplit;
  const int nchunks = (H + hch - 1) / hch * hsplit;
  const int D = g.D, hid = g.hid, ldw = D + g.lanes;
  __shared__ float q[2][256];
  for (int chunk = blockIdx.y; chunk < nchunks; chunk += gridDim.y) {
    const int hc = chunk / hsplit, half = chunk - hc * hsplit;  // history chunk, and which half of its hidden units this image holds
    __syncthreads();
    for (int i = threadIdx.x; i < hch * D; i += blockDim.x) {
      const int hs = i / D, d = i - hs * D, h = hch * hc + hs;
      float v = 0.f;
      if (h < H) {
        const int64_t e = hb + h;
        v = (d < br.w_poi) ? __ldg(br.hist_poi + (size_t)checked_id(__ldg(users.items + e), p.item_num, bad) * br.w_poi + d)
                           : __ldg(br.hist_reg + (size_t)checked_id(__ldg(users.region + e), p.region_num, bad) * br.w_reg + (d - br.w_poi));
      }
      q[hs][d] = v;
    }
    __syncthreads();
    const int64_t slot = chunk_base(users.offsets, u, hch, hsplit) - chunk_base(users.offsets, 0, hch, hsplit) + chunk;
    if (slot >= max_chunks) continue;  // workspace sized with a wrong nnz: never write out of bounds (the main kernel clamps too)
    unsigned char* cb = Bimg + (size_t)slot * g.b_chunk;
    for (int i = threadIdx.x; i < g.nrow * (g.kx + 1); i += blockDim.x) {
      const int c = i / g.nrow, n = i - c * g.nrow;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = 0.f;
      int hs = -1, kind = -1, k = 0;  // kind 0 main, 1 S, 2 L
      if (n < aux0) {
        hs = n / hid;
        kind = 0;
        k = perm[half * hid + n - hs * hid];
      } else if (n < aux0 + 2 * hch && half == 0) {  // S / L rows ride with the first half only (L already sums over ALL hidden units)
        hs = (n - aux0) >> 1;
        kind = 1 + ((n - aux0) & 1);
      }
      if (kind >= 0 && hch * hc + hs < H) {
        if (c < g.kx) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int d = c * 8 + e;
            const float qd = q[hs][d];
            if (kind == 0) v[e] = ck[k] * __ldg(br.w1 + (size_t)k * ldw + d) * qd * sc->sB;
            else if (kind == 1) v[e] = qd * sc->sS;
            else v[e] = uu[d] * qd * sc->sB;
          }
        } else if (g.mix) {  // handled below (the ext values carry their own hi/lo split inside the two ext k-chunks)
        } else {  // ext chunk: [2*hs + lane] distance lanes, [4] bias
          if (kind == 0) {
            if (g.lanes) {
              v[2 * hs] = ck[k] * __ldg(br.w1 + (size_t)k * ldw + D) * sc->sBe;
              v[2 * hs + 1] = ck[k] * __ldg(br.w1 + (size_t)k * ldw + D + 1) * sc->sBe;
            }
            v[4] = ck[k] * __ldg(br.b1 + k) * sc->sBe;
          } else if (kind == 2) {
            v[2 * hs] = sc->omega0 * sc->sBe;
            v[2 * hs + 1] = sc->omega1 * sc->sBe;
            v[4] = sc->omegab * sc->sBe;
          }
        }
      }
      __half hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) split_f16(v[e], hi[e], lo[e]);
      // image = [part][hi plane | lo section][k-chunk in part][row][16 B]; one part = one bulk copy = one smem stage.
      // g.pair (kp == 1): [half][hi plane | lo section][k-chunk][row % (nrow/2)][16 B] — each CTA of a pair copies its half
      const int part = g.kp == 1 ? 0 : min(c / g.kc_part, g.kp - 1);
      const int cp = c - part * g.kc_part;                          // k-chunk inside the part
      const int nkc = g.kc_part + (part == g.kp - 1 ? 1 + g.mix : 0);  // the last part also holds the ext k-chunk(s)
      const int nrw = g.pair ? g.nrow / 2 : g.nrow;                 // rows of an image plane
      const int nn = g.pair ? n % nrw : n;                          // row inside it
      unsigned char* pb = cb + (size_t)part * g.part_bytes + (g.pair ? (size_t)(n / nrw) * (g.b_chunk / 2) : 0);
      unsigned char* lb = pb + (size_t)nkc * nrw * 16;
      if (g.mix && c == g.kx) {
        // ext step of the MIX mode, ONE fp16 MMA over 16 K slots with the split inside (w = lane / bias weights * sBe):
        //   chunk e0: [2hs+l] = hi(w_l)   [4] = hi(w_b)  [5] = lo(w_b)        A_ext: [2hs+l] = hi(g_l)  [4] = [5] = sAe
        //   chunk e1: [2hs+l] = hi(w_l)   [4+2hs+l] = lo(w_l)                 A_ext: [2hs+l] = lo(g_l)  [4+2hs+l] = hi(g_l)
        float w0 = 0.f, w1 = 0.f, wb = 0.f;
        if (kind == 0 && hch * hc + hs < H) {
          if (g.lanes) {
            w0 = ck[k] * __ldg(br.w1 + (size_t)k * ldw + D) * sc->sBe;
            w1 = ck[k] * __ldg(br.w1 + (size_t)k * ldw + D + 1) * sc->sBe;
          }
          wb = ck[k] * __ldg(br.b1 + k) * sc->sBe;
        } else if (kind == 2 && hch * hc + hs < H) {
          w0 = sc->omega0 * sc->sBe;
          w1 = sc->omega1 * sc->sBe;
          wb = sc->omegab * sc->sBe;
        }
        __half e0[8], e1[8], h0, l0, h1, l1, hb, lb2;
#pragma unroll
        for (int e = 0; e < 8; ++e) e0[e] = e1[e] = __float2half(0.f);
        split_f16(w0, h0, l0);
        split_f16(w1, h1, l1);
        split_f16(wb, hb, lb2);
        if (hs >= 0) {
          e0[2 * hs] = h0;
          e0[2 * hs + 1] = h1;
          e0[4] = hb;
          e0[5] = lb2;
          e1[2 * hs] = h0;
          e1[2 * hs + 1] = h1;
          e1[4 + 2 * hs] = l0;
          e1[5 + 2 * hs] = l1;
        }
        *reinterpret_cast<uint4*>(pb + ((size_t)cp * nrw + nn) * 16) = *reinterpret_cast<uint4*>(e0);
        *reinterpret_cast<uint4*>(pb + ((size_t)(cp + 1) * nrw + nn) * 16) = *reinterpret_cast<uint4*>(e1);
        continue;
      }
      *reinterpret_cast<uint4*>(pb + ((size_t)cp * nrw + nn) * 16) = *reinterpret_cast<uint4*>(hi);
      if (g.mix) {
        unsigned char* b8 = lb + ((size_t)(cp >> 1) * nrw + nn) * 16 + (cp & 1) * 8;
        *reinterpret_cast<uint2*>(b8) = pack_e5m2(hi);
        *reinterpret_cast<uint2*>(b8 + (size_t)(g.kc_part / 2) * nrw * 16) = pack_e5m2(lo);
      } else if (g.split) {
        *reinterpret_cast<uint4*>(lb + ((size_t)cp * nrw + nn) * 16) = *reinterpret_cast<uint4*>(lo);
      } else if (n >= aux0 && n < aux0 + 16) {
        *reinterpret_cast<uint4*>(lb + ((size_t)cp * 16 + (n - aux0)) * 16) = *reinterpret_cast<uint4*>(lo);
      }
    }
  }
}

// chunks of user u that exist in the operand image (== ceil(H / hch) when the workspace was sized correctly)
__device__ __forceinline__ int user_chunks(const int64_t* offsets, int u, int hch, int64_t cb0, int64_t max_chunks, int hsplit = 1) {
  const int H = (int)(offsets[u + 1] - offsets[u]);
  const int64_t room = max_chunks - (chunk_base(offsets, u, hch, hsplit) - cb0);
  const int n = (H + hch - 1) / hch * hsplit;
  const int m = (int)(room < n ? (room < 0 ? 0 : room) : n);
  return m - m % hsplit;  // both halves of an item or neither (the two epilogue groups meet once per item)
}

struct MainArgs {
  NaisParams p;
  NaisCatalog cat;
  NaisUsers users;
  Geo g;
  int64_t poi_begin, poi_end;
  int k, exclude, groups;         // groups: candidate-tile groups of the range (pair kernels: rounded up to even, see groups_real)
  int groups_real;                // groups that exist (the key lists have this many per user)
  int64_t n_items;                // (user, group) items; pair kernels: (user, pair of groups) items
  const unsigned char* hdr;
  const unsigned char* Pimg;
  const unsigned char* Bimg;
  unsigned long long* part_keys;  // [n_users, groups, k]
  float* all_scores;              // optional [n_users, range]
  const float* score_in;          // optional [n_users, range]: added to the score before it is stored / ranked (the other
                                  // attention branch of the two-branch model, scored by an earlier pass; may alias all_scores)
  int64_t max_chunks;             // chunk slots the operand image holds (users beyond it are truncated, never read out of bounds)
  int gate;                       // -1: one pass scores every user; 0 / 1: the SPLIT / MIX pass of NAIS_PREC_TC_AUTO
  const int* pass_flags;          // [2] raised by pack_users_kernel for every pass that has users (gate >= 0)
  GeoMixArgs geo;                 // kGeo kernels: rank by the power-law mix (nais_fullrank_topk_geo_planned)
};

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

// kSinglePart: D <= 64, a B stage holds a whole chunk (kp == 1).  kHch: history items per MMA step (2: hid <= 64, 1: hid 96/128).
// 32 keys, one per lane -> sorted descending across the lanes (bitonic network on shuffles)
__device__ __forceinline__ unsigned long long warp_sort_desc(unsigned long long v, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, j);
      const bool desc = k == 32 || (lane & k) == 0, lower = (lane & j) == 0;
      v = (lower == desc) ? (v > o ? v : o) : (v < o ? v : o);
    }
  }
  return v;
}
// two descending rows -> the best 32 of both, descending
__device__ __forceinline__ unsigned long long warp_fold_top32(unsigned long long a, unsigned long long b, int lane) {
  const unsigned long long br = __shfl_sync(0xffffffffu, b, 31 - lane);
  unsigned long long v = a > br ? a : br;
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, j);
    v = ((lane & j) == 0) ? (v > o ? v : o) : (v < o ? v : o);
  }
  return v;
}

// kFix: 0 = generic (every shape is a run-time value); 1 / 2 = the D = hid = 64 shape of the headline workload in SPLIT / MIX
// precision with every tile constant known at compile time: a fully unrolled MMA issue sequence (descriptor = base +
// immediate; the generic issuer spends ~15 instructions per MMA, which paces the kernel once a step is 9 MMAs) and the
// specialised epilogue step loop (needs kSinglePart and kHch == 2).
// kS: the static shape D = hid = kS of kFix 1 / 2 (64: the headline workload; 32: the small end of the C5 sweep).
// kGeo (run-time-shape kernels only, kFix 0 / 4): every cell also adds its power-law term ln a + b ln max(0.01, d_km) to a
// per-candidate log G partial (same exactly-once guard and `comb` combination as sumE / sumES, the h = j cell included), and the
// item epilogue ranks by geo_mixed(score, log G, M_u).  Extra shared memory: geo_extra_smem.
template <bool kSinglePart, int kHch, int kFix, int kS = 64, bool kGeo = false>
__global__ void __launch_bounds__(THREADS, 1) fullrank_tc_kernel(const __grid_constant__ MainArgs A) {
  // kFix == 5 / 6: kFix 1 / 2 on CTA PAIRS (cta_group::2): the two CTAs of a cluster score the same user against two neighbouring
  // groups of candidate tiles with ONE M = 256 MMA per step — each supplies its 128 candidates (A) and HALF of the user's chunk (B)
  // from its own shared memory, which takes the operand traffic per MMA from 8.7 KB to 6.3 KB per SM (the measured limiter of the
  // one-CTA kernel: 94 % of the shared-memory port, tensor pipe 77 % active).  Rank 0 issues; rank 1's MMA warp relays "my operands
  // have landed" to rank 0's barriers; commits are multicast to both; the epilogue warps of both arrive on rank 0's e_full / acc_empty.
  constexpr bool kPair = kFix == 5 || kFix == 6;
  constexpr bool kFastEpi = kFix == 1 || kFix == 2 || kPair;
  // kFix == 3: D = hid = 128 (the reference's default, run.py:837-838) in SPLIT / MIX: the generic code paths below with the
  // shape constants known at compile time, so the K-part / K-step loops of the issuer unroll and its descriptors fold
  constexpr bool kD128 = kFix == 3;
  static_assert(!kGeo || kFix == 0 || kFix == 4, "geo mode lives in the run-time-shape epilogue");
  // `comb` arrays per partial set (sumE, sumES, excl [, log G]) and its tile stride: D > 64 aliases it on the 16 KB of A_ext + zero,
  // where 4 arrays fit only at the tpc <= 2 those kernels run with
  constexpr int kCombA = kGeo ? 4 : 3, kCombT = (kGeo && !kSinglePart) ? 2 : TPC;
  extern __shared__ __align__(128) unsigned char smem[];
  const Geo& g = A.g;
  unsigned char* sA = smem;
  unsigned char* sB = sA + g.tpc * g.a_tile;
  unsigned char* sE = sB + g.stages * g.stage_bytes;          // A_ext: [NBUF][hi 2KB | lo 2KB]
  unsigned char* sZ = sE + NBUF * 2 * TM * 16;            // 4 KB of zeros (aliased second k-chunk of the ext step)
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(sZ + 4096);  // [SORTN]
  // item-end partial sums [3 partial sets][3 arrays][TPC][TM] = 13.5 KB.  D <= 64: private region.  D > 64 (smem is full):
  // ALIASES A_ext + zero (16 KB), only touched between the item-end barriers, then re-initialised.
  float* comb = kSinglePart ? reinterpret_cast<float*>(keys + SORTN) : reinterpret_cast<float*>(sE);
  int* hm_id = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(keys + SORTN) + (kSinglePart ? 3 * kCombA * TPC * TM * 4 : 0));  // [HMETA]
  float* hm_la = reinterpret_cast<float*>(hm_id + HMETA);
  float* hm_lo = hm_la + HMETA;
  float* xch = hm_lo + HMETA;                                                   // [2][3][TM] partner-warp exchange (hch = 1; 3 senders when hsplit = 2)
  uint64_t* bars = reinterpret_cast<uint64_t*>(xch + 6 * TM);
  uint64_t* a_full = bars + 0;
  uint64_t* a_empty = bars + 1;
  uint64_t* b_full = bars + 2;                 // [MAX_STAGES]
  uint64_t* b_empty = bars + 2 + MAX_STAGES;   // [MAX_STAGES]
  uint64_t* e_full = bars + 2 + 2 * MAX_STAGES;          // [NBUF] A_ext written
  uint64_t* acc_full = e_full + NBUF;                    // [2][NBUF] MMA done, one set per epilogue group: a parity
                                                          // wait is only valid if the waiter observes EVERY phase in order
  uint64_t* acc_empty = acc_full + 2 * NBUF;             // [NBUF] accumulator drained
  uint32_t* tslot = reinterpret_cast<uint32_t*>(acc_empty + NBUF);
  float* hm_cos = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bars) + 384);  // [HMETA] (g.km only)
  uint64_t* a_full_peer = reinterpret_cast<uint64_t*>(tslot + 2);  // (pair kernels, rank 0) rank 1's A tiles / B half have landed
  uint64_t* b_full_peer = a_full_peer + 1;                         // [MAX_STAGES]
  uint32_t crank = 0;                                              // rank in the CTA pair
  if constexpr (kPair) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
  // one (user, group) item per CTA and iteration; a pair takes the two neighbouring groups 2 * (item % groups/2) + rank
  const int64_t item0 = kPair ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x, item_step = kPair ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;
  const int groups_it = kPair ? A.groups / 2 : A.groups;  // items per user

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const Scales sc = *reinterpret_cast<const Scales*>(A.hdr + 64);
  if (A.gate >= 0 && !A.pass_flags[A.gate]) return;  // NAIS_PREC_TC_AUTO, no user takes this pass: whole grid, before any barrier

  // ---- one-time setup ---------------------------------------------------------------------------------------------
  // A_ext (3 x hi|lo planes) and the zero region: everything 0 except column 4 of each hi plane = 1.0 * sAe (bias lane)
  auto init_ext_word = [&](int i) {  // i = 32-bit word index inside [sE, sZ + 4096)
    const int byte = i * 4, in_buf = byte % (2 * TM * 16);
    const bool bias = byte < NBUF * 2 * TM * 16 && in_buf < TM * 16 && (in_buf & 15) == 8;  // halves 4,5 of a hi-plane row
    const uint32_t one = (uint32_t)__half_as_ushort(__float2half(sc.sAe));
    // split / fast: slot 4 = 1 (bias).  mix: the buffer is [k-chunk 0 | k-chunk 1] and slots 4, 5 of chunk 0 pair with hi / lo of the bias
    reinterpret_cast<uint32_t*>(sE)[i] = bias ? (g.mix ? (one | (one << 16)) : one) : 0u;
  };
  for (int i = tid; i < (NBUF * 2 * TM * 16 + 4096) / 4; i += THREADS) init_ext_word(i);
  if (kFastEpi && tid < 16) xch[tid] = ((sc.npos & ~15) + tid < sc.npos) ? 1.f : -1.f;
  if (tid == 0) {
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int i = 0; i < MAX_STAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < NBUF; ++i) {
      mbar_init(&e_full[i], kPair ? 2 * ARRIVE_WARPS : ARRIVE_WARPS);
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_full[NBUF + i], 1);
      mbar_init(&acc_empty[i], kPair ? 2 * ARRIVE_WARPS : ARRIVE_WARPS);
    }
    if (kPair) {
      mbar_init(a_full_peer, 1);
      for (int i = 0; i < MAX_STAGES; ++i) mbar_init(&b_full_peer[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == EPI_WARPS) {
    if constexpr (kPair) tmem_alloc2(tslot, 512);
    else tmem_alloc(tslot, 512);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();  // both CTAs' barriers exist before anybody arrives on the other's
  tc_fence_after();
  const uint32_t tmem = *tslot;

  constexpr int tpc = kSinglePart ? TPC : (kFix == 4 ? 1 : 2);  // == g.tpc (kFix == 4: D > 128, one 128 KB candidate tile resident)
  const int hsplit = kHch == 1 ? g.hsplit : 1;
  const int64_t cb0 = chunk_base(A.users.offsets, 0, kHch, hsplit);

  if (warp == EPI_WARPS + 1) {
    // =================================================== bulk-copy producer ========================================
    // (warp-uniform control flow, one elected lane issues; see the MMA warp)
    {
      uint32_t it_n = 0, bstep = 0;  // it_n counts the items this pass processes (all three roles skip the same ones)
      for (int64_t item = item0; item < A.n_items; item += item_step) {
        const int u = (int)(item / groups_it), grp = kPair ? 2 * (int)(item % groups_it) + (int)crank : (int)(item % groups_it);
        if (!user_in_pass(A.gate, sc.use_mix, (int)(A.users.offsets[u + 1] - A.users.offsets[u]))) continue;
        const uint32_t it = it_n++;
        const int64_t cbu = __shfl_sync(0xffffffffu, chunk_base(A.users.offsets, u, kHch, hsplit) - cb0, 0);
        const int nchunks = __shfl_sync(0xffffffffu, user_chunks(A.users.offsets, u, kHch, cb0, A.max_chunks, hsplit), 0);
        mbar_wait(a_empty, (it & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(a_full, (uint32_t)(tpc * g.a_tile));
          for (int t = 0; t < tpc; ++t)
            bulk_g2s(sA + (size_t)t * g.a_tile, A.Pimg + ((size_t)grp * tpc + t) * g.a_tile, (uint32_t)g.a_tile, a_full);
        }
        __syncwarp();
        const unsigned char* src = A.Bimg + (size_t)cbu * g.b_chunk + (kPair ? (size_t)crank * (g.b_chunk / 2) : 0);
        for (int c = 0; c < nchunks; ++c) {
          const int kp_t = kSinglePart ? 1 : g.kp;
          for (int pp = 0; pp < kp_t; ++pp, ++bstep) {
            const int st = bstep % g.stages;
            const uint32_t bytes = kPair ? (uint32_t)(g.b_chunk / 2) : (uint32_t)(pp == kp_t - 1 ? g.part_last_bytes : g.part_bytes);
            mbar_wait(&b_empty[st], ((bstep / g.stages) & 1) ^ 1);
            if (elect_one()) {
              mbar_expect_tx(&b_full[st], bytes);
              bulk_g2s(sB + (size_t)st * g.stage_bytes, src + (size_t)c * g.b_chunk + (size_t)pp * g.part_bytes, bytes, &b_full[st]);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp == EPI_WARPS) {
    // =================================================== MMA issuer ================================================
    // One thread issues 3*(D/16+1) MMAs per step, so the issue path must be a handful of integer ops per MMA: every
    // shared-memory descriptor is (constant high word, low word = base + index*delta), and a K-step only adds a
    // constant to the 14-bit start-address field of the low word.
    // The whole warp runs the (warp-uniform) control flow so descriptors live in uniform registers; only the MMA and
    // commit instructions are predicated on one elected lane (a `if (lane == 0)` region would make ptxas wrap every
    // UTCHMMA in an R2UR waterfall loop, ~130 clk per MMA).
    // A B chunk arrives in g.kp K-parts (one smem stage each); the tpc accumulators of a chunk stay open across the
    // parts, the ext K-step and the commit come with the last part.
    if constexpr (kFastEpi) {
      // ---- static issuer: D = hid = kS, N = 2 kS + 16, K-steps kS/16 (fp16) + 1 (ext) [+ 2 x kS/32 e5m2], stages = 2, buffer == tile ----
      constexpr bool kMix = kFix == 2 || kFix == 6;
      constexpr uint32_t kStages = kPair ? 4u : 2u;  // B ring depth (== g.stages); pairs: half-chunk stages, same bytes in flight
      constexpr uint32_t kKx = kS / 8, kK16 = kS / 16, kK32 = kS / 32;               // x k-chunks, fp16 / e5m2 K-steps
      constexpr uint32_t kNrow = 2 * kS + 16, kALbo = TM * 16;                       // 144 (kS = 64) / 80 (32)
      constexpr uint32_t kBLbo = (kPair ? kNrow / 2 : kNrow) * 16;                  // rows of a B image plane in THIS CTA's stage
      constexpr uint32_t kAStep = (2 * kALbo) >> 4, kBStep = (2 * kBLbo) >> 4;      // one K-step = two 16-byte k-chunks
      constexpr uint32_t kAPlane = kKx * TM * 16, kATile = (2 * kAPlane) >> 4;      // (16-byte units)
      constexpr uint32_t kStage = (2 * (kKx + 1) * kBLbo) >> 4;
      constexpr uint32_t kExtBuf = (2 * TM * 16) >> 4;
      constexpr uint32_t idN = idesc_f16(kPair ? 2 * TM : TM, kNrow), idN8 = idesc_e5m2(kPair ? 2 * TM : TM, kNrow);
      auto mmaH = [](uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
        if constexpr (kPair) mma2_f16(d, a, b, id, acc);
        else mma_f16(d, a, b, id, acc);
      };
      auto mmaQ = [](uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
        if constexpr (kPair) mma2_f8(d, a, b, id, acc);
        else mma_f8(d, a, b, id, acc);
      };
      auto commit = [](uint64_t* bar) {
        if constexpr (kPair) mma2_commit_multicast(bar, 3);
        else mma_commit(bar);
      };
      const uint32_t zaddr = smem_u32(sZ);
      const uint32_t hi_word = (uint32_t)(smem_desc(0, 0, 128) >> 32);  // SBO = 128 B, version 1, no swizzle
      auto lo_of = [](uint32_t addr, uint32_t lbo) { return ((addr >> 4) & 0x3FFFu) | (((lbo >> 4) & 0x3FFFu) << 16); };
      auto mk = [&](uint32_t lo) { return ((uint64_t)hi_word << 32) | lo; };
      const uint32_t sa0 = smem_u32(sA), sb0 = smem_u32(sB), se0 = smem_u32(sE);
      const uint32_t A_hi = lo_of(sa0, kALbo);
      const uint32_t A_lo = lo_of(sa0 + kAPlane, kALbo);                    // split: fp16 lo plane ; mix: e5m2(hi) plane
      const uint32_t A_l8 = lo_of(sa0 + kAPlane + kAPlane / 2, kALbo);      // mix: e5m2(lo) plane
      // split: ext step = k-chunk [hi | lo plane] + zero-aliased second chunk (LBO shrinks as the start grows)
      const uint32_t E_hi = lo_of(se0, zaddr - se0), E_lo = lo_of(se0 + TM * 16, zaddr - se0 - TM * 16);
      constexpr uint32_t kEz = kExtBuf - (kExtBuf << 16), kBz = kStage - (kStage << 16);
      const uint32_t E_mx = lo_of(se0, TM * 16);                            // mix: [chunk 0 | chunk 1]
      const uint32_t B_hi = lo_of(sb0, kBLbo);
      const uint32_t Bx_hi = lo_of(sb0 + kKx * kBLbo, zaddr - (sb0 + kKx * kBLbo));                  // split: ext chunk of the hi plane
      const uint32_t Bx_lo = lo_of(sb0 + (2 * kKx + 1) * kBLbo, zaddr - (sb0 + (2 * kKx + 1) * kBLbo));  //  ... of the lo plane
      uint32_t it_n = 0, cc = 0, st = 0, stph = 0;
      for (int64_t item = item0; item < A.n_items; item += item_step) {
        const int u = (int)(item / groups_it);
        if (!user_in_pass(A.gate, sc.use_mix, (int)(A.users.offsets[u + 1] - A.users.offsets[u]))) continue;
        const uint32_t it = it_n++;
        const int nchunks = __shfl_sync(0xffffffffu, user_chunks(A.users.offsets, u, kHch, cb0, A.max_chunks, hsplit), 0);
        mbar_wait(a_full, it & 1);
        if constexpr (kPair) {
          if (crank != 0) {  // rank 1: nothing to issue — tell rank 0 when this CTA's A tiles / B halves have landed
            if (elect_one()) mbar_arrive_cluster(a_full_peer, 0);
            __syncwarp();
            for (int c = 0; c < nchunks; ++c) {
              mbar_wait(&b_full[st], stph);
              if (elect_one()) mbar_arrive_cluster(&b_full_peer[st], 0);
              __syncwarp();
              st = (st + 1u) % kStages;
              stph ^= (st == 0);
            }
            continue;
          }
          mbar_wait_cluster(a_full_peer, it & 1);
        }
        for (int c = 0; c < nchunks; ++c, ++cc) {
          mbar_wait(&b_full[st], stph);
          if constexpr (kPair) mbar_wait_cluster(&b_full_peer[st], stph);
          const uint32_t cph = cc & 1u;
          const uint32_t bh = B_hi + st * kStage;
          const uint32_t bxh = Bx_hi + st * kBz, bxl = Bx_lo + st * kBz;
          uint64_t* const accf = &acc_full[(c & 1) * NBUF];
#pragma unroll
          for (int t = 0; t < TPC; ++t) {
            const uint32_t d_t = tmem + t * ACC_STRIDE;
            const uint32_t ah = A_hi + t * kATile, al = A_lo + t * kATile, al8 = A_l8 + t * kATile;
            if constexpr (kPair) {  // (arrivals come from both CTAs' epilogue warps)
              mbar_wait_cluster(&acc_empty[t], cph ^ 1u);
              mbar_wait_cluster(&e_full[t], cph);
            } else {
              mbar_wait(&acc_empty[t], cph ^ 1u);
              mbar_wait(&e_full[t], cph);
            }
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
              for (int s2 = 0; s2 < (int)kK16; ++s2) mmaH(d_t, mk(ah + s2 * kAStep), mk(bh + s2 * kBStep), idN, s2 != 0);
              if constexpr (kMix) {
                mmaH(d_t, mk(E_mx + t * kExtBuf), mk(bh + kK16 * kBStep), idN, 1);            // ext: hi-plane chunks kKx, kKx + 1
                constexpr uint32_t b8h = ((kKx + 2) * kBLbo) >> 4, b8l = ((kKx + 2 + kKx / 2) * kBLbo) >> 4;  // e5m2(hi) / e5m2(lo) planes
#pragma unroll
                for (int s8 = 0; s8 < (int)kK32; ++s8) mmaQ(d_t, mk(al + s8 * kAStep), mk(bh + b8l + s8 * kBStep), idN8, 1);
#pragma unroll
                for (int s8 = 0; s8 < (int)kK32; ++s8) mmaQ(d_t, mk(al8 + s8 * kAStep), mk(bh + b8h + s8 * kBStep), idN8, 1);
              } else {
                constexpr uint32_t blo = ((kKx + 1) * kBLbo) >> 4;                                // lo plane
                mmaH(d_t, mk(E_hi + t * kEz), mk(bxh), idN, 1);
#pragma unroll
                for (int s2 = 0; s2 < (int)kK16; ++s2) mmaH(d_t, mk(ah + s2 * kAStep), mk(bh + blo + s2 * kBStep), idN, 1);
                mmaH(d_t, mk(E_hi + t * kEz), mk(bxl), idN, 1);
#pragma unroll
                for (int s2 = 0; s2 < (int)kK16; ++s2) mmaH(d_t, mk(al + s2 * kAStep), mk(bh + s2 * kBStep), idN, 1);
                mmaH(d_t, mk(E_lo + t * kEz), mk(bxh), idN, 1);
              }
              commit(&accf[t]);
            }
            __syncwarp();
          }
          if (elect_one()) commit(&b_empty[st]);
          __syncwarp();
          st = (st + 1u) % kStages;
          stph ^= (st == 0);
        }
        if (elect_one()) commit(a_empty);
        __syncwarp();
      }
    } else
    {
      const int nrow_c = kD128 ? 144 : g.nrow, a_plane_c = kD128 ? 16 * TM * 16 : g.a_plane, a_tile_c = kD128 ? 32 * TM * 16 : g.a_tile;
      const int stage_bytes_c = kD128 ? 10 * 144 * 16 : g.stage_bytes, stages_c = kD128 ? 3 : g.stages;
      const uint32_t idN = idesc_f16(TM, nrow_c), id16 = idesc_f16(TM, 16), idN8 = idesc_e5m2(TM, nrow_c);
      const uint32_t zaddr = smem_u32(sZ);
      const uint32_t a_lbo = TM * 16, b_lbo = nrow_c * 16, l_lbo = 16 * 16;
      const uint32_t a_step = (2 * a_lbo) >> 4, b_step = (2 * b_lbo) >> 4, l_step = (2 * l_lbo) >> 4;
      const uint32_t hi_word = (uint32_t)(smem_desc(0, 0, 128) >> 32);  // SBO = 128 B, version 1, no swizzle
      auto lo_of = [](uint32_t addr, uint32_t lbo) { return ((addr >> 4) & 0x3FFFu) | (((lbo >> 4) & 0x3FFFu) << 16); };
      auto mk = [&](uint32_t lo) { return ((uint64_t)hi_word << 32) | lo; };
      const uint32_t sa0 = smem_u32(sA), sb0 = smem_u32(sB), se0 = smem_u32(sE);
      // low words for index 0 and the per-index deltas (all linear in the tile / buffer / stage index)
      const uint32_t A_hi0 = lo_of(sa0, a_lbo), A_lo0 = lo_of(sa0 + a_plane_c, a_lbo), A_d = (uint32_t)a_tile_c >> 4;
      const uint32_t E_hi0 = lo_of(se0, zaddr - se0), E_lo0 = lo_of(se0 + TM * 16, zaddr - se0 - TM * 16);
      const uint32_t E_d = (uint32_t)((2 * TM * 16) >> 4) - ((uint32_t)((2 * TM * 16) >> 4) << 16);  // wraps: LBO shrinks as the start grows
      const uint32_t sbytes = (uint32_t)stage_bytes_c >> 4;
      const uint32_t B_d = sbytes, Bz_d = sbytes - (sbytes << 16);  // plain / zero-aliased-LBO descriptors, per stage
      const int kcp = kD128 ? 4 : g.kc_part, ks_part = kcp / 2;
      const bool split = g.split != 0, mix = g.mix != 0;
      // stage-0 low words.  Inside a stage: hi plane (nkc x k-chunks) then the lo section; nkc = kcp (+1 or, mix, +2 in the last part)
      const uint32_t B_hi0 = lo_of(sb0, b_lbo);
      const uint32_t lo_off_mid = (uint32_t)kcp * b_lbo, lo_off_last = (uint32_t)(kcp + 1 + g.mix) * b_lbo;  // byte offset of the lo section
      // mix: e5m2 planes.  A tile = [hi fp16 | e5m2(hi) | e5m2(lo)], a K = 32 step = two 16-byte k-chunks = a_step again;
      // B lo section = [e5m2(hi) : kcp/2 k-chunks | e5m2(lo) : kcp/2 k-chunks].  The ext step is one fp16 MMA over two real
      // k-chunks (A_ext buffer = [chunk 0 | chunk 1], B ext chunks kcp, kcp+1 of the hi plane): plain LBOs, no zero alias.
      const int ks8 = kcp / 4;
      const uint32_t A8_0 = lo_of(sa0 + a_plane_c, a_lbo), A8l_0 = lo_of(sa0 + a_plane_c + a_plane_c / 2, a_lbo);
      const uint32_t Em_0 = lo_of(se0, TM * 16), Em_d = (uint32_t)((2 * TM * 16) >> 4);
      const uint32_t Bem_0 = lo_of(sb0 + kcp * b_lbo, b_lbo);
      const uint32_t bex = sb0 + kcp * b_lbo;                                                       // ext k-chunk, hi plane (last part)
      const uint32_t Be_hi0 = lo_of(bex, zaddr - bex);
      const uint32_t belx = sb0 + lo_off_last + kcp * b_lbo;                                        // ext k-chunk, lo plane (split)
      const uint32_t Be_lo0 = lo_of(belx, zaddr - belx);
      const uint32_t bha = sb0 + g.aux0 * 16;                                                       // S/L rows inside the hi plane
      const uint32_t Ba_hi0 = lo_of(bha, b_lbo), Bae_hi0 = lo_of(bha + kcp * b_lbo, zaddr - (bha + kcp * b_lbo));
      const uint32_t baelx = sb0 + lo_off_last + kcp * l_lbo;                                       // ext k-chunk of the 16-row lo image
      const uint32_t Bae_lo0 = lo_of(baelx, zaddr - baelx);
      uint32_t it_n = 0, n = 0, st = 0, stph = 0;
      for (int64_t item = blockIdx.x; item < A.n_items; item += gridDim.x) {
        const int u = (int)(item / A.groups);
        if (!user_in_pass(A.gate, sc.use_mix, (int)(A.users.offsets[u + 1] - A.users.offsets[u]))) continue;
        const uint32_t it = it_n++;
        const int nchunks = __shfl_sync(0xffffffffu, user_chunks(A.users.offsets, u, kHch, cb0, A.max_chunks, hsplit), 0);
        mbar_wait(a_full, it & 1);
        for (int c = 0; c < nchunks; ++c, n += (uint32_t)tpc) {
          const int kp_m = kSinglePart ? 1 : (kD128 ? 4 : g.kp);
#pragma unroll
          for (int pp = 0; pp < (kD128 ? 4 : kp_m); ++pp) {
            const bool lastp = kSinglePart ? true : pp == kp_m - 1;
            mbar_wait(&b_full[st], stph);
            const uint32_t lo_off = lastp ? lo_off_last : lo_off_mid;
            const uint32_t bh = B_hi0 + st * B_d;                               // hi plane, x k-chunks of this part
            const uint32_t bl = lo_of(sb0 + lo_off, b_lbo) + st * B_d;          // lo plane (split)
            const uint32_t bal = lo_of(sb0 + lo_off, l_lbo) + st * B_d;         // 16-row lo image of the S/L rows (fast)
            const uint32_t bah = Ba_hi0 + st * B_d;
            const uint32_t beh = Be_hi0 + st * Bz_d, bel = Be_lo0 + st * Bz_d;
            const uint32_t baeh = Bae_hi0 + st * Bz_d, bael = Bae_lo0 + st * Bz_d;
            const uint32_t ka = (uint32_t)(pp * ks_part) * a_step;              // this part's first K-step inside the A tile
            const uint32_t ka8 = (uint32_t)(pp * ks8) * a_step;                 // same inside the e5m2 planes (K = 32 steps)
            const uint32_t b8h = bl, b8l = bl + (uint32_t)((kcp / 2) * b_lbo >> 4);  // mix: e5m2(hi) plane, e5m2(lo) plane
            const uint32_t bem = Bem_0 + st * B_d;
#pragma unroll
            for (int t = 0; t < TPC; ++t) {
              if (t >= tpc) break;
              const uint32_t nn = n + (uint32_t)t, buf = nn % NBUF, ph = (nn / NBUF) & 1u;
              const uint32_t ah = A_hi0 + t * A_d + ka, al = A_lo0 + t * A_d + ka;
              const uint32_t eh = E_hi0 + buf * E_d, el = E_lo0 + buf * E_d;
              const uint32_t d_t = tmem + buf * ACC_STRIDE, d_aux = d_t + g.aux0;
              if (pp == 0) mbar_wait(&acc_empty[buf], ph ^ 1);
              if (lastp) mbar_wait(&e_full[buf], ph);
              tc_fence_after();
              if (elect_one()) {
                // pass 1: A_hi x B_hi over all rows
                for (int s2 = 0; s2 < ks_part; ++s2) mma_f16(d_t, mk(ah + s2 * a_step), mk(bh + s2 * b_step), idN, (pp | s2) != 0);
                if (mix) {
                  // ext step with its inner hi/lo split, then the e5m2 corrections: e5m2(A_hi) x e5m2(B_lo) ; e5m2(A_lo) x e5m2(B_hi)
                  if (lastp) mma_f16(d_t, mk(Em_0 + buf * Em_d), mk(bem), idN, 1);
                  const uint32_t a8h = A8_0 + t * A_d + ka8, a8l = A8l_0 + t * A_d + ka8;
                  for (int s8 = 0; s8 < ks8; ++s8) mma_f8(d_t, mk(a8h + s8 * a_step), mk(b8l + s8 * b_step), idN8, 1);
                  for (int s8 = 0; s8 < ks8; ++s8) mma_f8(d_t, mk(a8l + s8 * a_step), mk(b8h + s8 * b_step), idN8, 1);
                } else if (split) {
                  if (lastp) mma_f16(d_t, mk(eh), mk(beh), idN, 1);
                  // pass 2: A_hi x B_lo ; pass 3: A_lo x B_hi
                  for (int s2 = 0; s2 < ks_part; ++s2) mma_f16(d_t, mk(ah + s2 * a_step), mk(bl + s2 * b_step), idN, 1);
                  if (lastp) mma_f16(d_t, mk(eh), mk(bel), idN, 1);
                  for (int s2 = 0; s2 < ks_part; ++s2) mma_f16(d_t, mk(al + s2 * a_step), mk(bh + s2 * b_step), idN, 1);
                  if (lastp) mma_f16(d_t, mk(el), mk(beh), idN, 1);
                } else {
                  if (lastp) mma_f16(d_t, mk(eh), mk(beh), idN, 1);
                  // S/L rows only (N = 16 at column aux0): A_hi x B_lo(aux rows) ; A_lo x B_hi(aux rows)
                  for (int s2 = 0; s2 < ks_part; ++s2) mma_f16(d_aux, mk(ah + s2 * a_step), mk(bal + s2 * l_step), id16, 1);
                  if (lastp) mma_f16(d_aux, mk(eh), mk(bael), id16, 1);
                  for (int s2 = 0; s2 < ks_part; ++s2) mma_f16(d_aux, mk(al + s2 * a_step), mk(bah + s2 * b_step), id16, 1);
                  if (lastp) mma_f16(d_aux, mk(el), mk(baeh), id16, 1);
                }
                if (lastp) mma_commit(&acc_full[(c & 1) * NBUF + buf]);
              }
              __syncwarp();
            }
            if (elect_one()) mma_commit(&b_empty[st]);
            __syncwarp();
            if (++st == (uint32_t)stages_c) {
              st = 0;
              stph ^= 1;
            }
          }
        }
        if (elect_one()) mma_commit(a_empty);
        __syncwarp();
      }
    }
  } else {
    // =================================================== epilogue warps ============================================
    // Two groups of 8 warps alternate history chunks (group = parity of the chunk index), so one group's TMEM-load /
    // exp latencies hide behind the other's FADD stream.  Within a group: lane quarter = warp % 4 (the TMEM
    // lanes a warp may touch), history slot = (warp / 4) % 2.
    const int egrp = warp >> 3;
    const int qd = warp & 3, hs = (warp >> 2) & 1;
    const int r = qd * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(qd * 32) << 16;
    // sigmoid(z) = 1 / (1 + 2^(-log2e * z)): -log2e and the input scale (100 / 1000) are folded into the 2x2 layer
    const float nl2e = -1.4426950408889634f, dsc = A.p.dist_scale * nl2e;
    const float w00 = g.lanes ? __ldg(A.p.dist_w + 0) * dsc : 0.f, w01 = g.lanes ? __ldg(A.p.dist_w + 1) * dsc : 0.f;
    const float w10 = g.lanes ? __ldg(A.p.dist_w + 2) * dsc : 0.f, w11 = g.lanes ? __ldg(A.p.dist_w + 3) * dsc : 0.f;
    const float bd0 = g.lanes ? __ldg(A.p.dist_b + 0) * nl2e : 0.f, bd1 = g.lanes ? __ldg(A.p.dist_b + 1) * nl2e : 0.f;
    const float beta = A.p.beta;
    const bool geo = g.lanes || g.km;
    // NAIS_DIST_KM (model.py:497-504, the reference only ever reads bucket 0): the coefficient, summed in the FP32 kernel's order
    float ckm = 0.f;
    if constexpr (!kFastEpi)
      if (g.km)
        for (int d = 0; d < g.D; ++d) ckm += __ldg(A.p.dist_embed + d);
    const int npos = sc.npos, hid = g.hid;
    constexpr int hch = kHch;
    const int ncols = hch == 2 ? hid : hid / 2;   // accumulator columns this thread sums per step
    const int col0 = hs * ncols;                  // hch = 2: slot hs's hidden units; hch = 1: this warp's half of them
    // hidden-unit index (in permuted order, positive v first) of column col0: with hsplit = 2 this group's chunks hold half `egrp`
    const int kidx0 = hch == 2 ? 0 : col0 + (hsplit == 2 ? egrp * hid : 0);
    auto div_tpc = [&](int x) { return x / tpc; };  // tpc is a compile-time constant: mul-shift, not a runtime division
    uint32_t n0 = 0;  // global index of the current item's first step (same sequence as the MMA warp)
    uint32_t phbits = 0;  // phase parity of this group's acc_full barrier, one bit per buffer
    // fast epilogue: one parity bit (every buffer completes once per own chunk), folded constants, sign split of the columns
    uint32_t fph = 0;
    const float c_a2 = sc.inv_sigma * 1.4426950408889634f, inv_sAe = 1.f / sc.sAe;
    const float bd0s = bd0 - log2f(sc.sAe), bd1s = bd1 - log2f(sc.sAe);
    const int nposb = npos >> 4, nposm = npos & 15;
    const float* sgn_mixed = xch;  // [16] +-1 of the one 16-column block that holds both signs (xch is unused when hch == 2)

    auto arrive_mma = [&](uint64_t* bar) {  // a barrier the MMA issuer waits on: rank 0's in a pair
      if constexpr (kPair) mbar_arrive_cluster(bar, 0);
      else mbar_arrive(bar);
    };
    for (int64_t item = item0; item < A.n_items; item += item_step) {
      const int u = (int)(item / groups_it), grp = kPair ? 2 * (int)(item % groups_it) + (int)crank : (int)(item % groups_it);
      const int64_t hb = A.users.offsets[u];
      const int H = (int)(A.users.offsets[u + 1] - hb);
      if (!user_in_pass(A.gate, sc.use_mix, H)) continue;
      const int nchunks = user_chunks(A.users.offsets, u, hch, cb0, A.max_chunks, hsplit);
      const int nsteps = nchunks * tpc;
      // stage this user's history ids / coords (previous item's readers are past their last epi_bar)
      epi_bar();
      for (int i = tid; i < H && i < HMETA; i += EPI_THREADS) {
        hm_id[i] = __ldg(A.users.items + hb + i);
        hm_la[i] = (geo || kGeo) ? __ldg(A.users.coords + 2 * (hb + i)) : 0.f;
        hm_lo[i] = (geo || kGeo) ? __ldg(A.users.coords + 2 * (hb + i) + 1) : 0.f;
        if constexpr (!kFastEpi)
          if (g.km || kGeo) hm_cos[i] = cosf((A.cat.center_lat + hm_la[i]) * 0.017453292519943295f);
      }
      // candidates of this thread's row in the item's tiles
      float clat[TPC], clon[TPC], ccos[TPC], sumE[TPC], sumES[TPC], sumL[TPC];
      int64_t jid[TPC];
      bool excl[TPC];
#pragma unroll
      for (int t = 0; t < TPC; ++t) {
        jid[t] = t < tpc ? A.poi_begin + ((int64_t)grp * tpc + t) * TM + r : A.poi_end;
        const bool v = jid[t] < A.poi_end;
        clat[t] = (v && (geo || kGeo)) ? __ldg(A.cat.coords + 2 * (jid[t] - A.cat.row_base)) : 0.f;
        clon[t] = (v && (geo || kGeo)) ? __ldg(A.cat.coords + 2 * (jid[t] - A.cat.row_base) + 1) : 0.f;
        ccos[t] = 1.f;
        if constexpr (!kFastEpi)
          if (g.km || kGeo) ccos[t] = cosf((A.cat.center_lat + clat[t]) * 0.017453292519943295f);
        sumE[t] = 0.f;
        sumES[t] = 0.f;
        sumL[t] = 0.f;
        excl[t] = false;
      }
      epi_bar();
      if constexpr (kFastEpi) {
        // ---- specialised step loop: hid == 64, two history items per step, tpc == NBUF == 3 -----------------------------
        // Every step index is then (chunk, t) with buffer == t, so the t loop unrolls with compile-time TMEM / A_ext
        // addresses, the per-chunk history lookups leave the step body, and this group's acc_full parity is one bit that
        // flips once per own chunk.  ~150 issue slots per warp-step instead of ~340 (the MIX mode is epilogue-issue bound).
        const unsigned char* ebase = sE + r * 16 + hs * 4;
        // A_ext of (chunk pc, tile t): 2 sigmoids -> hi/lo halves.  sAe / (1 + 2^z) = 1 / (1/sAe + 2^(z - log2 sAe))
        auto produce_f = [&](int t, bool on, float hla, float hlo, float cla, float clo) {
          float g0 = 0.f, g1 = 0.f;
          if (on) {
            const float l0 = fabsf(cla - hla), l1 = fabsf(clo - hlo);
            const float z0 = fmaf(l1, w01, fmaf(l0, w00, bd0s)), z1 = fmaf(l1, w11, fmaf(l0, w10, bd1s));
            g0 = rcp_approx(ex2_approx(z0) + inv_sAe);
            g1 = rcp_approx(ex2_approx(z1) + inv_sAe);
          }
          const __half2 hi2 = __floats2half2_rn(g0, g1);
          const float2 hif = __half22float2(hi2);
          const __half2 lo2 = __floats2half2_rn(g0 - hif.x, g1 - hif.y);
          unsigned char* eb = const_cast<unsigned char*>(ebase) + t * (2 * TM * 16);
          *reinterpret_cast<__half2*>(eb) = hi2;
          *reinterpret_cast<__half2*>(eb + TM * 16) = lo2;
          if (g.mix) *reinterpret_cast<__half2*>(eb + TM * 16 + 8) = hi2;
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) arrive_mma(&e_full[t]);
        };
        auto hist_coords = [&](int h, float& la, float& lo) {
          if (h < HMETA) {
            la = hm_la[h];
            lo = hm_lo[h];
          } else {
            la = __ldg(A.users.coords + 2 * (hb + h));
            lo = __ldg(A.users.coords + 2 * (hb + h) + 1);
          }
        };
        int jt[TPC];
#pragma unroll
        for (int t = 0; t < TPC; ++t) jt[t] = jid[t] < A.poi_end ? (int)jid[t] : -2;
        if (egrp == 0 && nchunks > 0) {  // prologue: chunk 0's A_ext
          const bool on = g.lanes && hs < H;
          float la = 0.f, lo = 0.f;
          if (on) hist_coords(hs, la, lo);
#pragma unroll
          for (int t = 0; t < TPC; ++t) produce_f(t, on, la, lo, clat[t], clon[t]);
        }
        const uint32_t tb_main = tmem + lane_addr + (uint32_t)(hs * kS), tb_aux = tmem + lane_addr + (uint32_t)(2 * kS) + (uint32_t)(2 * hs);
        for (int c = egrp; c < nchunks; c += 2) {
          const int h = 2 * c + hs;
          const bool hvalid = h < H;
          int hist_id = -1;
          if (hvalid) hist_id = h < HMETA ? hm_id[h] : __ldg(A.users.items + hb + h);
          const bool pn = c + 1 < nchunks;            // this group refills the A_ext buffers for the other group's next chunk
          const bool pon = pn && g.lanes && (h + 2 < H);
          float nla = 0.f, nlo = 0.f;
          if (pon) hist_coords(h + 2, nla, nlo);
#pragma unroll
          for (int t = 0; t < TPC; ++t) {
            mbar_wait(&acc_full[egrp * NBUF + t], fph);
            tc_fence_after();
            // The MMA issuer needs two things from this step before it may start step + 3: the accumulator drained
            // (acc_empty) and the next A_ext (e_full).  Issue the first TMEM loads, build A_ext while they are in flight,
            // and hand the accumulator back as soon as its last block is in registers.
            uint32_t aux[2], va[16], vb[16];
            float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
            auto blk = [&](const uint32_t(&v)[16], int b) {
              if (b < nposb) {
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                  p0 += fabsf(__uint_as_float(v[i]));
                  p1 += fabsf(__uint_as_float(v[i + 1]));
                  p2 += fabsf(__uint_as_float(v[i + 2]));
                  p3 += fabsf(__uint_as_float(v[i + 3]));
                }
              } else if (b > nposb || nposm == 0) {
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                  q0 += fabsf(__uint_as_float(v[i]));
                  q1 += fabsf(__uint_as_float(v[i + 1]));
                  q2 += fabsf(__uint_as_float(v[i + 2]));
                  q3 += fabsf(__uint_as_float(v[i + 3]));
                }
              } else {  // the one block that holds both signs: signed FFMA with the +-1 vector kept in shared memory
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                  const float4 sg = *reinterpret_cast<const float4*>(sgn_mixed + i);
                  p0 = fmaf(fabsf(__uint_as_float(v[i])), sg.x, p0);
                  p1 = fmaf(fabsf(__uint_as_float(v[i + 1])), sg.y, p1);
                  p2 = fmaf(fabsf(__uint_as_float(v[i + 2])), sg.z, p2);
                  p3 = fmaf(fabsf(__uint_as_float(v[i + 3])), sg.w, p3);
                }
              }
            };
            tmem_ld2(tb_aux + t * ACC_STRIDE, aux);
            tmem_ld16(tb_main + t * ACC_STRIDE, va);
            tmem_ld16(tb_main + t * ACC_STRIDE + 16, vb);
            if (pn) produce_f(t, pon, nla, nlo, clat[t], clon[t]);
            tmem_wait_ld16(va);
            tmem_wait_ld16(vb);
            if constexpr (kS == 64) {
              blk(va, 0);
              tmem_ld16(tb_main + t * ACC_STRIDE + 32, va);
              blk(vb, 1);
              tmem_ld16(tb_main + t * ACC_STRIDE + 48, vb);
              tmem_wait_ld16(va);
              tmem_wait_ld16(vb);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) arrive_mma(&acc_empty[t]);
            if constexpr (kS == 64) {
              blk(va, 2);
              blk(vb, 3);
            } else {  // hid = 32: the slot's 32 columns are already in registers
              blk(va, 0);
              blk(vb, 1);
            }
            const float asum = ((p0 + p1) + (p2 + p3)) - ((q0 + q1) + (q2 + q3));
            const float S = __uint_as_float(aux[0]) * sc.inv_s;
            const float a2 = (__uint_as_float(aux[1]) + asum) * c_a2;
            const bool same = hist_id == jt[t];  // (hist_id is -1 when this slot is past the end of the history)
            const float e = (hvalid && !same) ? ex2_approx(a2) : 0.f;
            sumE[t] += e;
            sumES[t] = fmaf(e, S, sumES[t]);
            excl[t] = excl[t] || (hvalid && same);
          }
          fph ^= 1u;
        }
      } else {
        // writes the g lanes of local step m into A_ext buffer (n0 + m) % NBUF
        auto produce = [&](int m) {
          const int pc = div_tpc(m), pt = m - pc * tpc;
          const uint32_t pbuf = (n0 + (uint32_t)m) % NBUF;
          const int h = hch == 2 ? 2 * pc + hs : pc / hsplit;
          float g0 = 0.f, g1 = 0.f;
          if (g.lanes && h < H && (hch == 2 || hs == 0)) {
            float hla, hlo;
            if (h < HMETA) {
              hla = hm_la[h];
              hlo = hm_lo[h];
            } else {
              hla = __ldg(A.users.coords + 2 * (hb + h));
              hlo = __ldg(A.users.coords + 2 * (hb + h) + 1);
            }
            const float ct_la = pt == 0 ? clat[0] : (pt == 1 ? clat[1] : clat[2]);
            const float ct_lo = pt == 0 ? clon[0] : (pt == 1 ? clon[1] : clon[2]);
            const float l0 = fabsf(ct_la - hla), l1 = fabsf(ct_lo - hlo);
            const float z0 = fmaf(l1, w01, fmaf(l0, w00, bd0)), z1 = fmaf(l1, w11, fmaf(l0, w10, bd1));
            g0 = __fdividef(sc.sAe, 1.f + exp2f(z0));
            g1 = __fdividef(sc.sAe, 1.f + exp2f(z1));
          }
          const __half2 hi2 = __floats2half2_rn(g0, g1);
          const float2 hif = __half22float2(hi2);
          const __half2 lo2 = __floats2half2_rn(g0 - hif.x, g1 - hif.y);
          if (hch == 2 || hs == 0) {
            // split / fast: [hi plane | lo plane], slots 2hs, 2hs+1.  mix: [k-chunk 0 | k-chunk 1]: chunk 0 slots 2hs.. = hi,
            // chunk 1 slots 2hs.. = lo and slots 4+2hs.. = hi again (pairs with the lo weights)
            unsigned char* eb = sE + (size_t)pbuf * 2 * TM * 16 + r * 16 + hs * 4;
            *reinterpret_cast<__half2*>(eb) = hi2;
            *reinterpret_cast<__half2*>(eb + TM * 16) = lo2;
            if (g.mix) *reinterpret_cast<__half2*>(eb + TM * 16 + 8) = hi2;
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&e_full[pbuf]);
        };
        // Group g owns the history chunks of parity g (a fixed set of h per partial sum, whatever tile / shard / item
        // order a candidate is scored in: results are bit-identical between a sharded and an unsharded catalogue).
        // prologue: the first NBUF steps (= chunk 0) are produced by its owner, group 0
        if (egrp == 0)
          for (int m = 0; m < NBUF && m < nsteps; ++m) produce(m);

        // steps of this group's chunks: (c, t) for c = egrp, egrp + 2, ... and t = 0 .. tpc-1
        for (int c = egrp, t = 0; c < nchunks; (t + 1 == tpc) ? (t = 0, c += 2) : ++t) {
          const int ls = c * tpc + t;
          const uint32_t n = n0 + (uint32_t)ls;
          const uint32_t buf = n % NBUF;
          const int h = hch == 2 ? 2 * c + hs : c / hsplit;
          int hist_id = -1;
          if (h < H) hist_id = h < HMETA ? hm_id[h] : __ldg(A.users.items + hb + h);
          mbar_wait(&acc_full[egrp * NBUF + buf], (phbits >> buf) & 1u);
          phbits ^= 1u << buf;
          tc_fence_after();
          // MMA(n) is complete, so its A_ext buffer is free: refill it for step ls + NBUF (keeps the MMA queue fed)
          if (ls + NBUF < nsteps) produce(ls + NBUF);
          // ---- TMEM -> registers, 32 columns at a time.  Loads and their wait are kept back to back: the destination
          // registers are written asynchronously, so no other code may sit between a tcgen05.ld and its wait::ld (the
          // other epilogue group hides the latency instead).
          const uint32_t t_main = tmem + lane_addr + buf * ACC_STRIDE + col0;
          uint32_t aux[2], v[32];
          float accp = 0.f, accn = 0.f;
          tmem_ld2(tmem + lane_addr + buf * ACC_STRIDE + g.aux0 + (hch == 2 ? 2 * hs : 0), aux);
          if (ncols >= 32) tmem_ld32(t_main, v);
          else tmem_ld16(t_main, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
          tmem_wait_ld();
          auto absum = [&](int c0, int cnt) {  // columns [c0, c0+cnt) of this thread's slice are in v[0..cnt)
  #pragma unroll
            for (int g16 = 0; g16 < 32; g16 += 16) {
              if (g16 < cnt) {
                const int cc = kidx0 + c0 + g16;
                if (cc + 16 <= npos || cc >= npos) {
                  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  #pragma unroll
                  for (int i = 0; i < 16; i += 4) {
                    s0 += fabsf(__uint_as_float(v[g16 + i]));
                    s1 += fabsf(__uint_as_float(v[g16 + i + 1]));
                    s2 += fabsf(__uint_as_float(v[g16 + i + 2]));
                    s3 += fabsf(__uint_as_float(v[g16 + i + 3]));
                  }
                  const float ssum = (s0 + s1) + (s2 + s3);
                  if (cc >= npos) accn += ssum;
                  else accp += ssum;
                } else {
  #pragma unroll
                  for (int i = 0; i < 16; ++i) {
                    const float av = fabsf(__uint_as_float(v[g16 + i]));
                    if (cc + i < npos) accp += av;
                    else accn += av;
                  }
                }
              }
            }
          };
          absum(0, ncols >= 32 ? 32 : 16);
          if (ncols > 32) {
            if (ncols >= 64) tmem_ld32(t_main + 32, v);
            else tmem_ld16(t_main + 32, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
            tmem_wait_ld();
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
          if (ncols > 32) absum(32, ncols >= 64 ? 32 : 16);
          float asum = accp - accn;
          if (hch == 1 && hsplit == 1) {
            // the other half of this cell's hidden units was summed by the partner warp (same lane quarter)
            float* slot = xch + ((ls & 1) * 2 + egrp) * TM + r;
            if (hs == 1) *slot = asum;
            asm volatile("bar.sync %0, 64;" ::"r"(2 + egrp * 4 + qd) : "memory");
            if (hs == 0) asum += *slot;
          } else if (hch == 1) {
            // hid = 256: this cell's 256 hidden units sit in TWO consecutive chunks (= the two groups, same t) x two warps each:
            // three senders, one 128-thread barrier per lane quarter, group 0 / hs 0 adds them in a fixed order
            const int par = ((c >> 1) * tpc + t) & 1;
            float* slots = xch + par * 3 * TM + r;
            const int sender = egrp * 2 + hs - 1;  // (0,1) -> 0, (1,0) -> 1, (1,1) -> 2
            if (sender >= 0) slots[sender * TM] = asum;
            asm volatile("bar.sync %0, 128;" ::"r"(10 + qd) : "memory");
            if (sender < 0) asum = ((asum + slots[0]) + slots[TM]) + slots[2 * TM];
          }
          const float S = __uint_as_float(aux[0]) * sc.inv_s;
          const float a = (__uint_as_float(aux[1]) + asum) * sc.inv_sigma;
          if (h < H && (hch == 2 || hs == 0) && (hsplit == 1 || egrp == 0)) {
            const int64_t j = t == 0 ? jid[0] : (t == 1 ? jid[1] : jid[2]);
            if constexpr (kGeo) {  // every cell once, the h = j cell included
              float hla, hlo, hcs;
              if (h < HMETA) {
                hla = hm_la[h];
                hlo = hm_lo[h];
                hcs = hm_cos[h];
              } else {
                hla = __ldg(A.users.coords + 2 * (hb + h));
                hlo = __ldg(A.users.coords + 2 * (hb + h) + 1);
                hcs = cosf((A.cat.center_lat + hla) * 0.017453292519943295f);
              }
              const float cla = t == 0 ? clat[0] : (t == 1 ? clat[1] : clat[2]), clo = t == 0 ? clon[0] : (t == 1 ? clon[1] : clon[2]);
              const float ccs = t == 0 ? ccos[0] : (t == 1 ? ccos[1] : ccos[2]);
              const float lt = powerlaw_log_term(dist_km_f(cla, clo, hla, hlo, ccs, hcs), A.geo.ln_a, A.geo.b);
              if (t == 0) sumL[0] += lt;
              else if (t == 1) sumL[1] += lt;
              else sumL[2] += lt;
            }
            if ((int64_t)hist_id != j) {
              float a_km = a;
              if (g.km) {  // logit += dist_km * coefficient (haversine from centred coordinates, as the FP32 kernel forms it)
                float hla, hlo, hcs;
                if (h < HMETA) {
                  hla = hm_la[h];
                  hlo = hm_lo[h];
                  hcs = hm_cos[h];
                } else {
                  hla = __ldg(A.users.coords + 2 * (hb + h));
                  hlo = __ldg(A.users.coords + 2 * (hb + h) + 1);
                  hcs = cosf((A.cat.center_lat + hla) * 0.017453292519943295f);
                }
                const float cla = t == 0 ? clat[0] : (t == 1 ? clat[1] : clat[2]), clo = t == 0 ? clon[0] : (t == 1 ? clon[1] : clon[2]);
                const float ccs = t == 0 ? ccos[0] : (t == 1 ? ccos[1] : ccos[2]);
                const float km = dist_km_f(cla, clo, hla, hlo, ccs, hcs);
                a_km = fmaf(km, ckm, a);
              }
              const float e = g.km ? expf(a_km) : __expf(a);
              if (t == 0) { sumE[0] += e; sumES[0] = fmaf(e, S, sumES[0]); }
              else if (t == 1) { sumE[1] += e; sumES[1] = fmaf(e, S, sumES[1]); }
              else { sumE[2] += e; sumES[2] = fmaf(e, S, sumES[2]); }
            } else {
              if (t == 0) excl[0] = true;
              else if (t == 1) excl[1] = true;
              else excl[2] = true;
            }
          }
        }
        n0 += (uint32_t)nsteps;
      }
      // ---- item epilogue: combine the 4 partial states (2 groups x 2 history slots), score, block top-k --------------
      const int part = egrp * 2 + hs;  // partial 0 is the combiner
      const bool small_k = A.k <= 32;
      unsigned long long kreg[TPC];
      if (!kSinglePart) epi_bar();  // every group is past its last step: all MMAs are complete, A_ext + zero may hold `comb`
      if (part != 0) {
#pragma unroll
        for (int t2 = 0; t2 < kCombT; ++t2) {
          comb[((part - 1) * kCombA + 0) * kCombT * TM + t2 * TM + r] = sumE[t2];
          comb[((part - 1) * kCombA + 1) * kCombT * TM + t2 * TM + r] = sumES[t2];
          comb[((part - 1) * kCombA + 2) * kCombT * TM + t2 * TM + r] = excl[t2] ? 1.f : 0.f;
          if constexpr (kGeo) comb[((part - 1) * kCombA + 3) * kCombT * TM + t2 * TM + r] = sumL[t2];
        }
      }
      epi_bar();
      if (part == 0) {
#pragma unroll
        for (int t2 = 0; t2 < TPC; ++t2) {
          float E = sumE[t2], ES = sumES[t2], Lg = sumL[t2];
          bool ex = excl[t2];
          if (t2 < kCombT) {  // (kCombT < TPC: tile t2 does not exist in this kernel)
#pragma unroll
            for (int q = 0; q < 3; ++q) {
              E += comb[(q * kCombA + 0) * kCombT * TM + t2 * TM + r];
              ES += comb[(q * kCombA + 1) * kCombT * TM + t2 * TM + r];
              ex = ex || comb[(q * kCombA + 2) * kCombT * TM + t2 * TM + r] != 0.f;
              if constexpr (kGeo) Lg += comb[(q * kCombA + 3) * kCombT * TM + t2 * TM + r];
            }
          }
          float score = ES / powf(E, beta);
          const bool valid = jid[t2] < A.poi_end;
          if (A.score_in && valid) score += A.score_in[(size_t)u * (A.poi_end - A.poi_begin) + (jid[t2] - A.poi_begin)];
          if constexpr (kGeo) score = geo_mixed(score, Lg, __ldg(A.geo.user_logmax + u), A.geo.alpha);
          if (A.all_scores && valid) A.all_scores[(size_t)u * (A.poi_end - A.poi_begin) + (jid[t2] - A.poi_begin)] = score;
          kreg[t2] = (valid && !(A.exclude && ex)) ? make_key(score, (int)jid[t2]) : 0ull;
          if (!small_k) keys[t2 * TM + r] = kreg[t2];
        }
        if (small_k) {
          // k <= 32: the item's 384 keys live in the registers of warps 0-3.  Sort each 32-key row with warp shuffles,
          // fold the rows keeping the best 32 (max of one sorted row against the other reversed is bitonic and holds the
          // top 32 of both), park 4 x 32 candidates in shared memory; warp 0 folds those after the barrier.  Same total
          // order as the 512-key sort below (keys are unique except the 0 = "no entry" filler), 2 barriers instead of 45.
          unsigned long long a = warp_sort_desc(kreg[0], lane);
          a = warp_fold_top32(a, warp_sort_desc(kreg[1], lane), lane);
          a = warp_fold_top32(a, warp_sort_desc(kreg[2], lane), lane);
          keys[r] = a;
        } else {
          for (int i = TPC * TM + r; i < SORTN; i += TM) keys[i] = 0ull;
        }
      }
      epi_bar();
      // `comb` is consumed: restore A_ext / zero for the next item's MMAs (generic writes -> async proxy fence)
      if (!kSinglePart) {
        for (int i = tid; i < (NBUF * 2 * TM * 16 + 4096) / 4; i += EPI_THREADS) init_ext_word(i);
        fence_proxy_async();
      }
      if (small_k) {
        if (warp == 0) {
          unsigned long long a = warp_fold_top32(keys[lane], keys[32 + lane], lane);
          a = warp_fold_top32(a, warp_fold_top32(keys[64 + lane], keys[96 + lane], lane), lane);
          if (lane < A.k && grp < A.groups_real) A.part_keys[((size_t)u * A.groups_real + grp) * A.k + lane] = a;
        }
        continue;  // (the next item's first epi_bar orders these reads of `keys` before its writes)
      }
      // bitonic sort (descending) of SORTN keys, one key pair per epilogue thread
      for (int kk = 2; kk <= SORTN; kk <<= 1) {
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
          for (int i = tid; i < SORTN; i += EPI_THREADS) {
            const int ixj = i ^ jj;
            if (ixj > i) {
              const unsigned long long x = keys[i], y = keys[ixj];
              const bool desc = (i & kk) == 0;
              if (desc ? (x < y) : (x > y)) {
                keys[i] = y;
                keys[ixj] = x;
              }
            }
          }
          epi_bar();
        }
      }
      if (grp < A.groups_real)
        for (int i = tid; i < A.k; i += EPI_THREADS) A.part_keys[((size_t)u * A.groups_real + grp) * A.k + i] = keys[i];
    }
  }
  // ---- teardown ---------------------------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync_all();  // nobody leaves while the other CTA may still signal it or read its operands
  if (warp == EPI_WARPS) {
    if constexpr (kPair) tmem_dealloc2(tmem, 512);
    else tmem_dealloc(tmem, 512);
  }
}


}  // namespace tc

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
int launch_topk_merge(const unsigned long long* in_keys, const float* in_score, const int32_t* in_id, int n_users,
                      int n_lists, int k, float* out_score, int32_t* out_id, cudaStream_t stream);
int launch_topk_merge_keys_multi(const unsigned long long* keys, unsigned long long* scratch, int64_t user_stride, int64_t list_stride,
                                 int n_users, int n_lists, int k, unsigned long long* out_keys, float* out_score, int32_t* out_id,
                                 cudaStream_t stream);
int merge_scratch_lists(int n_lists, int k);

static inline size_t al256(size_t x) { return (x + 255) / 256 * 256; }

// ---- plan: what depends on the weights and the catalogue range only -----------------------------------------------------------
//   [header 4 KB: table maxima | Scales | perm | c_k | u_d] [candidate image of the (first) pass] [AUTO: candidate image of the SPLIT pass]
struct PlanLayout {
  tc::Geo g, gs;       // geometry of the single pass / of AUTO's MIX pass; gs: AUTO's SPLIT pass
  bool two_pass;       // NAIS_PREC_TC_AUTO on a shape that has a MIX geometry
  bool pair;           // the shape has the CTA-pair kernel (and NAIS_PREC_FLAG_ONE_CTA is not set): the candidate image is padded to
                       // an even number of tile groups
  tc::Geo gp, gsp;     // g / gs with the pair kernels' half-chunk stage geometry
  int groups, n_tiles_pad;
  size_t hdr, pimg, pimg2, total;
};

static bool plan_layout(const NaisParams& p, int64_t poi_begin, int64_t poi_end, int precision, PlanLayout& L) {
  const int prec = precision & NAIS_PREC_MASK;
  if (!tc::make_geo(p, prec, L.g)) return false;
  L.two_pass = false;
  if (prec == NAIS_PREC_TC_AUTO) {
    if (!tc::make_geo(p, NAIS_PREC_TC_SPLIT, L.gs)) return false;
    // make_geo(AUTO) gives the MIX geometry where an e5m2 K-step exists; the two passes then share every size
    L.two_pass = L.g.mix != 0;
    if (L.two_pass && (L.gs.a_tile != L.g.a_tile || L.gs.b_chunk != L.g.b_chunk || L.gs.tpc != L.g.tpc || L.gs.hch != L.g.hch ||
                       L.gs.hsplit != L.g.hsplit))
      return false;
  } else {
    L.gs = L.g;
  }
  const int64_t range = poi_end - poi_begin;
  const int64_t tiles = (range + tc::TM - 1) / tc::TM;
  L.groups = (int)((tiles + L.g.tpc - 1) / L.g.tpc);
  if (L.groups < 1) L.groups = 1;
  // CTA pairs: the D = hid = 64 compile-time-shape kernels only; a stage then holds half a chunk
  auto pair_shape = [](const tc::Geo& q) {
    return q.D == 64 && q.hid == 64 && q.nrow == 144 && q.kp == 1 && q.hch == 2 && q.stages == 2 && !q.km && (q.mix || q.split);
  };
  L.pair = !(precision & (NAIS_PREC_FLAG_ONE_CTA | NAIS_PREC_FLAG_GENERIC)) && pair_shape(L.g) && pair_shape(L.gs) && L.groups >= 2;
  L.gp = L.g;
  L.gsp = L.gs;
  if (L.pair)
    for (tc::Geo* q : {&L.gp, &L.gsp}) {
      q->pair = 1;
      q->smem_bytes -= q->stages * q->stage_bytes;
      q->stage_bytes = q->b_chunk / 2;
      q->stages = 4;  // half-chunk stages: the same bytes in flight as the one-CTA kernel's two, twice the look-ahead (the relay of
      q->smem_bytes += q->stages * q->stage_bytes;  // "landed" and the multicast of "free" each cost a trip between the SMs)
    }
  L.n_tiles_pad = (L.pair ? (L.groups + 1) / 2 * 2 : L.groups) * L.g.tpc;
  size_t o = 0;
  L.hdr = o;
  o += tc::HDR_BYTES;
  L.pimg = o;
  o += al256((size_t)L.n_tiles_pad * L.g.a_tile);
  L.pimg2 = o;
  if (L.two_pass) o += al256((size_t)L.n_tiles_pad * L.g.a_tile);
  L.total = o;
  return true;
}

// ---- per-call workspace: [pass flags 256 B] [user operand image: everything that is left] [per-item keys] [merge scratch] -------
static inline size_t call_keys_bytes(int n_users, int groups, int k) { return al256((size_t)n_users * groups * k * 8); }
static inline size_t call_scratch_bytes(int n_users, int groups, int k) {
  return al256((size_t)n_users * merge_scratch_lists(groups, k) * k * 8 + 8);
}

// The two-branch (disentangled) model, model.py:467-534: two independent attentions whose scores add.  Each branch is scored as a
// one-branch model (its own plan section: scales, permutation, candidate image; its own user operand, built in the same per-call
// workspace one after the other); the first pass leaves its scores in a [n_users, range] buffer at the head of the workspace
// (MainArgs::all_scores), the second adds them before it ranks (MainArgs::score_in).
static NaisParams branch_view(const NaisParams& p, int bi) {
  NaisParams q = p;
  q.n_branch = 1;
  q.branch[0] = p.branch[bi];
  return q;
}
static inline size_t branch_scores_bytes(const NaisParams& p, int n_users, int64_t poi_begin, int64_t poi_end) {
  return p.n_branch > 1 ? al256((size_t)n_users * (size_t)(poi_end - poi_begin) * 4) : 0;
}

bool tc_supported(const NaisParams& p, int precision) {
  for (int bi = 0; bi < p.n_branch; ++bi) {
    tc::Geo g;
    if (!tc::make_geo(branch_view(p, bi), precision & NAIS_PREC_MASK, g)) return false;
  }
  return true;
}

static size_t plan_bytes_1(const NaisParams& p, int64_t poi_begin, int64_t poi_end, int precision) {
  PlanLayout L;
  return plan_layout(p, poi_begin, poi_end, precision, L) ? L.total : 0;
}
size_t fullrank_tc_plan_bytes(const NaisParams& p, int64_t poi_begin, int64_t poi_end, int precision) {
  size_t total = 0;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const size_t b = plan_bytes_1(branch_view(p, bi), poi_begin, poi_end, precision);
    if (!b) return 0;
    total += b;
  }
  return total;
}

static size_t call_workspace_bytes_1(const NaisParams& p, int n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end, int k,
                                     int precision) {
  PlanLayout L;
  if (!plan_layout(p, poi_begin, poi_end, precision, L)) return 0;
  const int64_t max_chunks = (L.g.hch == 2 ? (nnz + n_users) / 2 : nnz * L.g.hsplit) + 2;
  return 256 + al256((size_t)max_chunks * L.g.b_chunk) + call_keys_bytes(n_users, L.groups, k) + call_scratch_bytes(n_users, L.groups, k);
}
size_t fullrank_tc_call_workspace_bytes(const NaisParams& p, int n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end, int k,
                                        int precision) {
  size_t most = 0;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const size_t b = call_workspace_bytes_1(branch_view(p, bi), n_users, nnz, poi_begin, poi_end, k, precision);
    if (!b) return 0;
    most = b > most ? b : most;
  }
  return most + branch_scores_bytes(p, n_users, poi_begin, poi_end);
}

size_t fullrank_tc_workspace_bytes(const NaisParams& p, int n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end, int k,
                                   int precision) {
  const size_t a = fullrank_tc_plan_bytes(p, poi_begin, poi_end, precision);
  const size_t b = fullrank_tc_call_workspace_bytes(p, n_users, nnz, poi_begin, poi_end, k, precision);
  return (a && b) ? a + b + 1024 + (size_t)n_users * 8 : 0;
}

static int check_arch(int& sms) {
  int dev = 0, major = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return NAIS_ERR_ARCH;
  sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return 0;
}

// Once per (weights, catalogue range, precision): table maxima -> scales / permutation -> candidate image(s).
static int prepare_1(const NaisParams& p, const NaisCatalog& cat, int64_t poi_begin, int64_t poi_end, int precision, void* plan,
                     size_t plan_bytes, cudaStream_t stream) {
  if (poi_end <= poi_begin) return 0;
  int sms;
  int rc = check_arch(sms);
  if (rc) return rc;
  PlanLayout L;
  if (!plan_layout(p, poi_begin, poi_end, precision, L)) return NAIS_ERR_SHAPE;
  if (plan_bytes < L.total) return NAIS_ERR_WORKSPACE;
  unsigned char* base = reinterpret_cast<unsigned char*>(plan);
  unsigned char* hdr = base + L.hdr;
  const NaisBranch& br = p.branch[0];
  cudaError_t e = cudaMemsetAsync(hdr, 0, tc::HDR_BYTES, stream);
  if (e != cudaSuccess) return (int)e;
  unsigned* mx = reinterpret_cast<unsigned*>(hdr);
  auto amax = [&](const float* x, size_t n, unsigned* out) {
    if (!x || n == 0) return;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 4 * sms) blocks = 4 * sms;
    tc::absmax_kernel<<<blocks, 256, 0, stream>>>(x, n, out);
    NAIS_COUNT_LAUNCH(1);
  };
  amax(br.tgt_poi, (size_t)p.item_num * br.w_poi, mx + 0);
  amax(br.tgt_reg, (size_t)p.region_num * br.w_reg, mx + 1);
  amax(br.hist_poi, (size_t)p.item_num * br.w_poi, mx + 2);
  amax(br.hist_reg, (size_t)p.region_num * br.w_reg, mx + 3);
  tc::scales_kernel<<<1, 256, 0, stream>>>(p, hdr);
  NAIS_COUNT_LAUNCH(1);
  tc::pack_candidates_kernel<<<L.n_tiles_pad, 256, 0, stream>>>(p, cat, poi_begin, poi_end, L.g, hdr, base + L.pimg);
  NAIS_COUNT_LAUNCH(1);
  if (L.two_pass) {
    tc::pack_candidates_kernel<<<L.n_tiles_pad, 256, 0, stream>>>(p, cat, poi_begin, poi_end, L.gs, hdr, base + L.pimg2);
    NAIS_COUNT_LAUNCH(1);
  }
  e = cudaGetLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

int fullrank_tc_prepare(const NaisParams& p, const NaisCatalog& cat, int64_t poi_begin, int64_t poi_end, int precision, void* plan,
                        size_t plan_bytes, cudaStream_t stream) {
  size_t off = 0;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const NaisParams q = branch_view(p, bi);
    const size_t b = plan_bytes_1(q, poi_begin, poi_end, precision);
    if (!b) return NAIS_ERR_SHAPE;
    if (plan_bytes < off + b) return NAIS_ERR_WORKSPACE;
    const int rc = prepare_1(q, cat, poi_begin, poi_end, precision, reinterpret_cast<unsigned char*>(plan) + off, b, stream);
    if (rc) return rc;
    off += b;
  }
  return 0;
}

typedef void (*MainKernel)(const tc::MainArgs);

// compile-time-shape instantiations: kFix 1 / 2 = D = hid = 64 or 32 in SPLIT / MIX, kFix 3 = D = hid = 128 (generic code paths,
// constants folded); everything else (and NAIS_PREC_FLAG_GENERIC) runs the run-time-shape kernels
static MainKernel pick_kernel(const tc::Geo& gg, bool generic) {
  const bool s64 = gg.D == 64 && gg.hid == 64 && gg.nrow == 144, s32 = gg.D == 32 && gg.hid == 32 && gg.nrow == 80;
  if (gg.km) generic = true;  // the haversine bias lives in the run-time-shape epilogue only
  const int fix = ((s64 || s32) && gg.kp == 1 && gg.hch == 2 && gg.stages == 2 && !generic) ? (gg.mix ? 2 : (gg.split ? 1 : 0)) : 0;
  if (gg.pair) return gg.mix ? tc::fullrank_tc_kernel<true, 2, 6, 64> : tc::fullrank_tc_kernel<true, 2, 5, 64>;
  if (gg.kp == 1) {
    if (gg.hch != 2) return tc::fullrank_tc_kernel<true, 1, 0>;
    if (fix == 2) return s64 ? tc::fullrank_tc_kernel<true, 2, 2, 64> : tc::fullrank_tc_kernel<true, 2, 2, 32>;
    if (fix == 1) return s64 ? tc::fullrank_tc_kernel<true, 2, 1, 64> : tc::fullrank_tc_kernel<true, 2, 1, 32>;
    return tc::fullrank_tc_kernel<true, 2, 0>;
  }
  if (gg.tpc == 1) return gg.hch == 2 ? tc::fullrank_tc_kernel<false, 2, 4> : tc::fullrank_tc_kernel<false, 1, 4>;  // D > 128
  if (gg.hch == 2) return tc::fullrank_tc_kernel<false, 2, 0>;
  if (gg.D == 128 && gg.hid == 128 && gg.kp == 4 && gg.nrow == 144 && gg.stages == 3 && (gg.mix || gg.split) && !generic)
    return tc::fullrank_tc_kernel<false, 1, 3>;
  return tc::fullrank_tc_kernel<false, 1, 0>;
}

// Geo re-ranking (MainArgs::geo) runs the run-time-shape kernels only, like NAIS_DIST_KM: the compile-time-shape and CTA-pair
// kernels have no geo variant.  Extra shared memory: the fourth `comb` array of the D <= 64 kernels (private region) and the
// staged cos(latitude) of the history items where NAIS_DIST_KM has not already reserved it.
static MainKernel pick_geo_kernel(const tc::Geo& gg) {
  if (gg.kp == 1) return gg.hch == 2 ? tc::fullrank_tc_kernel<true, 2, 0, 64, true> : tc::fullrank_tc_kernel<true, 1, 0, 64, true>;
  if (gg.tpc == 1) return gg.hch == 2 ? tc::fullrank_tc_kernel<false, 2, 4, 64, true> : tc::fullrank_tc_kernel<false, 1, 4, 64, true>;
  return gg.hch == 2 ? tc::fullrank_tc_kernel<false, 2, 0, 64, true> : tc::fullrank_tc_kernel<false, 1, 0, 64, true>;
}
static int geo_extra_smem(const tc::Geo& gg) { return (gg.kp == 1 ? 3 * tc::TPC * tc::TM * 4 : 0) + (gg.km ? 0 : tc::HMETA * 4); }

// Per user batch: user operand image -> scoring pass(es) -> merge of the per-item lists.
static int run_1(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin, int64_t poi_end, int k,
                 int exclude, int precision, const void* plan, size_t plan_bytes, unsigned long long* out_keys, float* out_score,
                 int32_t* out_id, float* all_scores, const float* score_in, bool merge, void* ws, size_t ws_bytes, cudaStream_t stream,
                 const GeoMixArgs* geo = nullptr) {
  if (users.n_users == 0 || poi_end <= poi_begin) return 0;
  int sms;
  int rc = check_arch(sms);
  if (rc) return rc;
  PlanLayout L;
  if (!plan_layout(p, poi_begin, poi_end, precision, L)) return NAIS_ERR_SHAPE;
  if (!plan || plan_bytes < L.total) return NAIS_ERR_WORKSPACE;
  const unsigned char* pbase = reinterpret_cast<const unsigned char*>(plan);
  const unsigned char* hdr = pbase + L.hdr;
  // nnz is not known to the library (offsets live on the device): the caller sized the workspace with it; the chunk capacity
  // of the operand image is whatever the workspace leaves after the fixed-size parts.
  const size_t keys_bytes = call_keys_bytes(users.n_users, L.groups, k), scratch_bytes = call_scratch_bytes(users.n_users, L.groups, k);
  if (ws_bytes < 256 + keys_bytes + scratch_bytes + (size_t)L.g.b_chunk) return NAIS_ERR_WORKSPACE;
  unsigned char* base = reinterpret_cast<unsigned char*>(ws);
  int* pass_flags = reinterpret_cast<int*>(base);
  const size_t bimg_bytes = (ws_bytes - 256 - keys_bytes - scratch_bytes) / 256 * 256;
  unsigned char* bimg = base + 256;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(base + 256 + bimg_bytes);
  unsigned long long* scratch = reinterpret_cast<unsigned long long*>(base + 256 + bimg_bytes + keys_bytes);
  const int64_t max_chunks = (int64_t)(bimg_bytes / L.g.b_chunk);
  cudaError_t e;
  if (L.two_pass) {
    e = cudaMemsetAsync(pass_flags, 0, 8, stream);
    if (e != cudaSuccess) return (int)e;
  }
  const bool generic = (precision & NAIS_PREC_FLAG_GENERIC) != 0;
  // CTA pairs need two co-scheduled SMs of a TPC with the kernel's shared memory each: asked once per device (a partitioned GPU may
  // not offer any); without them the one-CTA kernels run on the same plan (its candidate image is a superset)
  bool use_pair = L.pair && !geo;
  if (geo) {
    if (L.g.smem_bytes + geo_extra_smem(L.g) > 227 * 1024 || (L.two_pass && L.gs.smem_bytes + geo_extra_smem(L.gs) > 227 * 1024))
      return NAIS_ERR_SHAPE;
  }
  if (use_pair) {
    static int pair_ok[64];  // 0 unknown, 1 yes, -1 no
    int dev = 0;
    cudaGetDevice(&dev);
    int& st = pair_ok[dev & 63];
    if (st == 0) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(2);
      cfg.blockDim = dim3(tc::THREADS);
      cfg.dynamicSmemBytes = L.gp.smem_bytes;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2;
      at[0].val.clusterDim.y = 1;
      at[0].val.clusterDim.z = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      MainKernel kp = pick_kernel(L.gp, false);
      int n = 0;
      const bool ok = cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, L.gp.smem_bytes) == cudaSuccess &&
                      cudaOccupancyMaxActiveClusters(&n, kp, &cfg) == cudaSuccess && n >= 1;
      if (!ok) cudaGetLastError();
      st = ok ? 1 : -1;
    }
    use_pair = st == 1;
  }
  const tc::Geo& g1 = use_pair ? L.gp : L.g;
  const tc::Geo& g2 = use_pair ? L.gsp : L.gs;
  {
    dim3 grid(users.n_users, 64);
    tc::pack_users_kernel<<<grid, 256, 0, stream>>>(p, users, g1, g2, L.two_pass ? 1 : 0, hdr, bimg, max_chunks, pass_flags,
                                                   bad_index_flag());
    NAIS_COUNT_LAUNCH(1);
  }
  auto run = [&](const tc::Geo& gg, const unsigned char* pimg, int gate) -> int {
    tc::MainArgs A;
    A.p = p;
    A.cat = cat;
    A.users = users;
    A.g = gg;
    A.poi_begin = poi_begin;
    A.poi_end = poi_end;
    A.k = k;
    A.exclude = exclude;
    A.groups = gg.pair ? (L.groups + 1) / 2 * 2 : L.groups;
    A.groups_real = L.groups;
    A.n_items = (int64_t)users.n_users * (gg.pair ? A.groups / 2 : A.groups);
    A.hdr = hdr;
    A.Pimg = pimg;
    A.Bimg = bimg;
    A.part_keys = keys;
    A.all_scores = all_scores;
    A.score_in = score_in;
    A.max_chunks = max_chunks;
    A.gate = gate;
    A.pass_flags = pass_flags;
    A.geo = geo ? *geo : GeoMixArgs{};
    MainKernel kern = geo ? pick_geo_kernel(gg) : pick_kernel(gg, generic);
    const int smem = gg.smem_bytes + (geo ? geo_extra_smem(gg) : 0);
    cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e2 != cudaSuccess) return (int)e2;
    if (gg.pair) {  // one cluster of two CTAs (the two SMs of a TPC) per pair item
      const int pairs = (int)(A.n_items < sms / 2 ? A.n_items : sms / 2);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(2 * pairs);
      cfg.blockDim = dim3(tc::THREADS);
      cfg.dynamicSmemBytes = gg.smem_bytes;
      cfg.stream = stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2;
      at[0].val.clusterDim.y = 1;
      at[0].val.clusterDim.z = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      e2 = cudaLaunchKernelEx(&cfg, kern, A);
      NAIS_COUNT_LAUNCH(1);
      return e2 == cudaSuccess ? 0 : (int)e2;
    }
    const int grid = (int)(A.n_items < sms ? A.n_items : sms);
    kern<<<grid, tc::THREADS, smem, stream>>>(A);
    NAIS_COUNT_LAUNCH(1);
    e2 = cudaGetLastError();
    return e2 == cudaSuccess ? 0 : (int)e2;
  };
  if (L.two_pass) {
    // the MIX pass and the SPLIT pass back to back; each user belongs to one (decided on the device: the library never
    // synchronises, so the choice cannot come back to the host); a pass nobody takes is one launch that exits at once
    rc = run(g1, pbase + L.pimg, 1);
    if (rc) return rc;
    rc = run(g2, pbase + L.pimg2, 0);
  } else {
    rc = run(g1, pbase + L.pimg, -1);
  }
  if (rc || !merge) return rc;
  return launch_topk_merge_keys_multi(keys, scratch, (int64_t)L.groups * k, k, users.n_users, L.groups, k, out_keys, out_score, out_id,
                                      stream);
}

int fullrank_tc_run(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin, int64_t poi_end, int k,
                    int exclude, int precision, const void* plan, size_t plan_bytes, unsigned long long* out_keys, float* out_score,
                    int32_t* out_id, float* all_scores, void* ws, size_t ws_bytes, cudaStream_t stream, const GeoMixArgs* geo) {
  if (users.n_users == 0 || poi_end <= poi_begin) return 0;
  if (p.n_branch == 1)
    return run_1(p, cat, users, poi_begin, poi_end, k, exclude, precision, plan, plan_bytes, out_keys, out_score, out_id, all_scores,
                 nullptr, true, ws, ws_bytes, stream, geo);
  const size_t sbytes = branch_scores_bytes(p, users.n_users, poi_begin, poi_end);
  if (!plan || ws_bytes < sbytes + 512) return NAIS_ERR_WORKSPACE;
  float* sbuf = reinterpret_cast<float*>(ws);  // running sum of the branch scores
  unsigned char* rest = reinterpret_cast<unsigned char*>(ws) + sbytes;
  size_t off = 0;
  for (int bi = 0; bi < p.n_branch; ++bi) {
    const NaisParams q = branch_view(p, bi);
    const size_t b = plan_bytes_1(q, poi_begin, poi_end, precision);
    if (!b) return NAIS_ERR_SHAPE;
    if (plan_bytes < off + b) return NAIS_ERR_WORKSPACE;
    const bool last = bi == p.n_branch - 1;
    const int rc = run_1(q, cat, users, poi_begin, poi_end, k, exclude, precision, reinterpret_cast<const unsigned char*>(plan) + off, b,
                         out_keys, out_score, out_id, last ? all_scores : sbuf, bi ? sbuf : nullptr, last, rest, ws_bytes - sbytes, stream,
                         last ? geo : nullptr);  // the mix needs the summed score: the last pass only
    if (rc) return rc;
    off += b;
  }
  return 0;
}

// The unplanned entry: plan at the head of the workspace, prepared on every call.
int launch_fullrank_tc(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin,
                       int64_t poi_end, int k, int exclude, int precision, float* out_score, int32_t* out_id,
                       float* all_scores, void* ws, size_t ws_bytes, cudaStream_t stream) {
  if (users.n_users == 0 || poi_end <= poi_begin) return 0;
  const size_t plan_bytes = fullrank_tc_plan_bytes(p, poi_begin, poi_end, precision);
  if (!plan_bytes) return NAIS_ERR_SHAPE;
  if (ws_bytes < plan_bytes + 512) return NAIS_ERR_WORKSPACE;
  int rc = fullrank_tc_prepare(p, cat, poi_begin, poi_end, precision, ws, plan_bytes, stream);
  if (rc) return rc;
  return fullrank_tc_run(p, cat, users, poi_begin, poi_end, k, exclude, precision, ws, plan_bytes, nullptr, out_score, out_id,
                         all_scores, reinterpret_cast<unsigned char*>(ws) + plan_bytes, ws_bytes - plan_bytes, stream, nullptr);
}

}  // namespace nais
