// extern "C" entry points of libnais_b200.so: argument validation + dispatch.  See include/nais_b200.h.
#include <cstdio>

#include <cstring>
#include <mutex>

#include "nais_common.cuh"
#include "nais_pairs_tile.cuh"

namespace nais {
// nais_fp32.cu
int launch_pairs_fwd(const NaisParams& p, const NaisPairs& b, float* score, float* row_sum, float* parts, cudaStream_t stream,
                     float* cell_e = nullptr, float* cell_es = nullptr);
int launch_fullrank_fp32(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin,
                         int64_t poi_end, int k, int exclude, float* out_score, int32_t* out_id, float* all_scores,
                         void* ws, size_t ws_bytes, cudaStream_t stream, const GeoMixArgs* geo = nullptr);
int launch_topk_merge(const unsigned long long* in_keys, const float* in_score, const int32_t* in_id, int n_users,
                      int n_lists, int k, float* out_score, int32_t* out_id, cudaStream_t stream);
int launch_topk_merge_keys_multi(const unsigned long long* keys, unsigned long long* scratch, int64_t user_stride, int64_t list_stride,
                                 int n_users, int n_lists, int k, unsigned long long* out_keys, float* out_score, int32_t* out_id,
                                 cudaStream_t stream);
int merge_scratch_lists(int n_lists, int k);
int choose_splits(int n_users, int64_t range);
// nais_bwd.cu
size_t pairs_bwd_workspace_bytes(const NaisParams& p, const NaisPairs& b);  // (the backward's steps: nais_common.cuh PairsBwd)
bool pairs_tc_bwd_supported(const NaisParams& p, const NaisPairs& b);
size_t rows_adagrad_workspace_bytes(int64_t n, int w);
int launch_rows_adagrad(const int32_t* keys, const float* rows, int64_t n, int w, int n_rows, float* grad_out, float* param, float* sum,
                        float lr, float eps, void* ws, size_t ws_bytes, cudaStream_t stream);
// nais_tc.cu
size_t fullrank_tc_workspace_bytes(const NaisParams& p, int n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end, int k,
                                   int precision);
int launch_fullrank_tc(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin,
                       int64_t poi_end, int k, int exclude, int precision, float* out_score, int32_t* out_id,
                       float* all_scores, void* ws, size_t ws_bytes, cudaStream_t stream);
bool tc_supported(const NaisParams& p, int precision);
size_t fullrank_tc_plan_bytes(const NaisParams& p, int64_t poi_begin, int64_t poi_end, int precision);
size_t fullrank_tc_call_workspace_bytes(const NaisParams& p, int n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end, int k,
                                        int precision);
int fullrank_tc_prepare(const NaisParams& p, const NaisCatalog& cat, int64_t poi_begin, int64_t poi_end, int precision, void* plan,
                        size_t plan_bytes, cudaStream_t stream);
int fullrank_tc_run(const NaisParams& p, const NaisCatalog& cat, const NaisUsers& users, int64_t poi_begin, int64_t poi_end, int k,
                    int exclude, int precision, const void* plan, size_t plan_bytes, unsigned long long* out_keys, float* out_score,
                    int32_t* out_id, float* all_scores, void* ws, size_t ws_bytes, cudaStream_t stream,
                    const GeoMixArgs* geo = nullptr);
// nais_sampler.cu
int launch_sample_batch(const int64_t* seg_offsets, const int64_t* hist, int n_seg, const int64_t* row_offsets, int num_ng, int item_num,
                        const int32_t* poi_region, const float* poi_coords, uint64_t seed, int max_hist, int64_t* tgt, float* label,
                        int64_t* treg, float* tgt_coords, cudaStream_t stream);
// nais_pairs_tc.cu
bool pairs_tc_supported(const NaisParams& p, const NaisPairs& b);
int launch_bce_dscore(const float* score, const float* label, const float* row_weight, int64_t B, float* dscore, float* loss,
                      cudaStream_t stream);
int launch_bpr_dscore(const float* score, const float* group_weight, int64_t B, int num_neg, float* dscore, float* loss,
                      cudaStream_t stream);
int launch_dense_adagrad(float* const* param, float* const* sum, const float* const* grad, const int* n, float lr, float eps,
                         cudaStream_t stream);
int launch_pairs_fwd_tc(const NaisParams& p, const NaisPairs& b, float* score, float* row_sum, float* parts,
                        unsigned long long* act_mask, cudaStream_t stream, float* cell_e = nullptr, float* cell_es = nullptr);
// nais_explain.cu
int launch_explain_select(const NaisParams& p, const NaisPairs& b, int m, const float* cell_e, const float* cell_es,
                          const float* row_sum, int32_t* out_pos, float* out_contrib, float* out_attn, cudaStream_t stream);
}  // namespace nais

namespace nais {
unsigned long long g_launches = 0;
// The one piece of library-owned device state: raised by any kernel that meets an id outside its table (nais_common.cuh
// checked_id), read and reset by nais_poll_bad_index.  Static device storage: one word per device, nothing is allocated.
__device__ int g_bad_index = 0;
int* bad_index_flag() {
  int* ptr = nullptr;
  cudaGetSymbolAddress(reinterpret_cast<void**>(&ptr), g_bad_index);
  return ptr;
}
}  // namespace nais
using namespace nais;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int check_params(const NaisParams* p) {
  if (!p) return NAIS_ERR_NULL;
  if (p->n_branch < 1 || p->n_branch > 2) return NAIS_ERR_SHAPE;
  if (p->hid < 1 || p->hid > 1024 || p->item_num < 1) return NAIS_ERR_SHAPE;
  if (p->dist_mode < NAIS_DIST_NONE || p->dist_mode > NAIS_DIST_KM) return NAIS_ERR_MODE;
  for (int i = 0; i < p->n_branch; ++i) {
    const NaisBranch& b = p->branch[i];
    const int D = b.w_poi + b.w_reg;
    if (b.w_poi < 0 || b.w_reg < 0 || D < 4 || D > MAXD || (D & 3)) return NAIS_ERR_SHAPE;
    if (b.w_poi && (!b.hist_poi || !b.tgt_poi)) return NAIS_ERR_NULL;
    if (b.w_reg && (!b.hist_reg || !b.tgt_reg || p->region_num < 1)) return NAIS_ERR_NULL;
    if (!b.w1 || !b.b1 || !b.w2) return NAIS_ERR_NULL;
  }
  if (p->dist_mode == NAIS_DIST_LATLON && (!p->dist_w || !p->dist_b)) return NAIS_ERR_NULL;
  if (p->dist_mode == NAIS_DIST_KM && (!p->dist_embed || p->dist_buckets < 1)) return NAIS_ERR_NULL;
  if (p->dist_mode == NAIS_DIST_KM && p->dist_buckets != 1) return NAIS_ERR_MODE;  // one bucket, like the reference (model.py:497-498)
  if (p->pairs_precision < NAIS_PAIRS_AUTO || p->pairs_precision > NAIS_PAIRS_TC) return NAIS_ERR_MODE;
  return 0;
}

static int check_pairs(const NaisParams* p, const NaisPairs* b) {
  if (!b) return NAIS_ERR_NULL;
  const bool seg = b->seg_offsets != nullptr;
  if (b->B < 0 || (!seg && b->H < 1)) return NAIS_ERR_SHAPE;
  if (b->B == 0) return 0;
  if (!b->hist || !b->tgt) return NAIS_ERR_NULL;
  bool need_reg = false;
  for (int i = 0; i < p->n_branch; ++i) need_reg |= p->branch[i].w_reg > 0;
  if (need_reg && (!b->hreg || !b->treg)) return NAIS_ERR_NULL;
  if (seg) {  // segmented (multi-user) layout: shared histories, distances formed in the kernel
    if (b->n_seg < 1 || b->n_tiles < 0 || b->n_cells < 0) return NAIS_ERR_SHAPE;
    if (!b->row_offsets || !b->seg_cell_offsets || (b->n_tiles && (!b->tile_seg || !b->tile_row0))) return NAIS_ERR_NULL;
    if (b->aux) return NAIS_ERR_MODE;
    if (p->dropout_p > 0.f && p->n_branch != 1) return NAIS_ERR_MODE;  // (the disentangled model has no dropout)
    if (p->dist_mode != NAIS_DIST_NONE && (!b->hist_coords || !b->tgt_coords)) return NAIS_ERR_NULL;
    return 0;
  }
  if (p->dist_mode != NAIS_DIST_NONE && !b->aux) return NAIS_ERR_NULL;
  return 0;
}

static size_t fp32_workspace_bytes(int n_users, int64_t poi_begin, int64_t poi_end, int k) {
  const int s = choose_splits(n_users, poi_end - poi_begin);
  return 1024 + (size_t)n_users * 8 + (s > 1 ? (size_t)n_users * s * k * sizeof(unsigned long long) : 0);
}

__global__ void pack_keys_kernel(const float* __restrict__ s, const int32_t* __restrict__ id, size_t n, unsigned long long* keys) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) keys[i] = id[i] >= 0 ? make_key(s[i], id[i]) : 0ull;
}

__global__ void fill_empty_topk_kernel(float* s, int32_t* id, size_t n) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) {
    s[i] = -INFINITY;
    id[i] = -1;
  }
}

// hits[u,i] = | set(pos(u)) & set(rec[u,:k_i]) | : one warp per user; duplicates in either list count once, like the
// reference's Python set intersection (eval_metrics.py:40-42).
// log of the power-law geographical score of powerLaw.py:85-92: G(u, j) = prod_{h in visited(u)} a * max(0.01, d(h, j))^b
//   log G = sum_h (ln a + b * ln max(0.01, d_km(h, j)))      (a product of ~100 factors leaves fp32 / fp64 range; its log does not)
// One thread per candidate j (invalid threads compute a dummy), the user's history coordinates staged through shared memory in
// tiles of 256; every thread of the block must call.  kHist: also report whether j is one of the user's history items.
template <bool kHist>
__device__ __forceinline__ float powerlaw_logg_block(const NaisCatalog& cat, const NaisUsers& users, int u, int64_t j, bool valid,
                                                     float ln_a, float b, bool* in_hist) {
  __shared__ float s_la[256], s_lo[256], s_cos[256];
  __shared__ int s_id[kHist ? 256 : 1];
  const int64_t hb = users.offsets[u];
  const int H = (int)(users.offsets[u + 1] - hb);
  float cla = 0.f, clo = 0.f, ccos = 1.f;
  if (valid) {
    cla = __ldg(cat.coords + 2 * (j - cat.row_base));
    clo = __ldg(cat.coords + 2 * (j - cat.row_base) + 1);
    ccos = cosf((cat.center_lat + cla) * 0.017453292519943295f);
  }
  float acc = 0.f;
  bool seen = false;
  for (int h0 = 0; h0 < H; h0 += 256) {
    __syncthreads();
    if (h0 + (int)threadIdx.x < H) {
      const float la = __ldg(users.coords + 2 * (hb + h0 + threadIdx.x)), lo = __ldg(users.coords + 2 * (hb + h0 + threadIdx.x) + 1);
      s_la[threadIdx.x] = la;
      s_lo[threadIdx.x] = lo;
      s_cos[threadIdx.x] = cosf((cat.center_lat + la) * 0.017453292519943295f);
      if constexpr (kHist) s_id[threadIdx.x] = __ldg(users.items + hb + h0 + threadIdx.x);
    }
    __syncthreads();
    const int n = min(256, H - h0);
    for (int i = 0; i < n; ++i) {
      acc += powerlaw_log_term(dist_km_f(cla, clo, s_la[i], s_lo[i], ccos, s_cos[i]), ln_a, b);
      if constexpr (kHist) seen = seen || (int64_t)s_id[i] == j;
    }
  }
  if (in_hist) *in_hist = seen;
  return acc;
}

__global__ void powerlaw_logscore_kernel(NaisCatalog cat, NaisUsers users, int64_t poi_begin, int64_t poi_end, float ln_a, float b,
                                         float* __restrict__ out) {
  const int u = blockIdx.x;  // users on grid.x (no 65 535 limit), candidate blocks on grid.y
  const int64_t j = poi_begin + (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  const bool valid = j < poi_end;
  const float acc = powerlaw_logg_block<false>(cat, users, u, j, valid, ln_a, b, nullptr);
  if (valid) out[(size_t)u * (poi_end - poi_begin) + (j - poi_begin)] = acc;
}

// Atomic max of a float by its bit pattern: non-negative floats order like signed ints, negative ones reversed like unsigned
// ints.  Exact, so the result does not depend on the order the blocks arrive in.
__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  if (v != v) return;
  if (__float_as_int(v) >= 0) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}

__global__ void fill_float_kernel(float* out, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

// M_u = max_j log G(u, j) over the candidates [poi_begin, poi_end) (minus the history when `exclude`), no [U, N] buffer:
// blocks stride over the range, reduce in the block and fold into out[u] (filled with -inf first).
__global__ void powerlaw_logmax_kernel(NaisCatalog cat, NaisUsers users, int64_t poi_begin, int64_t poi_end, float ln_a, float b,
                                       int exclude, float* __restrict__ out) {
  __shared__ float s_max[8];
  const int u = blockIdx.x;
  float m = -INFINITY;
  for (int64_t j0 = poi_begin + (int64_t)blockIdx.y * blockDim.x; j0 < poi_end; j0 += (int64_t)gridDim.y * blockDim.x) {
    const int64_t j = j0 + threadIdx.x;
    const bool valid = j < poi_end;
    bool in_hist = false;
    const float acc = exclude ? powerlaw_logg_block<true>(cat, users, u, j, valid, ln_a, b, &in_hist)
                              : powerlaw_logg_block<false>(cat, users, u, j, valid, ln_a, b, nullptr);
    if (valid && !in_hist) m = fmaxf(m, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, s_max[w]);
    if (m > -INFINITY) atomic_max_float(out + u, m);
  }
}

__global__ void hits_at_k_kernel(const int32_t* __restrict__ rec, int n_users, int k_rec, const int64_t* __restrict__ po,
                                 const int32_t* __restrict__ pi, const int32_t* __restrict__ k_list, int n_k, int32_t* hits) {
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u >= n_users) return;
  const int64_t p0 = po[u], p1 = po[u + 1];
  for (int ki = 0; ki < n_k; ++ki) {
    const int k = min(k_list[ki], k_rec);
    int cnt = 0;
    for (int r = lane; r < k; r += 32) {
      const int id = rec[(size_t)u * k_rec + r];
      if (id < 0) continue;
      bool dup = false;  // first occurrence within the prefix only
      for (int q = 0; q < r && !dup; ++q) dup = rec[(size_t)u * k_rec + q] == id;
      if (dup) continue;
      bool hit = false;
      for (int64_t q = p0; q < p1 && !hit; ++q) hit = pi[q] == id;
      cnt += hit ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) hits[(size_t)u * n_k + ki] = cnt;
  }
}

extern "C" {

int nais_abi_version(void) { return NAIS_ABI_VERSION; }
uint64_t nais_launch_count(void) { return __atomic_load_n(&nais::g_launches, __ATOMIC_RELAXED); }

const char* nais_strerror(int code) {
  switch (code) {
    case 0: return "ok";
    case NAIS_ERR_NULL: return "nais: required pointer is NULL";
    case NAIS_ERR_SHAPE: return "nais: unsupported or inconsistent dimension";
    case NAIS_ERR_ALIGN: return "nais: pointer or row width not 16-byte aligned";
    case NAIS_ERR_WORKSPACE: return "nais: workspace too small";
    case NAIS_ERR_MODE: return "nais: unknown mode or unsupported flag combination";
    case NAIS_ERR_ARCH: return "nais: tensor path needs an sm_100 device";
    case NAIS_ERR_INDEX: return "nais: index out of range in a POI / region id tensor";
    default: break;
  }
  if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
  return "nais: unknown error";
}

static bool device_is_sm100() {
  return device_info().major == 10;
}

// The pair forward for (p, b): the tcgen05 kernel where the shape has it on an sm_100 device, unless NAIS_PAIRS_FP32 asks for the
// FP32 kernel; NAIS_PAIRS_TC forces tcgen05 and is NAIS_ERR_SHAPE where it is not available.
static int choose_pairs_fwd(const NaisParams& p, const NaisPairs& b, bool* tc) {
  const bool tc_ok = pairs_tc_supported(p, b) && device_is_sm100();
  if (p.pairs_precision == NAIS_PAIRS_TC && !tc_ok) return NAIS_ERR_SHAPE;
  *tc = p.pairs_precision != NAIS_PAIRS_FP32 && tc_ok;
  return 0;
}

// tcgen05 contraction (fp16 two-term splits, fp32-grade products; writes act_mask when given) or the FP32 kernel
static int launch_chosen_fwd(bool tc, const NaisParams& p, const NaisPairs& b, float* score, float* row_sum, float* parts,
                             unsigned long long* act_mask, cudaStream_t stream) {
  return tc ? launch_pairs_fwd_tc(p, b, score, row_sum, parts, act_mask, stream) : launch_pairs_fwd(p, b, score, row_sum, parts, stream);
}

size_t nais_rows_adagrad_workspace_bytes(int64_t n, int32_t w) {
  if (n < 0 || w < 1 || w > 128) return 0;
  return rows_adagrad_workspace_bytes(n, w);
}

int nais_rows_adagrad(const int32_t* keys, const float* rows, int64_t n, int32_t w, int32_t n_rows, float* grad_out, float* param,
                      float* sum, float lr, float eps, void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  if (n < 0 || w < 1 || w > 128 || n_rows < 1) return NAIS_ERR_SHAPE;
  if (n == 0) return 0;
  if (!keys || !rows || !workspace || (sum ? !param : !grad_out)) return NAIS_ERR_NULL;
  if (sum && (!(lr >= 0.f) || !(eps >= 0.f))) return NAIS_ERR_MODE;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  return launch_rows_adagrad(keys, rows, n, w, n_rows, grad_out, param, sum, lr, eps, workspace, workspace_bytes,
                             static_cast<cudaStream_t>(stream));
}

int nais_sample_batch(const int64_t* seg_offsets, const int64_t* hist, int32_t n_seg, const int64_t* row_offsets, int32_t num_ng,
                      int32_t item_num, const int32_t* poi_region, const float* poi_coords, uint64_t seed, int32_t max_hist,
                      int64_t* tgt, float* label, int64_t* treg, float* tgt_coords, nais_stream_t stream) {
  if (n_seg < 0 || num_ng < 0 || item_num < 1 || max_hist < 0) return NAIS_ERR_SHAPE;
  if (n_seg == 0) return 0;
  if (!seg_offsets || !hist || !row_offsets || !tgt || !label) return NAIS_ERR_NULL;
  if ((treg && !poi_region) || (tgt_coords && !poi_coords)) return NAIS_ERR_NULL;
  if ((int64_t)max_hist * (num_ng + 1) >= item_num) return NAIS_ERR_SHAPE;  // not enough unvisited POIs to draw from
  return launch_sample_batch(seg_offsets, hist, n_seg, row_offsets, num_ng, item_num, poi_region, poi_coords, seed, max_hist, tgt,
                             label, treg, tgt_coords, static_cast<cudaStream_t>(stream));
}

int nais_pairs_dispatch(const NaisParams* p, const NaisPairs* batch, int32_t* fwd_tc, int32_t* bwd_tc) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!batch || !fwd_tc || !bwd_tc) return NAIS_ERR_NULL;
  if (batch->B < 0 || (!batch->seg_offsets && batch->H < 1)) return NAIS_ERR_SHAPE;
  NaisPairs b = *batch;
  if (b.B == 0) b.B = 1;  // the choice does not depend on the row count
  bool f_tc = false;
  rc = choose_pairs_fwd(*p, b, &f_tc);  // (a forced tcgen05 backward reports its own shape error)
  if (rc) return rc;
  *fwd_tc = f_tc ? 1 : 0;
  *bwd_tc = (p->pairs_precision != NAIS_PAIRS_FP32 && pairs_tc_bwd_supported(*p, b)) ? 1 : 0;
  return 0;
}

int nais_pairs_forward(const NaisParams* p, const NaisPairs* batch, float* score, float* row_sum, float* score_parts,
                       uint64_t* act_mask, nais_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  rc = check_pairs(p, batch);
  if (rc) return rc;
  if (batch->B && !score) return NAIS_ERR_NULL;
  if (batch->B == 0) return 0;
  bool tc = false;
  rc = choose_pairs_fwd(*p, *batch, &tc);
  if (rc) return rc;
  return launch_chosen_fwd(tc, *p, *batch, score, row_sum, score_parts, reinterpret_cast<unsigned long long*>(act_mask),
                           static_cast<cudaStream_t>(stream));
}

// Workspace of nais_pairs_explain: cell_e, cell_es [n_branch, cells], row_sum [n_branch, B] and the score [B] of a caller that
// passes none, each 256-byte aligned.  Host-known sizes only.
struct ExplainLayout {
  size_t cell_e, cell_es, row_sum, score, total;
};
static ExplainLayout explain_layout(const NaisParams& p, const NaisPairs& b) {
  auto up = [](size_t n) { return (n + 255) & ~(size_t)255; };
  const size_t cells = (size_t)p.n_branch * (size_t)pairs_n_cells(b) * sizeof(float);
  ExplainLayout L;
  L.cell_e = 0;
  L.cell_es = L.cell_e + up(cells);
  L.row_sum = L.cell_es + up(cells);
  L.score = L.row_sum + up((size_t)p.n_branch * b.B * sizeof(float));
  L.total = L.score + up((size_t)b.B * sizeof(float));
  return L;
}

size_t nais_pairs_explain_workspace_bytes(const NaisParams* p, const NaisPairs* batch) {
  if (check_params(p) || check_pairs(p, batch) || batch->B == 0) return 0;
  return explain_layout(*p, *batch).total;
}

int nais_pairs_explain(const NaisParams* p, const NaisPairs* batch, int32_t m, float* score, int32_t* out_pos, float* out_contrib,
                       float* out_attn, void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  rc = check_pairs(p, batch);
  if (rc) return rc;
  if (m < 1 || m > 32) return NAIS_ERR_SHAPE;
  if (p->dropout_p > 0.f) return NAIS_ERR_MODE;  // explanations are inference: no dropout
  if (batch->B == 0) return 0;
  if (!out_pos || !out_contrib) return NAIS_ERR_NULL;
  const ExplainLayout L = explain_layout(*p, *batch);
  if (workspace_bytes < L.total) return NAIS_ERR_WORKSPACE;
  if (!workspace) return NAIS_ERR_NULL;
  char* ws = static_cast<char*>(workspace);
  float *cell_e = reinterpret_cast<float*>(ws + L.cell_e), *cell_es = reinterpret_cast<float*>(ws + L.cell_es);
  float* row_sum = reinterpret_cast<float*>(ws + L.row_sum);
  if (!score) score = reinterpret_cast<float*>(ws + L.score);
  bool tc = false;
  rc = choose_pairs_fwd(*p, *batch, &tc);  // the forward nais_pairs_forward runs for (p, batch), with the per-cell terms stored
  if (rc) return rc;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = tc ? launch_pairs_fwd_tc(*p, *batch, score, row_sum, nullptr, nullptr, st, cell_e, cell_es)
          : launch_pairs_fwd(*p, *batch, score, row_sum, nullptr, st, cell_e, cell_es);
  if (rc) return rc;
  return launch_explain_select(*p, *batch, m, cell_e, cell_es, row_sum, out_pos, out_contrib, out_attn, st);
}

size_t nais_pairs_backward_workspace_bytes(const NaisParams* p, const NaisPairs* batch) {
  if (check_params(p) || !batch || batch->B < 0 || (!batch->seg_offsets && batch->H < 1)) return 0;
  return pairs_bwd_workspace_bytes(*p, *batch);
}

// The checks every backward-type entry point makes, in this order: the first failing one decides the code.  0 also when B == 0,
// where the caller has nothing to do.  `grads`: the NaisGrads (and the fused optimizer's NaisAdagrad) are given; `one_branch`: the
// presorting pair takes one branch only; `opt`: the fused optimizer's state; `inputs`: the entry point's other arrays are given.
static int check_backward_call(const NaisParams* p, const NaisPairs* batch, bool grads, bool one_branch, const NaisAdagrad* opt,
                               bool inputs, const void* workspace, size_t workspace_bytes) {
  int rc = check_params(p);
  if (rc) return rc;
  rc = check_pairs(p, batch);
  if (rc) return rc;
  if (!grads) return NAIS_ERR_NULL;
  if ((one_branch && p->n_branch != 1) || (opt && (!pairs_fused_layout(*p) || !(opt->lr >= 0.f) || !(opt->eps >= 0.f)))) return NAIS_ERR_MODE;
  if (batch->B == 0) return 0;
  if (!inputs || !workspace) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  if (workspace_bytes < pairs_bwd_workspace_bytes(*p, *batch)) return NAIS_ERR_WORKSPACE;
  return 0;
}

// The backward of nais_pairs_backward, of nais_pairs_backward_adagrad (the fused optimizer `opt`) and of
// nais_pairs_backward_presorted (one branch, on lists sorted and joined by nais_pairs_forward_presort: finish only).  Sort, then
// finish, one branch at a time: two branches of the general layout may share a list, whose workspace buffers then serve one after
// the other.
static int backward_call(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                         const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, bool grads_given,
                         const NaisAdagrad* opt, bool presorted, void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_backward_call(p, batch, grads_given, presorted, opt, score_parts && row_sum && dscore, workspace, workspace_bytes);
  if (rc || batch->B == 0) return rc;
  PairsBwd bwd;
  rc = bwd.open(*p, *batch, *grads, opt, score_parts, row_sum, reinterpret_cast<const unsigned long long*>(act_mask), dscore,
                workspace, workspace_bytes, presorted);
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int bi = 0; bi < bwd.n_branch && !rc; ++bi) {
    if (!presorted) bwd.sort(bi, st, false);
    rc = bwd.finish(bi, st, false, nullptr);
  }
  return rc;
}

int nais_pairs_backward(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                        const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, void* workspace,
                        size_t workspace_bytes, nais_stream_t stream) {
  return backward_call(p, batch, score_parts, row_sum, act_mask, dscore, grads, grads, nullptr, false, workspace, workspace_bytes, stream);
}

// Training forward of the autograd path: the coming backward's id sorts are forked onto the side streams, the forward kernel runs
// next to them on the caller's stream, and the sorts are joined back before the call returns.
int nais_pairs_forward_presort(const NaisParams* p, const NaisPairs* batch, const NaisGrads* grads, float* score, float* row_sum,
                               float* score_parts, uint64_t* act_mask, void* bwd_workspace, size_t bwd_workspace_bytes,
                               nais_stream_t stream) {
  int rc = check_backward_call(p, batch, grads, true, nullptr, score, bwd_workspace, bwd_workspace_bytes);
  if (rc || batch->B == 0) return rc;
  bool tc = false;
  rc = choose_pairs_fwd(*p, *batch, &tc);
  PairsBwd bwd;
  if (!rc) rc = bwd.open(*p, *batch, *grads, nullptr, nullptr, nullptr, nullptr, nullptr, bwd_workspace, bwd_workspace_bytes, true);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int bi = 0; bi < bwd.n_branch; ++bi) bwd.sort(bi, st, true);
  rc = (int)cudaGetLastError();
  if (rc) return rc;
  rc = launch_chosen_fwd(tc, *p, *batch, score, row_sum, score_parts, reinterpret_cast<unsigned long long*>(act_mask), st);
  // (also after a failed forward launch: the caller may release the workspace as soon as this returns)
  const int rj = bwd.join_sorts(st);
  return rc ? rc : rj;
}

int nais_pairs_backward_presorted(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                                  const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, void* workspace,
                                  size_t workspace_bytes, nais_stream_t stream) {
  return backward_call(p, batch, score_parts, row_sum, act_mask, dscore, grads, grads, nullptr, true, workspace, workspace_bytes, stream);
}

int nais_pairs_backward_adagrad(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                                const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, const NaisAdagrad* opt,
                                void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  return backward_call(p, batch, score_parts, row_sum, act_mask, dscore, grads, grads && opt, opt, false, workspace, workspace_bytes,
                       stream);
}

// ---- nais_pairs_train_step: forward -> sigmoid + BCE -> backward (tables stepped in the segment reduce) -> dense Adagrad ----------
namespace {
inline size_t ts_al(size_t x) { return (x + 255) / 256 * 256; }
struct TrainStepLayout {
  size_t score, row_sum, parts, dscore, mask, gw1[2], gb1[2], gw2[2], gdw, gdb, gde, bwd, total;
};
TrainStepLayout train_step_layout(const NaisParams& p, const NaisPairs& b) {
  TrainStepLayout L;
  const int64_t B = b.B, cells = pairs_n_cells(b);
  const int lanes = p.dist_mode == NAIS_DIST_LATLON ? 2 : 0;
  size_t o = 0;
  L.score = o, o += ts_al((size_t)B * 4);
  L.row_sum = o, o += ts_al((size_t)p.n_branch * B * 4);
  L.parts = o, o += ts_al((size_t)p.n_branch * B * 4);
  L.dscore = o, o += ts_al((size_t)B * 4);
  L.mask = o, o += ts_al((size_t)p.n_branch * cells * 8);  // [n_branch, cells] ReLU patterns of the tcgen05 forward
  for (int bi = 0; bi < 2; ++bi) {  // per-branch MLP gradient scratch (branch 1: the disentangled layout's region MLP)
    const NaisBranch& br = p.branch[bi];
    const int ldw = br.w_poi + br.w_reg + lanes;
    const bool on = bi < p.n_branch;
    L.gw1[bi] = o, o += on ? ts_al((size_t)p.hid * ldw * 4) : 0;
    L.gb1[bi] = o, o += on ? ts_al((size_t)p.hid * 4) : 0;
    L.gw2[bi] = o, o += on ? ts_al((size_t)p.hid * 4) : 0;
  }
  L.gdw = o, o += 256;
  L.gdb = o, o += 256;
  L.gde = o, o += p.dist_mode == NAIS_DIST_KM ? ts_al((size_t)MAXD * 4) : 0;  // embed_distance row 0 (param_reduce writes D of a branch)
  L.bwd = o, o += ts_al(pairs_bwd_workspace_bytes(p, b));
  L.total = o;
  return L;
}
}  // namespace

size_t nais_pairs_train_step_workspace_bytes(const NaisParams* p, const NaisPairs* batch) {
  if (check_params(p) || !batch || batch->B < 0 || (!batch->seg_offsets && batch->H < 1)) return 0;
  if (!pairs_fused_layout(*p)) return 0;
  return train_step_layout(*p, *batch).total;
}

static int check_train_state(const NaisParams* p, const NaisAdagrad* tables, const NaisDenseAdagrad* dense) {
  if (!tables || !dense) return NAIS_ERR_NULL;
  if (!pairs_fused_layout(*p)) return NAIS_ERR_MODE;
  const bool two = pairs_disentangled(*p);
  if (p->n_branch == 1 && p->dist_mode == NAIS_DIST_KM) return NAIS_ERR_MODE;
  if (!(tables->lr >= 0.f) || !(tables->eps >= 0.f) || !(dense->lr >= 0.f) || !(dense->eps >= 0.f)) return NAIS_ERR_MODE;
  if (!dense->sum_w1 || !dense->sum_b1 || !dense->sum_w2) return NAIS_ERR_NULL;
  if (p->dist_mode == NAIS_DIST_LATLON && (!dense->sum_dist_w || !dense->sum_dist_b)) return NAIS_ERR_NULL;
  if (two && (!dense->sum_region_w1 || !dense->sum_region_b1 || !dense->sum_region_w2)) return NAIS_ERR_NULL;
  if (two && p->dist_mode == NAIS_DIST_KM && !dense->sum_dist_embed) return NAIS_ERR_NULL;
  return 0;
}

// One optimizer step in its workspace (arguments already checked): the forward's kernel choice, the backward's context with the
// gradient scratch of the MLP / distance layer (which also tells the backward which lists it needs), and per branch the dense
// Adagrad of those tensors.  That Adagrad rides behind the kernel that finishes their gradients, next to the table reduces: one
// launch less on the step's chain of dependent launches.  Two branches: branch 1's also steps row 0 of embed_distance, whose
// gradient both branches' param_reduce add up.
struct TrainStep {
  TrainStepLayout L;
  char* base;
  bool fwd_tc = false;
  unsigned long long* mask;
  DenseAdagradLaunch da[2];
  PairsBwd bwd;
  float* f(size_t off) const { return reinterpret_cast<float*>(base + off); }
};

static int open_train_step(TrainStep& s, const NaisParams* p, const NaisPairs* batch, const NaisAdagrad* tables,
                           const NaisDenseAdagrad* dense, void* workspace, size_t workspace_bytes) {
  const TrainStepLayout& L = s.L = train_step_layout(*p, *batch);
  if (workspace_bytes < L.total) return NAIS_ERR_WORKSPACE;
  s.base = reinterpret_cast<char*>(workspace);
  NaisGrads g = {};
  for (int bi = 0; bi < p->n_branch; ++bi) {
    g.w1[bi] = s.f(L.gw1[bi]);
    g.b1[bi] = s.f(L.gb1[bi]);
    g.w2[bi] = s.f(L.gw2[bi]);
  }
  if (p->dist_mode == NAIS_DIST_LATLON) {
    g.dist_w = s.f(L.gdw);
    g.dist_b = s.f(L.gdb);
  }
  if (p->dist_mode == NAIS_DIST_KM) g.dist_embed = s.f(L.gde);
  const NaisBranch& br = p->branch[0];
  const int lanes = p->dist_mode == NAIS_DIST_LATLON ? 2 : 0, ldw = br.w_poi + br.w_reg + lanes;
  s.da[0] = {{const_cast<float*>(br.w1), const_cast<float*>(br.b1), const_cast<float*>(br.w2),
              lanes ? const_cast<float*>(p->dist_w) : nullptr, lanes ? const_cast<float*>(p->dist_b) : nullptr},
             {dense->sum_w1, dense->sum_b1, dense->sum_w2, dense->sum_dist_w, dense->sum_dist_b},
             {g.w1[0], g.b1[0], g.w2[0], g.dist_w, g.dist_b},
             {p->hid * ldw, p->hid, p->hid, 4, 2},
             dense->lr, dense->eps};
  if (p->n_branch == 2) {
    const NaisBranch& r = p->branch[1];
    const bool km = p->dist_mode == NAIS_DIST_KM;
    s.da[1] = {{const_cast<float*>(r.w1), const_cast<float*>(r.b1), const_cast<float*>(r.w2), km ? const_cast<float*>(p->dist_embed) : nullptr,
                nullptr},
               {dense->sum_region_w1, dense->sum_region_b1, dense->sum_region_w2, dense->sum_dist_embed, nullptr},
               {g.w1[1], g.b1[1], g.w2[1], g.dist_embed, nullptr},
               {p->hid * (r.w_poi + r.w_reg), p->hid, p->hid, r.w_poi + r.w_reg, 0},
               dense->lr, dense->eps};
  }
  const int rc = choose_pairs_fwd(*p, *batch, &s.fwd_tc);
  if (rc) return rc;
  s.mask = (s.fwd_tc && p->hid <= 64) ? reinterpret_cast<unsigned long long*>(s.base + L.mask) : nullptr;
  return s.bwd.open(*p, *batch, g, tables, s.f(L.parts), s.f(L.row_sum), s.mask, s.f(L.dscore), s.base + L.bwd, workspace_bytes - L.bwd,
                    true);
}

// The backward's id sorts depend on the batch only: forked onto the side streams, they run next to what `st` runs after them.
static int train_step_sorts(const TrainStep& s, cudaStream_t st) {
  for (int bi = 0; bi < s.bwd.n_branch; ++bi) s.bwd.sort(bi, st, true);
  return (int)cudaGetLastError();
}

// The loss a training step takes on its [B] scores: sigmoid + BCE on `label` (weights `row_weight`, NULL = batch mean), or, with
// bpr_num_neg > 0, BPR over groups of 1 + bpr_num_neg rows (weights `group_weight`, NULL = mean over pairs).
struct StepLoss {
  const float* label;
  const float* row_weight;
  int bpr_num_neg;
  const float* group_weight;
};

// forward -> loss -> backward (MLP / distance-layer gradients to scratch, tables stepped in place).  wait_sorted0: the lists were
// sorted by this step's train_step_sorts and not joined since.
static int train_step_rest(const TrainStep& s, const StepLoss& sl, float* loss, float* score_out, cudaStream_t st, bool wait_sorted0) {
  int rc = launch_chosen_fwd(s.fwd_tc, s.bwd.p, s.bwd.b, s.f(s.L.score), s.f(s.L.row_sum), s.f(s.L.parts), s.mask, st);
  if (rc) return rc;
  if (score_out) {
    cudaError_t e = cudaMemcpyAsync(score_out, s.f(s.L.score), (size_t)s.bwd.b.B * 4, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  rc = sl.bpr_num_neg > 0 ? launch_bpr_dscore(s.f(s.L.score), sl.group_weight, s.bwd.b.B, sl.bpr_num_neg, s.f(s.L.dscore), loss, st)
                          : launch_bce_dscore(s.f(s.L.score), sl.label, sl.row_weight, s.bwd.b.B, s.f(s.L.dscore), loss, st);
  for (int bi = 0; bi < s.bwd.n_branch && !rc; ++bi) rc = s.bwd.finish(bi, st, wait_sorted0, &s.da[bi]);
  return rc;
}

// nais_pairs_train_step / nais_pairs_train_step_bpr: `bpr` NULL = the BCE step on `label`.
static int pairs_train_step(const NaisParams* p, const NaisPairs* batch, const float* label, const float* row_weight,
                            const NaisBprLoss* bpr, const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* loss,
                            float* score_out, void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  rc = check_pairs(p, batch);
  if (rc) return rc;
  if (bpr && (bpr->num_neg < 1 || batch->B % (1 + (int64_t)bpr->num_neg) != 0)) return NAIS_ERR_SHAPE;
  if (!loss) return NAIS_ERR_NULL;
  rc = check_train_state(p, tables, dense);
  if (rc) return rc;
  if (batch->B == 0) return 0;
  if ((!bpr && !label) || !workspace) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  TrainStep s;
  rc = open_train_step(s, p, batch, tables, dense, workspace, workspace_bytes);
  if (!rc) rc = train_step_sorts(s, st);
  const StepLoss sl = {label, row_weight, bpr ? bpr->num_neg : 0, bpr ? bpr->group_weight : nullptr};
  return rc ? rc : train_step_rest(s, sl, loss, score_out, st, true);
}

int nais_pairs_train_step(const NaisParams* p, const NaisPairs* batch, const float* label, const float* row_weight,
                          const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* loss, float* score_out, void* workspace,
                          size_t workspace_bytes, nais_stream_t stream) {
  return pairs_train_step(p, batch, label, row_weight, nullptr, tables, dense, loss, score_out, workspace, workspace_bytes, stream);
}

int nais_pairs_train_step_bpr(const NaisParams* p, const NaisPairs* batch, const NaisBprLoss* bpr, const NaisAdagrad* tables,
                              const NaisDenseAdagrad* dense, float* loss, float* score_out, void* workspace, size_t workspace_bytes,
                              nais_stream_t stream) {
  if (!bpr) return NAIS_ERR_NULL;
  return pairs_train_step(p, batch, nullptr, nullptr, bpr, tables, dense, loss, score_out, workspace, workspace_bytes, stream);
}

// ---- nais_train_users: the reference's one-user-per-step schedule, a list of users per call ---------------------------------------
namespace {
// the segment structure of a ONE-segment batch (H history items, R rows): offsets + the tile table, written on the device
__global__ void single_segment_kernel(int H, int R, int rpt, int n_tiles, int64_t* seg_offsets, int64_t* row_offsets, int64_t* cell_offsets,
                                      int32_t* tile_seg, int64_t* tile_row0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    seg_offsets[0] = 0, seg_offsets[1] = H;
    row_offsets[0] = 0, row_offsets[1] = R;
    cell_offsets[0] = 0, cell_offsets[1] = (int64_t)R * H;
  }
  if (i < n_tiles) {
    tile_seg[i] = 0;
    tile_row0[i] = (int64_t)i * rpt;
  }
}
struct UsersLayout {
  size_t seg, row, cell, tseg, trow, tgt, label, treg, tco, step, total;
};
inline int host_rows_per_tile(int H) {
  int r = H <= 128 ? 128 / (H > 0 ? H : 1) : 1;
  return r > 16 ? 16 : r;
}
NaisPairs max_user_batch(int max_hist, int num_ng) {
  NaisPairs b;
  memset(&b, 0, sizeof(b));
  static const int64_t dummy[2] = {0, 0};
  b.seg_offsets = dummy;  // (marks the segmented layout: only sizes are read from this struct)
  b.n_seg = 1;
  b.B = (int64_t)max_hist * (num_ng + 1);
  b.n_cells = b.B * max_hist;
  b.n_tiles = b.B;  // (an upper bound for every history length)
  return b;
}
UsersLayout users_layout(const NaisParams& p, int max_hist, int num_ng) {
  UsersLayout L;
  const NaisPairs b = max_user_batch(max_hist, num_ng);
  size_t o = 0;
  L.seg = o, o += 256;
  L.row = o, o += 256;
  L.cell = o, o += 256;
  L.tseg = o, o += ts_al((size_t)b.n_tiles * 4);
  L.trow = o, o += ts_al((size_t)b.n_tiles * 8);
  L.tgt = o, o += ts_al((size_t)b.B * 8);
  L.label = o, o += ts_al((size_t)b.B * 4);
  L.treg = o, o += ts_al((size_t)b.B * 8);
  L.tco = o, o += ts_al((size_t)b.B * 8);
  L.step = o, o += train_step_layout(p, b).total;
  L.total = o;
  return L;
}

// The preparation stream of nais_train_users: one per device, created on first use (like the side streams of the backward).
std::mutex g_prep_mu;
cudaStream_t prep_stream() {
  static cudaStream_t pool[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(g_prep_mu);
  if (!pool[dev] && cudaStreamCreateWithFlags(&pool[dev], cudaStreamNonBlocking) != cudaSuccess) pool[dev] = nullptr;
  return pool[dev];
}
}  // namespace

size_t nais_train_users_workspace_bytes(const NaisParams* p, int32_t max_hist, int32_t num_ng) {
  if (check_params(p) || !pairs_fused_layout(*p) || max_hist < 1 || num_ng < 0) return 0;
  return 2 * users_layout(*p, max_hist, num_ng).total;  // two users in flight: one being prepared, one being stepped
}

int nais_train_users(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices, const int64_t* entry_region,
                     const float* entry_coords, const int32_t* poi_region, const float* poi_coords, const int64_t* host_users,
                     int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* losses,
                     void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  return nais_train_users_centred(p, host_indptr, n_rows, indices, entry_region, entry_coords, poi_region, poi_coords, host_users, n_users,
                                  num_ng, seed, tables, dense, losses, workspace, workspace_bytes, 0.f, 0.f, stream);
}

int nais_train_users_centred(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                             const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region, const float* poi_coords,
                             const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables,
                             const NaisDenseAdagrad* dense, float* losses, void* workspace, size_t workspace_bytes, float center_lat,
                             float center_lon, nais_stream_t stream) {
  if (p && p->dropout_p > 0.f) return NAIS_ERR_MODE;  // one seed for every step would repeat the mask: nais_train_users_dropout
  return nais_train_users_dropout(p, host_indptr, n_rows, indices, entry_region, entry_coords, poi_region, poi_coords, host_users, n_users,
                                  num_ng, seed, tables, dense, losses, workspace, workspace_bytes, center_lat, center_lon, nullptr, stream);
}

// The body of nais_train_users_dropout (bpr = false: the batch-mean BCE per user) and nais_train_users_bpr (the mean BPR loss over
// the user's H * num_ng pairs: groups of 1 + num_ng rows, as the sampler writes them).
static int train_users(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices, const int64_t* entry_region,
                       const float* entry_coords, const int32_t* poi_region, const float* poi_coords, const int64_t* host_users,
                       int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables, const NaisDenseAdagrad* dense,
                       float* losses, void* workspace, size_t workspace_bytes, float center_lat, float center_lon,
                       const uint64_t* host_dropout_seeds, bool bpr, nais_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  rc = check_train_state(p, tables, dense);
  if (rc) return rc;
  if (n_users < 0 || num_ng < (bpr ? 1 : 0)) return NAIS_ERR_SHAPE;
  if (p->dropout_p > 0.f && !host_dropout_seeds) return NAIS_ERR_NULL;
  if (n_users == 0) return 0;
  if (!host_indptr || !indices || !host_users || !losses || !workspace) return NAIS_ERR_NULL;
  bool need_reg = false;
  for (int i = 0; i < p->n_branch; ++i) need_reg |= p->branch[i].w_reg > 0;
  const bool need_co = p->dist_mode != NAIS_DIST_NONE;
  if ((need_reg && (!entry_region || !poi_region)) || (need_co && (!entry_coords || !poi_coords))) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  int max_hist = 0;
  for (int i = 0; i < n_users; ++i) {
    const int64_t u = host_users[i];
    if (u < 0 || u >= n_rows) return NAIS_ERR_SHAPE;
    const int64_t H = host_indptr[u + 1] - host_indptr[u];
    if (H < 0 || H > 0x7fffffff / (num_ng + 2)) return NAIS_ERR_SHAPE;
    if ((int)H > max_hist) max_hist = (int)H;
  }
  if (max_hist == 0) return (int)cudaMemsetAsync(losses, 0, (size_t)n_users * 4, static_cast<cudaStream_t>(stream));
  if ((int64_t)max_hist * (num_ng + 1) >= p->item_num) return NAIS_ERR_SHAPE;  // not enough unvisited POIs to draw from
  const UsersLayout L = users_layout(*p, max_hist, num_ng);
  if (workspace_bytes < 2 * L.total) return NAIS_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // One user per optimizer step is a chain of small dependent launches (GPU latency, not throughput).  What depends on the batch
  // only — the segment structure, the sampler and the id sorts of the backward — is enqueued one user AHEAD on a library-owned
  // preparation stream into the other half of the workspace; the step itself (forward, loss, backward on the sorted lists, Adagrad)
  // stays on the caller's stream.  Same kernels on the same inputs in the same order per user: results do not change.
  cudaStream_t ps = prep_stream();
  if (!ps) return (int)cudaErrorUnknown;
  cudaEvent_t prepared[2] = {nullptr, nullptr}, stepped[2] = {nullptr, nullptr}, begin = nullptr;
  bool ev_ok = cudaEventCreateWithFlags(&begin, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; i < 2 && ev_ok; ++i)
    ev_ok = cudaEventCreateWithFlags(&prepared[i], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&stepped[i], cudaEventDisableTiming) == cudaSuccess;
  auto release = [&]() {  // (destroying an event that is still pending is legal: its resources go when it completes)
    if (begin) cudaEventDestroy(begin);
    for (int i = 0; i < 2; ++i) {
      if (prepared[i]) cudaEventDestroy(prepared[i]);
      if (stepped[i]) cudaEventDestroy(stepped[i]);
    }
  };
  if (!ev_ok) {
    release();
    return (int)cudaErrorUnknown;
  }
  auto bail = [&](int code) {  // order the caller's stream after everything the preparation stream still holds, then report
    if (cudaEventRecord(begin, ps) == cudaSuccess) cudaStreamWaitEvent(st, begin, 0);
    release();
    return code;
  };
  struct UserBatch {
    NaisPairs b;
    const float* label;
    char* step;
  };
  auto buffers = [&](int i, int slot, UserBatch& ub) {  // the batch of host_users[i] in workspace half `slot` (H > 0)
    char* base = reinterpret_cast<char*>(workspace) + (size_t)slot * L.total;
    auto I64 = [&](size_t off) { return reinterpret_cast<int64_t*>(base + off); };
    const int64_t u = host_users[i], a = host_indptr[u];
    const int H = (int)(host_indptr[u + 1] - a);
    const int R = H * (num_ng + 1), rpt = host_rows_per_tile(H), n_tiles = (R + rpt - 1) / rpt;
    NaisPairs& b = ub.b;
    memset(&b, 0, sizeof(b));
    b.hist = indices + a;
    b.tgt = I64(L.tgt);
    b.hreg = need_reg ? entry_region + a : nullptr;
    b.treg = need_reg ? I64(L.treg) : nullptr;
    b.B = R;
    b.n_seg = 1;
    b.seg_offsets = I64(L.seg);
    b.row_offsets = I64(L.row);
    b.seg_cell_offsets = I64(L.cell);
    b.tile_seg = reinterpret_cast<int32_t*>(base + L.tseg);
    b.tile_row0 = I64(L.trow);
    b.n_tiles = n_tiles;
    b.n_cells = (int64_t)R * H;
    b.hist_coords = need_co ? entry_coords + 2 * a : nullptr;
    b.tgt_coords = need_co ? reinterpret_cast<float*>(base + L.tco) : nullptr;
    b.center_lat = center_lat;
    b.center_lon = center_lon;
    ub.label = reinterpret_cast<float*>(base + L.label);
    ub.step = base + L.step;
  };
  auto prepare = [&](int i, int slot) -> int {  // on the preparation stream
    UserBatch ub;
    buffers(i, slot, ub);
    const int64_t u = host_users[i], a = host_indptr[u];
    const int H = (int)(host_indptr[u + 1] - a);
    char* base = reinterpret_cast<char*>(workspace) + (size_t)slot * L.total;
    single_segment_kernel<<<((int)ub.b.n_tiles + 255) / 256, 256, 0, ps>>>(
        H, (int)ub.b.B, host_rows_per_tile(H), (int)ub.b.n_tiles, const_cast<int64_t*>(ub.b.seg_offsets), const_cast<int64_t*>(ub.b.row_offsets),
        const_cast<int64_t*>(ub.b.seg_cell_offsets), const_cast<int32_t*>(ub.b.tile_seg), const_cast<int64_t*>(ub.b.tile_row0));
    NAIS_COUNT_LAUNCH(1);
    int r = launch_sample_batch(ub.b.seg_offsets, indices + a, 1, ub.b.row_offsets, num_ng, p->item_num, need_reg ? poi_region : nullptr,
                                need_co ? poi_coords : nullptr, seed + (uint64_t)u, H, const_cast<int64_t*>(ub.b.tgt),
                                reinterpret_cast<float*>(base + L.label), need_reg ? const_cast<int64_t*>(ub.b.treg) : nullptr,
                                need_co ? const_cast<float*>(ub.b.tgt_coords) : nullptr, ps);
    TrainStep s;  // the step's id sorts, joined to the preparation stream (the step waits for `prepared`)
    if (!r) r = open_train_step(s, p, &ub.b, tables, dense, ub.step, L.total - L.step);
    if (!r) r = train_step_sorts(s, ps);
    return r ? r : s.bwd.join_sorts(ps);
  };
  // users with a history, in order; the others only get a zero loss
  int next = 0;
  auto advance = [&](int from) {
    while (from < n_users && host_indptr[host_users[from] + 1] == host_indptr[host_users[from]]) ++from;
    return from;
  };
  for (int i = 0; i < n_users; ++i)
    if (host_indptr[host_users[i] + 1] == host_indptr[host_users[i]]) {
      cudaError_t e = cudaMemsetAsync(losses + i, 0, 4, st);
      if (e != cudaSuccess) return bail((int)e);
    }
  // the preparation stream starts after the work already in the caller's stream (the parameters, the CSR arrays)
  if (cudaEventRecord(begin, st) != cudaSuccess || cudaStreamWaitEvent(ps, begin, 0) != cudaSuccess) return bail((int)cudaErrorUnknown);
  next = advance(0);
  int slot = 0;
  if (next < n_users) {
    rc = prepare(next, slot);
    if (rc) return bail(rc);
    cudaEventRecord(prepared[slot], ps);
  }
  int done = 0;  // steps enqueued so far
  while (next < n_users) {
    const int cur = next, cur_slot = slot;
    next = advance(cur + 1);
    slot ^= 1;
    if (next < n_users) {  // prepare the next user into the other half: free once the step before `cur` has finished with it
      if (done >= 1) cudaStreamWaitEvent(ps, stepped[slot], 0);
      rc = prepare(next, slot);
      if (rc) return bail(rc);
      cudaEventRecord(prepared[slot], ps);
    }
    UserBatch ub;
    buffers(cur, cur_slot, ub);
    NaisParams pu = *p;  // (the id sorts of the preparation depend on the batch only, not on the dropout seed)
    if (p->dropout_p > 0.f) pu.dropout_seed = host_dropout_seeds[cur];
    cudaStreamWaitEvent(st, prepared[cur_slot], 0);
    TrainStep s;  // the rest of the step, on the lists the preparation sorted
    rc = open_train_step(s, &pu, &ub.b, tables, dense, ub.step, L.total - L.step);
    const StepLoss sl = {ub.label, nullptr, bpr ? num_ng : 0, nullptr};
    if (!rc) rc = train_step_rest(s, sl, losses + cur, nullptr, st, false);
    if (rc) return bail(rc);
    cudaEventRecord(stepped[cur_slot], st);
    ++done;
  }
  cudaError_t e = cudaGetLastError();
  release();
  return e == cudaSuccess ? 0 : (int)e;
}

int nais_train_users_dropout(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                             const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region, const float* poi_coords,
                             const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables,
                             const NaisDenseAdagrad* dense, float* losses, void* workspace, size_t workspace_bytes, float center_lat,
                             float center_lon, const uint64_t* host_dropout_seeds, nais_stream_t stream) {
  return train_users(p, host_indptr, n_rows, indices, entry_region, entry_coords, poi_region, poi_coords, host_users, n_users, num_ng, seed,
                     tables, dense, losses, workspace, workspace_bytes, center_lat, center_lon, host_dropout_seeds, false, stream);
}

int nais_train_users_bpr(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                         const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region, const float* poi_coords,
                         const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables,
                         const NaisDenseAdagrad* dense, float* losses, void* workspace, size_t workspace_bytes, float center_lat,
                         float center_lon, const uint64_t* host_dropout_seeds, nais_stream_t stream) {
  return train_users(p, host_indptr, n_rows, indices, entry_region, entry_coords, poi_region, poi_coords, host_users, n_users, num_ng, seed,
                     tables, dense, losses, workspace, workspace_bytes, center_lat, center_lon, host_dropout_seeds, true, stream);
}

static int check_fullrank(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                          int64_t poi_end, int precision) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!cat || !users) return NAIS_ERR_NULL;
  if (users->n_users < 0 || poi_begin < 0 || poi_end < poi_begin || poi_end > p->item_num) return NAIS_ERR_SHAPE;
  if (poi_begin < cat->row_base || poi_end > cat->row_base + cat->n_rows) return NAIS_ERR_SHAPE;
  if (users->n_users && (!users->offsets || !users->items)) return NAIS_ERR_NULL;
  bool need_reg = false;
  for (int i = 0; i < p->n_branch; ++i) need_reg |= p->branch[i].w_reg > 0;
  const bool work = users->n_users > 0 && poi_end > poi_begin;
  if (work && need_reg && (!cat->region || !users->region)) return NAIS_ERR_NULL;
  if (work && p->dist_mode != NAIS_DIST_NONE && (!cat->coords || !users->coords)) return NAIS_ERR_NULL;
  const int prec = precision & NAIS_PREC_MASK;
  if (precision & ~(NAIS_PREC_MASK | NAIS_PREC_FLAG_GENERIC | NAIS_PREC_FLAG_ONE_CTA)) return NAIS_ERR_MODE;
  if (prec < NAIS_PREC_FP32 || prec > NAIS_PREC_TC_AUTO) return NAIS_ERR_MODE;
  if (prec != NAIS_PREC_FP32 && !tc_supported(*p, precision)) return NAIS_ERR_SHAPE;
  return 0;
}

size_t nais_fullrank_workspace_bytes(const NaisParams* p, int32_t n_users, int64_t nnz, int64_t poi_begin,
                                     int64_t poi_end, int32_t k, int32_t precision) {
  if (check_params(p) || n_users < 0 || poi_end < poi_begin || k < 1) return 0;
  if ((precision & NAIS_PREC_MASK) != NAIS_PREC_FP32) return fullrank_tc_workspace_bytes(*p, n_users, nnz, poi_begin, poi_end, k, precision);
  return fp32_workspace_bytes(n_users, poi_begin, poi_end, k);
}

size_t nais_fullrank_plan_bytes(const NaisParams* p, int64_t poi_begin, int64_t poi_end, int32_t precision) {
  if (check_params(p) || poi_end < poi_begin || (precision & NAIS_PREC_MASK) == NAIS_PREC_FP32) return 0;
  return fullrank_tc_plan_bytes(*p, poi_begin, poi_end, precision);
}

size_t nais_fullrank_planned_workspace_bytes(const NaisParams* p, int32_t n_users, int64_t nnz, int64_t poi_begin, int64_t poi_end,
                                             int32_t k, int32_t precision) {
  if (check_params(p) || n_users < 0 || poi_end < poi_begin || k < 1) return 0;
  if ((precision & NAIS_PREC_MASK) != NAIS_PREC_FP32)
    return fullrank_tc_call_workspace_bytes(*p, n_users, nnz, poi_begin, poi_end, k, precision) + 1024 + (size_t)n_users * 8;
  return fp32_workspace_bytes(n_users, poi_begin, poi_end, k) + (size_t)n_users * k * 12 + 512;  // + score / id staging for out_keys
}

int nais_fullrank_prepare(const NaisParams* p, const NaisCatalog* cat, int64_t poi_begin, int64_t poi_end, int32_t precision,
                          void* plan, size_t plan_bytes, nais_stream_t stream) {
  NaisUsers none = {};
  int rc = check_fullrank(p, cat, &none, poi_begin, poi_end, precision);
  if (rc) return rc;
  if ((precision & NAIS_PREC_MASK) == NAIS_PREC_FP32 || poi_end == poi_begin) return 0;  // nothing to precompute
  if (!plan) return NAIS_ERR_NULL;
  if (!aligned16(plan)) return NAIS_ERR_ALIGN;
  const NaisBranch& br = p->branch[0];
  if (br.w_reg > 0 && !cat->region) return NAIS_ERR_NULL;
  return fullrank_tc_prepare(*p, *cat, poi_begin, poi_end, precision, plan, plan_bytes, static_cast<cudaStream_t>(stream));
}

// Geo re-ranking arguments (nais_fullrank_topk_geo_planned): checked before any CUDA call
static int check_geo(const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin, int64_t poi_end, const NaisGeoMix* geo) {
  if (!geo) return NAIS_ERR_NULL;
  if (!(geo->a > 0.f) || !isfinite(geo->a) || !isfinite(geo->b) || !isfinite(geo->alpha)) return NAIS_ERR_MODE;
  if (users->n_users > 0 && poi_end > poi_begin && (!cat->coords || !users->coords || !geo->user_logmax)) return NAIS_ERR_NULL;
  return 0;
}

static int fullrank_topk_planned_impl(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                                      int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, const void* plan,
                                      size_t plan_bytes, const NaisGeoMix* geo, uint64_t* out_keys, float* out_score, int32_t* out_id,
                                      void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_fullrank(p, cat, users, poi_begin, poi_end, precision);
  if (rc) return rc;
  if (k < 1 || k > KCAP) return NAIS_ERR_SHAPE;
  if (geo && (rc = check_geo(cat, users, poi_begin, poi_end, geo))) return rc;
  if (users->n_users == 0) return 0;
  if ((!out_score) != (!out_id) || (!out_score && !out_keys) || !workspace) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  GeoMixArgs gm = {};
  if (geo) gm = GeoMixArgs{logf(geo->a), geo->b, geo->alpha, geo->user_logmax};
  const GeoMixArgs* gp = geo ? &gm : nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(out_keys);
  const size_t n = (size_t)users->n_users * k;
  if (poi_end == poi_begin) {  // empty shard: every list is padding
    if (out_score) {
      fill_empty_topk_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(out_score, out_id, n);
      NAIS_COUNT_LAUNCH(1);
    }
    if (keys) {
      cudaError_t e = cudaMemsetAsync(keys, 0, n * 8, st);
      if (e != cudaSuccess) return (int)e;
    }
    return (int)cudaGetLastError();
  }
  if ((precision & NAIS_PREC_MASK) != NAIS_PREC_FP32)
    return fullrank_tc_run(*p, *cat, *users, poi_begin, poi_end, k, exclude_history, precision, plan, plan_bytes, keys, out_score,
                           out_id, nullptr, workspace, workspace_bytes, st, gp);
  // FP32 kernel: no plan.  It writes score / id; keys (if wanted) are re-packed from them.
  float* sc = out_score;
  int32_t* id = out_id;
  char* rest = reinterpret_cast<char*>(workspace);
  size_t rest_bytes = workspace_bytes;
  if (!sc) {  // stage score / id at the head of the workspace
    const size_t head = (n * 8 + 255) & ~size_t(255);
    if (workspace_bytes < head) return NAIS_ERR_WORKSPACE;
    sc = reinterpret_cast<float*>(workspace);
    id = reinterpret_cast<int32_t*>(sc + n);
    rest += head;
    rest_bytes -= head;
  }
  rc = launch_fullrank_fp32(*p, *cat, *users, poi_begin, poi_end, k, exclude_history, sc, id, nullptr, rest, rest_bytes, st, gp);
  if (rc || !keys) return rc;
  pack_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sc, id, n, keys);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

int nais_fullrank_topk_planned(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                               int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, const void* plan,
                               size_t plan_bytes, uint64_t* out_keys, float* out_score, int32_t* out_id, void* workspace,
                               size_t workspace_bytes, nais_stream_t stream) {
  return fullrank_topk_planned_impl(p, cat, users, poi_begin, poi_end, k, exclude_history, precision, plan, plan_bytes, nullptr, out_keys,
                                    out_score, out_id, workspace, workspace_bytes, stream);
}

int nais_fullrank_topk_geo_planned(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                                   int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, const void* plan,
                                   size_t plan_bytes, const NaisGeoMix* geo, uint64_t* out_keys, float* out_score, int32_t* out_id,
                                   void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  if (!geo) return NAIS_ERR_NULL;
  return fullrank_topk_planned_impl(p, cat, users, poi_begin, poi_end, k, exclude_history, precision, plan, plan_bytes, geo, out_keys,
                                    out_score, out_id, workspace, workspace_bytes, stream);
}

int nais_topk_merge_keys(const uint64_t* in_keys, int64_t user_stride, int64_t list_stride, int32_t n_users, int32_t n_lists,
                         int32_t k, uint64_t* out_keys, float* out_score, int32_t* out_id, nais_stream_t stream) {
  if (n_users < 0 || n_lists < 1 || k < 1 || k > KCAP || user_stride < k || list_stride < k) return NAIS_ERR_SHAPE;
  if (n_users == 0) return 0;
  if (!in_keys || (!out_score) != (!out_id) || (!out_score && !out_keys)) return NAIS_ERR_NULL;
  if (merge_scratch_lists(n_lists, k) != 0) return NAIS_ERR_SHAPE;  // one level: n_lists * k <= 8192 (shards of a node, not tiles)
  return launch_topk_merge_keys_multi(reinterpret_cast<const unsigned long long*>(in_keys), nullptr, user_stride, list_stride, n_users,
                                      n_lists, k, reinterpret_cast<unsigned long long*>(out_keys), out_score, out_id,
                                      static_cast<cudaStream_t>(stream));
}

int nais_poll_bad_index(int32_t* host_flag, nais_stream_t stream) {
  if (!host_flag) return NAIS_ERR_NULL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int* flag = bad_index_flag();
  if (!flag) return (int)cudaGetLastError();
  cudaError_t e = cudaMemcpyAsync(host_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(flag, 0, sizeof(int), st);
  return (int)e;
}

int nais_fullrank_topk(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                       int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, float* out_score,
                       int32_t* out_id, void* workspace, size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_fullrank(p, cat, users, poi_begin, poi_end, precision);
  if (rc) return rc;
  if (k < 1 || k > KCAP) return NAIS_ERR_SHAPE;
  if (users->n_users && (!out_score || !out_id || !workspace)) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (users->n_users && poi_end == poi_begin) {  // empty shard: every list is padding
    const size_t n = (size_t)users->n_users * k;
    fill_empty_topk_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(out_score, out_id, n);
    NAIS_COUNT_LAUNCH(1);
    return (int)cudaGetLastError();
  }
  if ((precision & NAIS_PREC_MASK) == NAIS_PREC_FP32)
    return launch_fullrank_fp32(*p, *cat, *users, poi_begin, poi_end, k, exclude_history, out_score, out_id, nullptr,
                                workspace, workspace_bytes, st);
  return launch_fullrank_tc(*p, *cat, *users, poi_begin, poi_end, k, exclude_history, precision, out_score, out_id,
                            nullptr, workspace, workspace_bytes, st);
}

int nais_fullrank_scores(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                         int64_t poi_end, int32_t precision, float* all_scores, void* workspace,
                         size_t workspace_bytes, nais_stream_t stream) {
  int rc = check_fullrank(p, cat, users, poi_begin, poi_end, precision);
  if (rc) return rc;
  if (users->n_users && (!all_scores || !workspace)) return NAIS_ERR_NULL;
  if (!aligned16(workspace)) return NAIS_ERR_ALIGN;
  // top-1 lists are produced into the head of the workspace and ignored
  const size_t head = ((size_t)users->n_users * (sizeof(float) + sizeof(int32_t)) + 255) & ~size_t(255);
  if (workspace_bytes < head) return NAIS_ERR_WORKSPACE;
  float* sc = reinterpret_cast<float*>(workspace);
  int32_t* id = reinterpret_cast<int32_t*>(sc + users->n_users);
  char* rest = reinterpret_cast<char*>(workspace) + head;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((precision & NAIS_PREC_MASK) == NAIS_PREC_FP32)
    return launch_fullrank_fp32(*p, *cat, *users, poi_begin, poi_end, 1, 0, sc, id, all_scores, rest,
                                workspace_bytes - head, st);
  return launch_fullrank_tc(*p, *cat, *users, poi_begin, poi_end, 1, 0, precision, sc, id, all_scores, rest,
                            workspace_bytes - head, st);
}

int nais_hits_at_k(const int32_t* rec, int32_t n_users, int32_t k_rec, const int64_t* pos_offsets, const int32_t* pos_items,
                   const int32_t* k_list, int32_t n_k, int32_t* hits, nais_stream_t stream) {
  if (n_users < 0 || k_rec < 1 || n_k < 1) return NAIS_ERR_SHAPE;
  if (n_users == 0) return 0;
  if (!rec || !pos_offsets || !k_list || !hits) return NAIS_ERR_NULL;
  const int64_t threads = (int64_t)n_users * 32;
  hits_at_k_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rec, n_users, k_rec, pos_offsets,
                                                                                                  pos_items, k_list, n_k, hits);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

int nais_powerlaw_logscore(const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin, int64_t poi_end, float a, float b,
                           float* out_logg, nais_stream_t stream) {
  if (!cat || !users) return NAIS_ERR_NULL;
  if (users->n_users < 0 || poi_begin < cat->row_base || poi_end < poi_begin || poi_end > cat->row_base + cat->n_rows) return NAIS_ERR_SHAPE;
  if (!(a > 0.f)) return NAIS_ERR_MODE;
  if (users->n_users == 0 || poi_end == poi_begin) return 0;
  if (!cat->coords || !users->coords || !users->offsets || !out_logg) return NAIS_ERR_NULL;
  if ((poi_end - poi_begin + 255) / 256 > 65535) return NAIS_ERR_SHAPE;  // > 16.7 M candidates in one call: pass sub-ranges
  dim3 grid((unsigned)users->n_users, (unsigned)((poi_end - poi_begin + 255) / 256));
  powerlaw_logscore_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*cat, *users, poi_begin, poi_end, logf(a), b, out_logg);
  NAIS_COUNT_LAUNCH(1);
  return (int)cudaGetLastError();
}

int nais_powerlaw_logmax(const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin, int64_t poi_end, float a, float b,
                         int32_t exclude_history, float* out_logmax, nais_stream_t stream) {
  if (!cat || !users) return NAIS_ERR_NULL;
  if (users->n_users < 0 || poi_begin < cat->row_base || poi_end < poi_begin || poi_end > cat->row_base + cat->n_rows) return NAIS_ERR_SHAPE;
  if (!(a > 0.f) || !isfinite(a) || !isfinite(b)) return NAIS_ERR_MODE;
  if (users->n_users == 0) return 0;
  if (!out_logmax || !users->offsets) return NAIS_ERR_NULL;
  if (poi_end > poi_begin && (!cat->coords || !users->coords || (exclude_history && !users->items))) return NAIS_ERR_NULL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  fill_float_kernel<<<(users->n_users + 255) / 256, 256, 0, st>>>(out_logmax, users->n_users, -INFINITY);
  NAIS_COUNT_LAUNCH(1);
  if (poi_end > poi_begin) {
    const int64_t blocks = (poi_end - poi_begin + 255) / 256;
    dim3 grid((unsigned)users->n_users, (unsigned)(blocks < 64 ? blocks : 64));
    powerlaw_logmax_kernel<<<grid, 256, 0, st>>>(*cat, *users, poi_begin, poi_end, logf(a), b, exclude_history ? 1 : 0, out_logmax);
    NAIS_COUNT_LAUNCH(1);
  }
  return (int)cudaGetLastError();
}

int nais_topk_merge(const float* in_score, const int32_t* in_id, int32_t n_users, int32_t n_lists, int32_t k,
                    float* out_score, int32_t* out_id, nais_stream_t stream) {
  if (n_users < 0 || n_lists < 1 || k < 1) return NAIS_ERR_SHAPE;
  if (n_users == 0) return 0;
  if (!in_score || !in_id || !out_score || !out_id) return NAIS_ERR_NULL;
  return launch_topk_merge(nullptr, in_score, in_id, n_users, n_lists, k, out_score, out_id,
                           static_cast<cudaStream_t>(stream));
}

}  // extern "C"
