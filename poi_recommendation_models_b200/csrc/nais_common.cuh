// Shared device helpers for the NAIS kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "nais_b200.h"

namespace nais {

// launch counter (diagnostic): every kernel launch of the library goes through NAIS_COUNT_LAUNCH
extern unsigned long long g_launches;
#define NAIS_COUNT_LAUNCH(n) (__atomic_fetch_add(&::nais::g_launches, (unsigned long long)(n), __ATOMIC_RELAXED))

// Host-side caches, per device, of what the launch paths would otherwise ask the driver on every call.  The one-user-per-step
// training loop (nais_train_users) enqueues ~14 launches per ~100 us and is bound by the host's API calls
// (examples/diag_train_users_timing.py), so each launcher sets its kernel's shared-memory attributes once per device (again only
// if a call needs more than any before it) and reads compute capability / SM count from a table.
struct DeviceInfo {
  int dev, major, sms;
};
inline DeviceInfo device_info() {
  static std::atomic<int> cache[64];  // 0 = unknown, else (major << 16 | sms) + 1
  DeviceInfo d{0, 0, 148};
  if (cudaGetDevice(&d.dev) != cudaSuccess) return d;
  const bool slot = d.dev >= 0 && d.dev < 64;
  const int c = slot ? cache[d.dev].load(std::memory_order_relaxed) : 0;
  if (c) {
    d.major = (c - 1) >> 16;
    d.sms = (c - 1) & 0xffff;
    return d;
  }
  cudaDeviceGetAttribute(&d.major, cudaDevAttrComputeCapabilityMajor, d.dev);
  cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, d.dev);
  if (slot && d.major > 0 && d.sms > 0) cache[d.dev].store(((d.major << 16) | d.sms) + 1, std::memory_order_relaxed);
  return d;
}
// One of these (static) per launch site: `smem` bytes of dynamic shared memory (and the max-shared carveout) for `kernel`.
struct SmemAttrOnce {
  std::atomic<int> set[64] = {};
  template <typename K>
  cudaError_t operator()(K kernel, size_t smem, bool carveout = false) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool slot = dev >= 0 && dev < 64;
    if (slot && (int)smem <= set[dev].load(std::memory_order_relaxed) - 1) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && carveout) e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess && slot) set[dev].store((int)smem + 1, std::memory_order_relaxed);
    return e;
  }
};

// The dense Adagrad step of the MLP / distance-layer tensors (nais_pairs_train_step), as launch_pairs_bwd enqueues it right behind
// the kernel that finishes their gradients: w1, b1, w2, dist_w, dist_b (NULL param = absent).
struct DenseAdagradLaunch {
  float* param[5];
  float* sum[5];
  const float* grad[5];
  int n[5];
  float lr, eps;
};

// What one launch_pairs_bwd call enqueues (nais_bwd.cu).  The id sorts depend on the batch only, so a caller may fork them ahead:
enum BwdPhase : int {
  BWD_ALL = 0,         // the whole backward
  BWD_SORTS = 1,       // only the id sorts, ALL of them on side streams (the one-call training step forks them before its forward)
  BWD_AFTER_SORTS = 2, // the rest, on lists sorted by a BWD_SORTS call (same p, b, g, opt, ws)
  BWD_AFTER_JOIN = 3,  // BWD_AFTER_SORTS after a BWD_JOIN_SORTS (no wait of its own for the long list)
  BWD_JOIN_SORTS = 4,  // join the sort streams of a BWD_SORTS call to `stream` (so that nothing enqueued on `stream` later — or
                       // the caller's allocator — can overtake the sorts)
};

// Device address (current device) of the library's 4-byte bad-index word (nais_capi.cu); every launcher passes it to its kernel.
int* bad_index_flag();
// An id as the kernels use it: inside [0, n) or replaced by 0 with the bad-index word set (include/nais_b200.h,
// nais_poll_bad_index).  `ok` tells the caller to drop the contribution of this id (backward) instead of crediting row 0.
__device__ __forceinline__ int checked_id(long long v, int n, int* bad, bool* ok = nullptr) {
  const bool in = (unsigned long long)v < (unsigned long long)n;
  if (!in && bad) *bad = 1;
  if (ok) *ok = in;
  return in ? (int)v : 0;
}

constexpr int TC = 128;   // cells (history item x candidate pairs) per tile of the FP32 tile-GEMM
constexpr int TCP = 132;  // padded cell stride of cell-major smem rows (16B-aligned, breaks bank regularity)
constexpr int KB = 64;    // hidden units per k-block
constexpr int NT = 256;   // threads per CTA of the FP32 kernels
constexpr int HC = 32;    // history rows staged in smem per chunk
constexpr int KCAP = 128; // max k of the fused top-k
constexpr int MAXD = 256; // max embed_size

// Order-preserving float -> uint32 (larger float => larger uint).  NaN is mapped to -inf by the callers.
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
// Ranking key: score descending, then POI id ascending.  0 = "no candidate".
__device__ __forceinline__ unsigned long long make_key(float score, int id) {
  if (score != score) score = -INFINITY;
  return ((unsigned long long)f2ord(score) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)id);
}
__device__ __forceinline__ void split_key(unsigned long long key, float& score, int& id) {
  if (key == 0ull) {
    score = -INFINITY;
    id = -1;
  } else {
    score = ord2f((uint32_t)(key >> 32));
    id = (int)(0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull));
  }
}

// Descending bitonic sort of n (power of two) keys in shared memory by all threads of the CTA.
__device__ __forceinline__ void bitonic_sort_desc(unsigned long long* buf, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        int ixj = i ^ j;
        if (ixj > i) {
          unsigned long long a = buf[i], b = buf[ixj];
          bool desc_half = ((i & k) == 0);
          if (desc_half ? (a < b) : (a > b)) {
            buf[i] = b;
            buf[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

// Dropout keep-mask (see NaisParams::dropout_p): counter-based, so forward and backward regenerate the same mask.
__host__ __device__ __forceinline__ uint32_t dropout_bits(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + idx * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (uint32_t)(z >> 32);
}
__host__ __device__ __forceinline__ uint32_t dropout_threshold(float p) {
  const double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
}
constexpr uint64_t DROPOUT_GOLDEN = 0x9E3779B97F4A7C15ull;
// dropout_bits(seed, idx) given z = seed + idx * DROPOUT_GOLDEN, so that a caller can hoist the per-cell part of z.  Bit-exact:
// only the high half of the last product is formed (hi32(z * C) = umulhi(lo, C_lo) + lo * C_hi + hi * C_lo, mod 2^32), and the
// final z ^= z >> 31 reaches the high half as h ^ (h >> 31).
__host__ __device__ __forceinline__ uint32_t dropout_bits_z(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27;
  const uint32_t lo = (uint32_t)z, hi = (uint32_t)(z >> 32);
  const uint32_t h = (uint32_t)(((uint64_t)lo * 0x133111EBu) >> 32) + lo * 0x94D049BBu + hi * 0x133111EBu;
  return h ^ (h >> 31);
}
// Keep bits of N consecutive mask elements idx0 .. idx0 + N - 1 (bit i = element idx0 + i kept), z0 = seed + idx0 * DROPOUT_GOLDEN.
template <int N>
__host__ __device__ __forceinline__ uint32_t dropout_keep_bits(uint64_t z0, uint32_t thresh) {
  uint32_t w = 0u;
#pragma unroll
  for (int i = 0; i < N; ++i) w |= (dropout_bits_z(z0 + (uint64_t)i * DROPOUT_GOLDEN) >= thresh ? 1u : 0u) << i;
  return w;
}

__device__ __forceinline__ float sigmoidf_exact(float z) { return 1.0f / (1.0f + expf(-z)); }

// Embedding-row gathers of the pair kernels use 128-bit loads when every row is 16-byte aligned: both widths a multiple
// of 4 floats (so a group of 4 never straddles the POI | region boundary at w_poi) and 16-byte aligned table bases.
__host__ __device__ inline bool rows_vec4(const NaisBranch& br, int half_split) {
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  return (br.w_poi & 3) == 0 && (br.w_reg & 3) == 0 && (half_split & 3) == 0 && al(br.hist_poi) && al(br.hist_reg);
}
// 4 consecutive elements d..d+3 (d % 4 == 0) of the concatenated history row [hist_poi[item] ; hist_reg[region]]
__device__ __forceinline__ float4 ldg_row4(const float* qp, const float* qr, int w_poi, int d) {
  return __ldg(reinterpret_cast<const float4*>(d < w_poi ? qp + d : qr + (d - w_poi)));
}

// Great-circle km from centred coordinates, haversine form (well conditioned in fp32 for short distances; equals the
// reference's law-of-cosines value powerLaw.py:7-21 mathematically, incl. its 1e-6 short-circuit).
__device__ __forceinline__ float dist_km_f(float lat1, float lon1, float lat2, float lon2, float coslat1, float coslat2) {
  float dlat = lat1 - lat2, dlon = lon1 - lon2;
  if (fabsf(dlat) < 1e-6f && fabsf(dlon) < 1e-6f) return 0.f;
  const float d2r = 0.017453292519943295f;
  float sa = sinf(0.5f * dlat * d2r), sb = sinf(0.5f * dlon * d2r);
  float h = sa * sa + coslat1 * coslat2 * sb * sb;
  return 2.f * 6371.f * asinf(fminf(1.f, sqrtf(h)));
}

// One history item's term of the power-law log score log G(u, j) = sum_h (ln a + b * ln max(0.01, d_km(h, j)))
// (powerLaw.py:85-92 in log space: a product of ~100 factors leaves the fp32 range, its log does not).  Every kernel that
// forms log G adds these terms in history order, so their sums agree bit for bit.
__device__ __forceinline__ float powerlaw_log_term(float km, float ln_a, float b) { return fmaf(b, logf(fmaxf(0.01f, km)), ln_a); }

// Geo re-ranking (NaisGeoMix): mixed = (1 - alpha) * sigmoid(score) + alpha * exp(log G - M_u)
struct GeoMixArgs {
  float ln_a, b, alpha;
  const float* user_logmax;  // [n_users] M_u
};
__device__ __forceinline__ float geo_mixed(float score, float logg, float logmax, float alpha) {
  return (1.f - alpha) * sigmoidf_exact(score) + alpha * expf(logg - logmax);
}

}  // namespace nais
