/*
 * nais_b200.h — C ABI of the B200-native NAIS scorer (libnais_b200.so).
 *
 * The reference (muyeon-jo/POI_recommendation_models) has NO plugin / FFI / operator registry: the boundary of its
 * hot path is the Python class API of model.py (SURVEY.md §8b).  This header is the C-level boundary a maintainer
 * binds (ctypes stub in INTEGRATION.md) to replace the bodies of
 *
 *   model.py:246-297   NAIS_region_distance_Embedding.attention_network   -> nais_pairs_forward / nais_pairs_backward
 *   model.py:57-89, 144-180, 355-401, 467-534   the sibling scorers        -> same entry points, other NaisParams
 *   validation.py:84-127   per-user candidate loop + torch.topk            -> nais_fullrank_topk
 *   torch.cat/topk merge across catalogue shards (new, multi-GPU)          -> nais_topk_merge
 *   eval_metrics.py:36-69  set-overlap counts behind precision/recall/hit@k  -> nais_hits_at_k
 *   run.py:252-254         embedding_dense_backward + dense Adagrad.step      -> nais_pairs_backward_adagrad
 *   powerLaw.py:85-92      PowerLaw.predict over a candidate list             -> nais_powerlaw_logscore
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into memory owned by the caller (PyTorch tensors); the library never
 *     allocates, frees or synchronises, and enqueues only on the given stream (documented exceptions: the pair backward /
 *     training entry points fork library-owned side streams from it and join them back before they return);
 *   - return 0 = OK; negative = argument error found before any launch (see NAIS_ERR_*); positive = cudaError_t;
 *   - all entry points are stateless and re-entrant (no environment variables, no hidden switches: every option is an
 *     argument or a struct field declared here); one host thread per GPU is the intended use.  Library-owned state per device:
 *     a 4-byte "bad index" word (nais_poll_bad_index), the side streams + events of nais_pairs_backward and the preparation
 *     stream of nais_train_users;
 *   - no C++ types, no torch types: plain pointers and sizes.
 */
#ifndef NAIS_B200_H_
#define NAIS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NAIS_ABI_VERSION 2

#if defined(__GNUC__)
#define NAIS_API __attribute__((visibility("default")))
#else
#define NAIS_API
#endif

/* distance modes (SURVEY.md §0.1 row 1) */
#define NAIS_DIST_NONE 0   /* NAIS_basic, NAIS_regionEmbedding */
#define NAIS_DIST_LATLON 1 /* sigmoid(Linear(2,2)(scale*|dlat,dlon|)) -> 2 extra input lanes of attn_layer1 (model.py:265, :366) */
#define NAIS_DIST_KM 2     /* logit += dist_km * sum_d embed_distance[0,d]  (model.py:497-504) */

/* precision of the attention-MLP contraction in nais_fullrank_topk */
#define NAIS_PREC_FP32 0     /* FP32 FFMA on CUDA cores (exact path) */
#define NAIS_PREC_TC_SPLIT 1 /* tcgen05 fp16 MMA, operands split hi+lo (3 MMAs, ~fp32 products), fp32 accumulate in TMEM */
#define NAIS_PREC_TC_FAST 2  /* tcgen05 fp16 MMA, single pass (11-bit operands), fp32 accumulate in TMEM */
#define NAIS_PREC_TC_MIX 3   /* tcgen05 fp16 MMA for hi*hi + two e5m2 (kind::f8f6f4) MMAs for the hi*lo, lo*hi corrections */
#define NAIS_PREC_TC_AUTO 4  /* MIX when a device-side bound on the logit scale keeps its error 4x under 1e-4, else SPLIT */
#define NAIS_PREC_MASK 0xff
/* OR-ed into `precision`: run the tensor path's run-time-shape kernel even where a compile-time-shape instantiation exists
 * (D = hid = 32 / 64 / 128).  Same math, another epilogue instruction order (results agree to fp32 rounding); the parity
 * suite uses it to cover both code paths. */
#define NAIS_PREC_FLAG_GENERIC 0x100
/* The D = hid = 64 compile-time-shape kernels (one branch, no NAIS_DIST_KM, at least two groups of candidate tiles in the range)
 * run on CTA PAIRS by default (tcgen05 cta_group::2: the two SMs of a TPC execute one M = 256 MMA per step and each stages half of
 * every user-operand chunk; +3.5 % users/s at the 1 kW power cap, DESIGN.md §4.1).  OR this flag into `precision` to keep one CTA
 * per SM: bit-identical results (same products, same summation order per accumulator element); the parity suite compares the two.
 * A plan prepared with the flag may only be used with the flag (the pair kernels pad the candidate image to an even number of
 * tile groups); a plan prepared without it serves both. */
#define NAIS_PREC_FLAG_ONE_CTA 0x200

/* NaisParams::pairs_precision — which kernels nais_pairs_forward / nais_pairs_backward[_adagrad] run */
#define NAIS_PAIRS_AUTO 0 /* tcgen05 kernels wherever the shape has them (see the entry points), FP32 CUDA-core kernels elsewhere */
#define NAIS_PAIRS_FP32 1 /* always the FP32 CUDA-core kernels */
#define NAIS_PAIRS_TC 2   /* tcgen05 kernels; NAIS_ERR_SHAPE if the shape has none */

#define NAIS_ERR_NULL -1      /* required pointer is NULL */
#define NAIS_ERR_SHAPE -2     /* unsupported / inconsistent dimension */
#define NAIS_ERR_ALIGN -3     /* pointer or row width not 16-byte aligned */
#define NAIS_ERR_WORKSPACE -4 /* workspace too small (ask nais_*_workspace_bytes) */
#define NAIS_ERR_MODE -5      /* unknown mode / flag combination */
#define NAIS_ERR_ARCH -6      /* device is not sm_100 (tensor path) */
#define NAIS_ERR_INDEX -7     /* a POI / region id was outside its table (reported by nais_poll_bad_index) */

typedef void* nais_stream_t; /* cudaStream_t */

/* One attention branch: q = [hist_poi[item] ; hist_reg[region]], p = [tgt_poi[item] ; tgt_reg[region]].
 * NAIS_region_distance_Embedding: w_poi = w_reg = embed_size/2, hist_reg == tgt_reg == embed_region (model.py:253-259).
 * NAIS_basic / NAIS_distance_Embedding: w_reg = 0.  Disentangled: branch 0 = (w_poi=D, w_reg=0, attn_layer*),
 * branch 1 = (w_poi=0, w_reg=D, region_attn_layer*), scores added (model.py:467-534). */
typedef struct NaisBranch {
  const float* hist_poi; /* [item_num, w_poi]   embed_history.weight */
  const float* tgt_poi;  /* [item_num, w_poi]   embed_target.weight  */
  const float* hist_reg; /* [region_num, w_reg] embed_region.weight  */
  const float* tgt_reg;  /* [region_num, w_reg] embed_region.weight  */
  const float* w1;       /* [hid, w_poi+w_reg+lanes] attn_layer1.weight, row-major; lanes = 2 iff NAIS_DIST_LATLON */
  const float* b1;       /* [hid] attn_layer1.bias */
  const float* w2;       /* [hid] attn_layer2.weight (no bias) */
  int32_t w_poi;
  int32_t w_reg;
} NaisBranch;

typedef struct NaisParams {
  NaisBranch branch[2];
  int32_t n_branch;   /* 1, or 2 for the disentangled model */
  int32_t hid;        /* hidden_size */
  int32_t item_num;   /* rows of the POI tables */
  int32_t region_num; /* rows of the region table (0 if unused) */
  int32_t dist_mode;  /* NAIS_DIST_* */
  float dist_scale;   /* 100 (model.py:265) or 1000 (model.py:366) */
  const float* dist_w; /* [2,2] dist_layer.weight (LATLON) */
  const float* dist_b; /* [2]   dist_layer.bias   (LATLON) */
  const float* dist_embed; /* [1, D] embed_distance.weight (KM): the reference allocates dist_embed_size rows and reads row 0 only (model.py:497-498) */
  int32_t dist_buckets;    /* must be 1 (row 0 of embed_distance); anything else is NAIS_ERR_MODE */
  float dist_bucket_km;    /* reserved (ignored) */
  float beta;              /* smoothing exponent of the softmax denominator (model.py:284-285) */
  /* Train-mode dropout on the attention hidden layer, relu(drop(W x + b)) (NAIS_basic / NAIS_regionEmbedding,
   * model.py:71,162).  0 disables.  Element (cell, hidden k) is kept iff
   * hi32(splitmix64(dropout_seed + (cell*hid + k))) >= dropout_p * 2^32, kept values are scaled by 1/(1-p), where cell is the
   * per-cell index of NaisPairs (act_mask's): b*H + h in the dense layout, seg_cell_offsets[s] + (r - row_offsets[s])*H_s + h in
   * the segmented one — so a one-segment batch draws the mask of the dense batch with the same rows.  Forward and backward of
   * one step must be given the same seed.  Pair API only; one branch. */
  float dropout_p;
  uint64_t dropout_seed;
  int32_t pairs_precision; /* NAIS_PAIRS_* (pair API only) */
  int32_t reserved0;
} NaisParams;

/* A batch of explicit (history row, target) pairs: the argument list of model.forward (model.py:231).
 *
 * Dense layout (seg_offsets == NULL) — what the reference builds: every row carries its own history, B rows x H items
 * (batches.py:97 literally repeats one user's history once per target).
 *
 * Segmented layout (seg_offsets != NULL) — many users in one step without the repeat and without a materialised [B,H,2]
 * distance tensor (SURVEY.md §8 f1): rows are grouped by segment (= a user); the rows [row_offsets[s], row_offsets[s+1]) of
 * segment s all share the history hist[seg_offsets[s] .. seg_offsets[s+1]) (hreg / hist_coords alike), H is ignored, aux must
 * be NULL and the LATLON lanes are formed in the kernel from centred coordinates (hist_coords per history item, tgt_coords per
 * row; NaisCatalog conventions).  Per-cell arrays (act_mask) are indexed cell(row r of segment s, item h) =
 * seg_cell_offsets[s] + (r - row_offsets[s]) * H_s + h.  The work decomposition is host-known: tile t covers rows
 * tile_row0[t] .. of segment tile_seg[t], at most min(16, 128 / H_s) rows (1 row when H_s > 128), never crossing a segment;
 * segments without history or without rows have no tile (a host loop over the segments builds these arrays: INTEGRATION.md).  NAIS_DIST_KM
 * forms dist_km per cell from the same centred coordinates (haversine, cos(latitude) = cos(center_lat + centred lat); NaisCatalog
 * conventions). */
typedef struct NaisPairs {
  const int64_t* hist; /* dense [B,H] / segmented [nnz]: history POI ids */
  const int64_t* tgt;  /* [B]   target POI ids */
  const int64_t* hreg; /* like hist: region id of each history POI (NULL when no branch has w_reg) */
  const int64_t* treg; /* [B]   region id of each target */
  const float* aux;    /* dense — LATLON: ll[B,H,2] = |dlat|,|dlon| degrees; KM: dist_km[B,H]; NONE: NULL.  Segmented: NULL */
  int64_t B;
  int32_t H;
  int32_t n_seg;                   /* segmented: number of segments */
  const int64_t* seg_offsets;      /* [n_seg+1] history CSR; NULL = dense layout */
  const int64_t* row_offsets;      /* [n_seg+1] */
  const int64_t* seg_cell_offsets; /* [n_seg+1] exclusive sum of (rows of s) * H_s */
  const int32_t* tile_seg;         /* [n_tiles] */
  const int64_t* tile_row0;        /* [n_tiles] */
  int64_t n_tiles;
  int64_t n_cells;                 /* seg_cell_offsets[n_seg] (host copy: sizes the backward workspace and act_mask) */
  const float* hist_coords;        /* [nnz,2] centred (lat, lon) of every history item (LATLON, KM) */
  const float* tgt_coords;         /* [B,2]   centred (lat, lon) of every target (LATLON, KM) */
  float center_lat;                /* segmented KM: the (lat, lon) that was subtracted from the coordinates */
  float center_lon;
} NaisPairs;

/* Gradients of nais_pairs_backward.  Dense tables must be zero-filled by the caller; the library writes each touched
 * row exactly once (sorted-segment accumulation, no atomics), and writes w1/b1/w2/dist_w/dist_b in full. */
typedef struct NaisGrads {
  float* hist_poi[2]; /* [item_num, w_poi]  per branch (NULL to skip) */
  float* tgt_poi[2];
  float* reg[2];      /* [region_num, w_reg] history-side + target-side contributions summed (shared table) */
  float* w1[2];
  float* b1[2];
  float* w2[2];
  float* dist_w; /* [2,2] */
  float* dist_b; /* [2]   */
  float* dist_embed; /* [dist_buckets, D] */
  /* Row-compacted table gradients (data-parallel training on catalogues where a dense [item_num, w] gradient is hundreds of
   * MB): when remap_X[b] != NULL, the gradient of table row r is written to row remap_X[b][r] of X[b] — a caller-sized
   * [n_touched, w] buffer — instead of row r; the caller fills remap (int32 [table rows]) for the rows its batch touches
   * (e.g. remap[unique(ids)] = 0..n_touched-1).  Untouched rows are never written in either form.  Ignored by the fused
   * Adagrad path. */
  const int32_t* remap_hist_poi[2];
  const int32_t* remap_tgt_poi[2];
  const int32_t* remap_reg[2];
} NaisGrads;

/* Candidate side of full-rank scoring: rows [row_base, row_base+n_rows) of the POI catalogue.  tgt_poi in NaisParams
 * is indexed by GLOBAL id (replicated table); region/coords here are indexed by (id - row_base) so a shard can pass
 * its slice only. */
typedef struct NaisCatalog {
  const int32_t* region; /* [n_rows] dense region id (businessRegionEmbedList, run.py:218-223) */
  const float* coords;   /* [n_rows,2] (lat,lon) degrees, centred on the host in float64 before the cast (DESIGN.md) */
  int64_t row_base;
  int64_t n_rows;
  float center_lat; /* the (lat, lon) that was subtracted from every coordinate (catalogue AND user items);      */
  float center_lon; /* NAIS_DIST_KM needs cos(latitude) = cos(center_lat + centred lat) for the haversine distance */
} NaisCatalog;

/* User histories as CSR (train_matrix.getrow(u).indices, validation.py:86), with the per-item side data gathered. */
typedef struct NaisUsers {
  const int64_t* offsets; /* [n_users+1] */
  const int32_t* items;   /* [nnz] POI ids */
  const int32_t* region;  /* [nnz] region id of each item */
  const float* coords;    /* [nnz,2] centred coords of each item */
  int32_t n_users;
} NaisUsers;

NAIS_API int nais_abi_version(void);
NAIS_API const char* nais_strerror(int code);
/* Number of kernels this library has launched in this process (diagnostic; bench.py reports it as gpu_launches). */
NAIS_API uint64_t nais_launch_count(void);

/* Which kernels the pair entry points run for (p, batch): *fwd_tc / *bwd_tc = 1 for the tcgen05 kernels, 0 for the FP32 CUDA-core
 * kernels (NaisParams::pairs_precision, the shape and the device decide; nothing is launched).  With dropout_p > 0, *bwd_tc = 1
 * holds for a backward given the forward's act_mask: without one, NAIS_PAIRS_AUTO runs the FP32 backward (which regenerates the
 * mask) and NAIS_PAIRS_TC returns NAIS_ERR_NULL.  Returns 0 or NAIS_ERR_*. */
NAIS_API int nais_pairs_dispatch(const NaisParams* p, const NaisPairs* batch, int32_t* fwd_tc, int32_t* bwd_tc);

/* score[b] = attention_network(pairs)  (pre-sigmoid, model.py:246-297).  Saved for backward (each may be NULL):
 * row_sum[n_branch,B] = sum_h E_bh, score_parts[n_branch,B] = per-branch score (their sum over branches is score),
 * act_mask[n_branch, cells] = the ReLU pattern of attn_layer1 (of branch bi's first layer from word bi*cells on): bit k of word
 * `cell` (b*H + h dense; NaisPairs) is set iff hidden unit k of that cell was active (t_k > 0) — with dropout, active AND kept.
 * act_mask is written only by the tcgen05 forward with hid <= 64 (nais_pairs_dispatch: fwd_tc).  One branch: [cells], as
 * before; the disentangled two branches run the tcgen05 kernels too and write both patterns.  The tcgen05 backward then takes the
 * unit-step of ReLU from it instead of thresholding its own recomputed t (bf16 two-term splits: ~1e-5 relative, enough to flip a
 * unit that sits on the kink and move a gradient by one cell's whole contribution).  With dropout the tcgen05 backward NEEDS it:
 * it draws no mask of its own. */
NAIS_API int nais_pairs_forward(const NaisParams* p, const NaisPairs* batch, float* score, float* row_sum, float* score_parts,
                       uint64_t* act_mask, nais_stream_t stream);

/* Explanations: which history items a pair score is made of (NAIS's attention, per cell).  For row r (a history and target j),
 * branch b (0, or 0 and 1 for the disentangled model) and history position h:
 *   E_bh = exp(a_bh) * [hist_h != j]     exactly the forward's, no max-shift
 *   S_b  = sum_h E_bh                    the forward's row_sum
 *   s_bh                                 the forward's similarity
 *   pi_bh = E_bh / S_b                   attention share: sums to 1 over h
 *   c_h  = sum_b E_bh * s_bh / S_b^beta  contribution: sums over h to the row's pre-sigmoid score
 * (position h is the same history item in both branches of the disentangled model: its POI in branch 0, its region in branch 1).
 * Per row, the m positions with the largest c_h are written in descending order, ties by ascending position (the ranking key of
 * nais_fullrank_topk): out_pos [B,m] indexes the row's own history — hist[b, pos] dense, hist[seg_offsets[s] + pos] segmented —
 * out_contrib [B,m] holds c_h and out_attn [n_branch,B,m] (optional) pi_bh.  A masked cell (history id == target id, read from
 * the ids) is never selected; a row with fewer than m selectable cells is padded with pos -1, contrib -inf, attn 0.  score [B]
 * (optional) is the pre-sigmoid score, bit-identical to nais_pairs_forward's for the same inputs.
 * Both layouts; the kernels of nais_pairs_forward (NaisParams::pairs_precision, nais_pairs_dispatch: fwd_tc), each storing every
 * cell's E and E*s in the workspace, then one warp per row selects.  Deterministic.  Argument errors before any CUDA call: m
 * outside [1, 32] -> NAIS_ERR_SHAPE, dropout_p > 0 -> NAIS_ERR_MODE (inference only), out_pos / out_contrib NULL -> NAIS_ERR_NULL,
 * workspace_bytes < nais_pairs_explain_workspace_bytes -> NAIS_ERR_WORKSPACE. */
NAIS_API size_t nais_pairs_explain_workspace_bytes(const NaisParams* p, const NaisPairs* batch);
NAIS_API int nais_pairs_explain(const NaisParams* p, const NaisPairs* batch, int32_t m, float* score, int32_t* out_pos,
                                float* out_contrib, float* out_attn, void* workspace, size_t workspace_bytes, nais_stream_t stream);

NAIS_API size_t nais_pairs_backward_workspace_bytes(const NaisParams* p, const NaisPairs* batch);
/* Given dscore[B] = dL/dscore, write every parameter gradient.  score_parts / row_sum / act_mask are the forward's outputs
 * (act_mask: [n_branch, cells] as nais_pairs_forward writes it, branch bi's backward reads words bi*cells ..; NULL unless the
 * tcgen05 forward wrote it; required by the tcgen05 backward with dropout, see nais_pairs_dispatch).
 * Streams: everything is ordered after the work already in `stream`, and `stream` is ordered after everything this call
 * enqueues, as for any other entry point — but the sort + reduce of the target-id and region-id lists and the reduce of the
 * per-CTA MLP-gradient partials run on three streams the library creates once per device (forked from / joined to `stream`
 * with events inside the call; legal under stream capture).
 * The call holds a process-wide mutex while it enqueues, so concurrent callers on one device share those streams safely. */
NAIS_API int nais_pairs_backward(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                        const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, void* workspace,
                        size_t workspace_bytes, nais_stream_t stream);

/* The pair above for a training step whose backward is known to follow (the torch.autograd.Function of the Python host layer):
 * the backward's three id sorts depend on the batch only, so nais_pairs_forward_presort forks them onto the library's side streams
 * BEFORE it enqueues the forward kernel (they run next to it: -50 us of a C3-sized step) and joins them to `stream` before it
 * returns — everything enqueued on `stream` afterwards is ordered after the sorts, and `bwd_workspace` may be released like any
 * other buffer of the call.  `grads`: only the NULL-ness of the table pointers (hist_poi / tgt_poi / reg, [0]) is read — it must
 * match the NaisGrads of the backward.  nais_pairs_backward_presorted is nais_pairs_backward on the lists that call left in the
 * workspace: same p, batch and workspace (nais_pairs_backward_workspace_bytes; contents untouched in between); one use per
 * presort.  One branch only (NAIS_ERR_MODE otherwise: use the plain pair). */
NAIS_API int nais_pairs_forward_presort(const NaisParams* p, const NaisPairs* batch, const NaisGrads* grads, float* score,
                               float* row_sum, float* score_parts, uint64_t* act_mask, void* bwd_workspace,
                               size_t bwd_workspace_bytes, nais_stream_t stream);
NAIS_API int nais_pairs_backward_presorted(const NaisParams* p, const NaisPairs* batch, const float* score_parts, const float* row_sum,
                                  const uint64_t* act_mask, const float* dscore, const NaisGrads* grads, void* workspace,
                                  size_t workspace_bytes, nais_stream_t stream);

/* One row-sparse Adagrad step from a key-ordered list of (table row id, gradient row) pairs — the union of the touched-row lists
 * the ranks of a data-parallel step exchange (SURVEY.md §8e 'Train partitioning').  keys [n] int32 ascending (equal ids
 * adjacent: their rows are summed first, in list order — deterministic, identical on every rank that holds the same list),
 * rows [n, w].  For every distinct id r with summed gradient g:  sum[r] += g*g ; param[r] -= lr * g / (sqrt(sum[r]) + eps)
 * (torch.optim.Adagrad, weight_decay = lr_decay = 0).  With sum == NULL the summed rows are written to grad_out[r] instead
 * (a dense [n_rows, w] table; rows not listed are not touched).  ids outside [0, n_rows) are skipped. */
NAIS_API size_t nais_rows_adagrad_workspace_bytes(int64_t n, int32_t w);
NAIS_API int nais_rows_adagrad(const int32_t* keys, const float* rows, int64_t n, int32_t w, int32_t n_rows, float* grad_out,
                               float* param, float* sum, float lr, float eps, void* workspace, size_t workspace_bytes,
                               nais_stream_t stream);

/* Device-side training-batch construction for the segmented layout (batches.py:67-108 `get_NAIS_batch_region`, many users per
 * call).  For every segment s (history hist[seg_offsets[s] .. seg_offsets[s+1]), H_s items) the rows
 * [row_offsets[s], row_offsets[s] + (num_ng + 1) * H_s) are written interleaved like the reference: positive i at
 * + i * (num_ng + 1) (label 1), its num_ng negatives behind it (label 0).  Negatives are H_s * num_ng POIs drawn uniformly
 * WITHOUT replacement from the POIs outside the history (the distribution of the reference's shuffle-and-take-a-prefix), by a
 * counter-based generator keyed on (seed, segment, slot, attempt): the same seed gives the same batch; it is NOT Python's
 * `random` stream.  Positives keep their stored order.  poi_region [item_num] / poi_coords [item_num,2] (centred) fill treg /
 * tgt_coords (each may be NULL together with its output).  max_hist >= every H_s (host-known, sizes the per-segment hash set);
 * item_num must exceed (num_ng + 1) * H_s for every segment.  Outputs: tgt [B] int64, label [B] float, treg [B] int64,
 * tgt_coords [B,2] with B = row_offsets[n_seg]. */
NAIS_API int nais_sample_batch(const int64_t* seg_offsets, const int64_t* hist, int32_t n_seg, const int64_t* row_offsets,
                               int32_t num_ng, int32_t item_num, const int32_t* poi_region, const float* poi_coords, uint64_t seed,
                               int32_t max_hist, int64_t* tgt, float* label, int64_t* treg, float* tgt_coords, nais_stream_t stream);

/* Row-sparse Adagrad fused into the embedding-gradient segment reduce.  Replaces, for the embedding tables, the dense
 * `embedding_dense_backward` + `torch.optim.Adagrad.step()` of run.py:225,252-254 (weight_decay = 0, lr_decay = 0: a row
 * whose gradient is zero does not move, so stepping only the touched rows IS the dense step).  For every table with a
 * non-NULL `sum_*` pointer (the optimizer's `state['sum']`, same shape as the table) the summed row gradient g is applied
 * in place instead of being written to NaisGrads:  sum += g*g ;  param -= lr * g / (sqrt(sum) + eps).  The parameter
 * tables are the ones NaisParams points to (they ARE written).  Two branches only in the disentangled layout (see below). */
typedef struct NaisAdagrad {
  float lr, eps;
  float* sum_hist_poi[2];
  float* sum_tgt_poi[2];
  float* sum_reg[2];
} NaisAdagrad;
/* Same as nais_pairs_backward (MLP / dist-layer gradients go to `grads`; table pointers in `grads` may be NULL). */
NAIS_API int nais_pairs_backward_adagrad(const NaisParams* p, const NaisPairs* batch, const float* score_parts,
                                const float* row_sum, const uint64_t* act_mask, const float* dscore, const NaisGrads* grads,
                                const NaisAdagrad* opt, void* workspace, size_t workspace_bytes, nais_stream_t stream);

/* One whole optimizer step of run.py:248-254 — zero_grad, forward, sigmoid + BCELoss, backward, Adagrad.step — in ONE call (the
 * reference's schedule is one user per step: 17 Python-level ops and ~25 launches per step make it host-bound; this is 8-12
 * launches and one call).  loss = sum_b w_b * BCE(sigmoid(score_b), label_b) with w_b = row_weight[b], or 1/B when row_weight is
 * NULL (the batch mean of nn.BCELoss); log terms clamped at -100 and the gradient's denominator at 1e-12 like torch.
 * Embedding tables: row-sparse Adagrad as in nais_pairs_backward_adagrad (`tables`).  MLP / distance-layer parameters: dense
 * Adagrad on the optimizer's state['sum'] tensors in `dense`:  sum += g*g ;  param += -lr * (g / (sqrt(sum) + eps))  (torch's
 * update with weight_decay = lr_decay = 0).  Every parameter NaisParams points to IS written.
 * loss: device float[1]; score (optional): device float[B], the pre-sigmoid scores of the forward.
 *
 * Two branches (nais_pairs_backward_adagrad, nais_pairs_train_step, nais_train_users): accepted for the disentangled layout only —
 * branch[0].w_reg == 0 and branch[1].w_poi == 0, so every table belongs to exactly one branch and one row-sparse step per id list IS
 * the dense step — with NAIS_DIST_NONE or NAIS_DIST_KM; any other two-branch input is NAIS_ERR_MODE.  Branch 0's tables go in
 * NaisAdagrad slot [0], branch 1's region table in sum_reg[1]; the sum_region_* / sum_dist_embed fields below are required
 * (NAIS_ERR_NULL) exactly then.  embed_distance: only row 0 is read (dist_buckets == 1), so only row 0 moves. */
typedef struct NaisDenseAdagrad {
  float lr, eps;
  float* sum_w1;
  float* sum_b1;
  float* sum_w2;
  float* sum_dist_w; /* NULL unless NAIS_DIST_LATLON */
  float* sum_dist_b;
  float* sum_region_w1;  /* disentangled layout: region_attn_layer1.weight / .bias, region_attn_layer2.weight */
  float* sum_region_b1;
  float* sum_region_w2;
  float* sum_dist_embed; /* disentangled layout: [D], row 0 of embed_distance's state */
} NaisDenseAdagrad;
NAIS_API size_t nais_pairs_train_step_workspace_bytes(const NaisParams* p, const NaisPairs* batch);
NAIS_API int nais_pairs_train_step(const NaisParams* p, const NaisPairs* batch, const float* label, const float* row_weight,
                                   const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* loss, float* score,
                                   void* workspace, size_t workspace_bytes, nais_stream_t stream);

/* nais_pairs_train_step with the pairwise BPR loss -log sigmoid(s+ - s-) instead of BCE (the batch's `label` is not read).  The B
 * rows come in groups of G = 1 + num_neg consecutive rows: row g*G is the positive, rows g*G + 1 .. g*G + num_neg its negatives —
 * the order nais_sample_batch writes.  With d_gj = score[g*G] - score[g*G + j]:
 *   loss = sum_g w_g sum_{j=1..num_neg} softplus(-d_gj),  w_g = group_weight[g], or 1 / (n_groups * num_neg) when group_weight is
 *   NULL (the mean over pairs: -logsigmoid(d).mean());  softplus(-d) = max(-d, 0) + log1p(exp(-|d|)), finite for any score.
 *   dL/dscore[g*G + j] = w_g sigma(-d_gj) (torch's log_sigmoid backward form), dL/dscore[g*G] = -sum_j w_g sigma(-d_gj), j ascending.
 * The loss is summed by one CTA in a fixed order (deterministic, no atomics).  group_weight = 1 / (pairs of the user of g) makes a
 * segmented multi-user step the sum of the per-user mean BPR losses.  Optimizer, workspace (nais_pairs_train_step_workspace_bytes)
 * and outputs as nais_pairs_train_step.  bpr NULL is NAIS_ERR_NULL; num_neg < 1 or B % (1 + num_neg) != 0 is NAIS_ERR_SHAPE. */
typedef struct NaisBprLoss {
  int32_t num_neg;           /* >= 1: rows in groups of 1 + num_neg, positive first */
  int32_t reserved0;
  const float* group_weight; /* [B / (1 + num_neg)] device, or NULL = mean over pairs */
} NaisBprLoss;
NAIS_API int nais_pairs_train_step_bpr(const NaisParams* p, const NaisPairs* batch, const NaisBprLoss* bpr, const NaisAdagrad* tables,
                                       const NaisDenseAdagrad* dense, float* loss, float* score, void* workspace, size_t workspace_bytes,
                                       nais_stream_t stream);

/* The reference's training schedule — ONE optimizer step per user (run.py:227-255) — for a list of users in one call: per user,
 * nais_sample_batch over his history (every positive + num_ng negatives each, labels [1, 0..0]: batches.py:67-108) and
 * nais_pairs_train_step with the batch-mean BCE, enqueued back to back with no host work in between but the launches (~15 per
 * user).  The user's history is the slice [host_indptr[u], host_indptr[u + 1]) of `indices` (the train matrix' CSR; no copy);
 * entry_region / entry_coords are the region id / centred (lat, lon) of every CSR entry (region[indices], coords[indices]; NULL
 * when the variant has no region table / distance lanes).  host_indptr [n_rows + 1] and host_users are HOST arrays (read during
 * the call; a user id outside [0, n_rows) is an argument error).
 * User i samples with seed + host_users[i].  losses: device float[n_users] (0 for a user without history).  Two branches: as
 * nais_pairs_train_step.  entry_coords / poi_coords are needed for NAIS_DIST_KM as for NAIS_DIST_LATLON.
 * Streams: what depends on the batch only (segment structure, sampler, the id sorts of the backward) is enqueued ONE USER AHEAD on
 * a library-owned preparation stream (one per device, created on first use) into the other half of the workspace, so the chain
 * of dependent launches per optimizer step is forward -> BCE -> backward -> Adagrad; the preparation stream starts after the work
 * already in `stream` and everything it does is consumed by work in `stream` before the call's last launch (events created and
 * destroyed inside the call).  Same kernels on the same inputs per user: results are those of the sequential loop, bit for bit. */
NAIS_API size_t nais_train_users_workspace_bytes(const NaisParams* p, int32_t max_hist, int32_t num_ng);
NAIS_API int nais_train_users(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices, const int64_t* entry_region,
                              const float* entry_coords, const int32_t* poi_region, const float* poi_coords, const int64_t* host_users,
                              int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables, const NaisDenseAdagrad* dense,
                              float* losses, void* workspace, size_t workspace_bytes, nais_stream_t stream);
/* nais_train_users for coordinates centred on (center_lat, center_lon): the (lat, lon) that was subtracted from entry_coords /
 * poi_coords (NaisCatalog conventions).  NAIS_DIST_KM needs it for cos(latitude); nais_train_users is this call with (0, 0).
 * Both return NAIS_ERR_MODE for dropout_p > 0 (one seed for every step would repeat the mask): use nais_train_users_dropout. */
NAIS_API int nais_train_users_centred(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                                      const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region,
                                      const float* poi_coords, const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed,
                                      const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* losses, void* workspace,
                                      size_t workspace_bytes, float center_lat, float center_lon, nais_stream_t stream);
/* nais_train_users_centred with train-mode dropout (NaisParams::dropout_p > 0): host_dropout_seeds is a HOST array of n_users
 * seeds, the step of host_users[i] runs with dropout_seed = host_dropout_seeds[i] (entries of users without a history are
 * ignored).  NULL with dropout_p > 0 is NAIS_ERR_NULL; with dropout_p == 0 the array is not read. */
NAIS_API int nais_train_users_dropout(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                                      const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region,
                                      const float* poi_coords, const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed,
                                      const NaisAdagrad* tables, const NaisDenseAdagrad* dense, float* losses, void* workspace,
                                      size_t workspace_bytes, float center_lat, float center_lon, const uint64_t* host_dropout_seeds,
                                      nais_stream_t stream);
/* nais_train_users_dropout with the BPR loss of nais_pairs_train_step_bpr: per user, the sampler (seed + user id) draws num_ng
 * negatives for each positive, and one optimizer step takes the mean BPR loss over the user's H * num_ng (positive, negative)
 * pairs.  losses[i] is that mean (0 for a user without history).  Workspace: nais_train_users_workspace_bytes; preparation one
 * user ahead, streams and dropout seeds as nais_train_users_dropout.  num_ng < 1 is NAIS_ERR_SHAPE. */
NAIS_API int nais_train_users_bpr(const NaisParams* p, const int64_t* host_indptr, int64_t n_rows, const int64_t* indices,
                                  const int64_t* entry_region, const float* entry_coords, const int32_t* poi_region, const float* poi_coords,
                                  const int64_t* host_users, int32_t n_users, int32_t num_ng, uint64_t seed, const NaisAdagrad* tables,
                                  const NaisDenseAdagrad* dense, float* losses, void* workspace, size_t workspace_bytes, float center_lat,
                                  float center_lon, const uint64_t* host_dropout_seeds, nais_stream_t stream);

/* Workspace for nais_fullrank_topk / nais_fullrank_scores: n_users and nnz = offsets[n_users] are host-known. */
NAIS_API size_t nais_fullrank_workspace_bytes(const NaisParams* p, int32_t n_users, int64_t nnz, int64_t poi_begin,
                                     int64_t poi_end, int32_t k, int32_t precision);
/* For every user: score all POIs in [poi_begin, poi_end) (history items excluded when exclude_history != 0),
 * keep the k best by (score desc, id asc).  out_score [n_users,k] (pre-sigmoid; -inf padding), out_id [n_users,k]
 * (global POI id; -1 padding).  Replaces validation.py:84-127. */
NAIS_API int nais_fullrank_topk(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                       int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, float* out_score, int32_t* out_id, void* workspace, size_t workspace_bytes,
                       nais_stream_t stream);

/* ---- planned full-rank scoring: the per-model / per-catalogue constants are computed ONCE --------------------------------------
 * nais_fullrank_topk recomputes, on every call, things that only depend on the weights and the catalogue range: the table maxima
 * and power-of-two scales, the hidden-unit permutation, and the packed candidate image (tensor path).  An evaluation scores many
 * user batches against the same weights (validation.py:69 loops over all users with a frozen model), so:
 *
 *   plan = caller-owned device buffer of nais_fullrank_plan_bytes(...) bytes
 *   nais_fullrank_prepare(...)        once per (weights, catalogue range, precision); enqueued on `stream`, never synchronises
 *   nais_fullrank_topk_planned(...)   per user batch: packs the users' operand, scores, block top-k, merge
 *
 * The plan is read-only at call time (several streams may score against one plan).  It is valid until a parameter tensor, the
 * catalogue arrays or the range change; the caller re-prepares after an optimizer step.  NAIS_PREC_FP32 needs no plan
 * (plan_bytes = 0, plan may be NULL).  Results are bit-identical to nais_fullrank_topk. */
NAIS_API size_t nais_fullrank_plan_bytes(const NaisParams* p, int64_t poi_begin, int64_t poi_end, int32_t precision);
NAIS_API int nais_fullrank_prepare(const NaisParams* p, const NaisCatalog* cat, int64_t poi_begin, int64_t poi_end,
                                   int32_t precision, void* plan, size_t plan_bytes, nais_stream_t stream);
/* Workspace of a planned call (no candidate image inside: smaller than nais_fullrank_workspace_bytes). */
NAIS_API size_t nais_fullrank_planned_workspace_bytes(const NaisParams* p, int32_t n_users, int64_t nnz, int64_t poi_begin,
                                                      int64_t poi_end, int32_t k, int32_t precision);
/* Outputs: out_score / out_id as nais_fullrank_topk (both or neither may be NULL) and / or out_keys [n_users, k]: the packed
 * ranking keys (ordered(score) << 32 | ~id; 0 = no entry) that nais_topk_merge_keys consumes — one 8-byte word per entry, so
 * the per-shard lists of a range-sharded catalogue travel in ONE all-gather. */
NAIS_API int nais_fullrank_topk_planned(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                                        int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, const void* plan,
                                        size_t plan_bytes, uint64_t* out_keys, float* out_score, int32_t* out_id, void* workspace,
                                        size_t workspace_bytes, nais_stream_t stream);

/* Merge n_lists key lists per user into one (score desc, id asc — the order of nais_fullrank_topk).  List l of user u starts at
 * in_keys + u * user_stride + l * list_stride (strides in 8-byte words), so the [world, n_users, k] buffer an all-gather
 * produces is merged in place: user_stride = k, list_stride = n_users * k.  out_keys / (out_score, out_id): either may be NULL. */
NAIS_API int nais_topk_merge_keys(const uint64_t* in_keys, int64_t user_stride, int64_t list_stride, int32_t n_users,
                                  int32_t n_lists, int32_t k, uint64_t* out_keys, float* out_score, int32_t* out_id,
                                  nais_stream_t stream);

/* Out-of-range ids.  nn.Embedding raises IndexError on an id outside its table (the reference's behaviour for a bad batch or
 * a region_num mismatch).  The kernels cannot raise and the library never synchronises, so: every id read by the pair kernels
 * (hist, tgt, hreg, treg) and by the user-operand pack of the full-rank path is range-checked on the device; an out-of-range
 * id is never used as an address (reads fall back to row 0, its gradient contribution is dropped, no table / optimizer row
 * is written for it) and sets the device's bad-index word.  nais_poll_bad_index enqueues, on `stream`, a copy of that word
 * into *host_flag (pinned host memory recommended: then the call is asynchronous) followed by its reset; once the stream has
 * reached that point, *host_flag != 0 means some kernel enqueued before the poll saw a bad id -> the caller raises
 * (NAIS_ERR_INDEX).  Returns 0 or a cudaError_t. */
NAIS_API int nais_poll_bad_index(int32_t* host_flag, nais_stream_t stream);

/* Merge n_lists sorted top-k lists per user (e.g. one per catalogue shard after an all-gather) into one.
 * in_score/in_id: [n_users, n_lists, k]; out: [n_users, k].  Same order rule as nais_fullrank_topk. */
NAIS_API int nais_topk_merge(const float* in_score, const int32_t* in_id, int32_t n_users, int32_t n_lists, int32_t k,
                    float* out_score, int32_t* out_id, nais_stream_t stream);

/* Per-user hit counts behind eval_metrics.precision_at_k / recall_at_k / hitrate_at_k (eval_metrics.py:36-69):
 * hits[u, i] = |positives(u) ∩ rec[u, :k_list[i]]| for the recommended lists rec [n_users, k_rec] (ids, -1 padding) and the
 * positives CSR (pos_offsets [n_users+1], pos_items).  Integer work only: the float means are formed by the caller in the
 * reference's order, so the metrics stay bit-identical.  k_list is a DEVICE array of n_k ints. */
NAIS_API int nais_hits_at_k(const int32_t* rec, int32_t n_users, int32_t k_rec, const int64_t* pos_offsets,
                            const int32_t* pos_items, const int32_t* k_list, int32_t n_k, int32_t* hits,
                            nais_stream_t stream);

/* Power-law geographical score of powerLaw.py:57-92 (PowerLaw.predict), in log space, for every user against the POIs
 * [poi_begin, poi_end):  out_logg[u, j - poi_begin] = sum_{h in history(u)} ln(a * max(0.01, d_km(h, j))^b),  a > 0.
 * d_km = powerLaw.dist (great circle, R = 6371 km, 0 below 1e-6 degrees) from the centred float32 coordinates of
 * NaisCatalog / NaisUsers.  The caller exponentiates relative to the per-user maximum (run.py:55-59 `normalize`). */
NAIS_API int nais_powerlaw_logscore(const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin, int64_t poi_end, float a,
                           float b, float* out_logg, nais_stream_t stream);

/* ---- geo re-ranking: the power-law mix of run.py:523-546 inside the full-rank top-k ----------------------------------------------
 *   logG(u, j)  = sum_{h in history(u)} (ln a + b * ln max(0.01, d_km(h, j)))        (as nais_powerlaw_logscore)
 *   M_u         = max_j logG(u, j) over the ranked candidates: the whole catalogue (every shard), minus the history when excluded
 *   mixed(u, j) = (1 - alpha) * sigmoid(score(u, j)) + alpha * exp(logG(u, j) - M_u)
 * The top-k is taken by `mixed` (desc, then id asc).  A history item that is not excluded includes its own h = j term (d = 0).
 *
 * nais_powerlaw_logmax writes out_logmax[n_users] = max over the candidates of [poi_begin, poi_end) (-inf for a user without
 * candidates); the per-shard maxima of a range-sharded catalogue combine with a max.  It sums log G in the order of
 * nais_powerlaw_logscore, so M_u equals the maximum of that output bit for bit.  Needs the coordinates of NaisCatalog and
 * NaisUsers.  a <= 0 or a non-finite a / b -> NAIS_ERR_MODE.
 *
 * nais_fullrank_topk_geo_planned = nais_fullrank_topk_planned ranked by `mixed`: out_score (and the keys) hold mixed, not a
 * pre-sigmoid score; the workspace is nais_fullrank_planned_workspace_bytes.  The tensor path runs the run-time-shape kernel
 * (never the compile-time-shape or CTA-pair kernels); NAIS_PREC_FP32 takes a NULL plan.  a <= 0 or a non-finite a / b / alpha ->
 * NAIS_ERR_MODE; geo, the coordinates or user_logmax missing -> NAIS_ERR_NULL (all checked before any CUDA call). */
typedef struct NaisGeoMix {
  float a, b, alpha;          /* power law a * d^b (a > 0) and the mixing weight (Args.powerlaw_weight) */
  const float* user_logmax;   /* [n_users] device: M_u from nais_powerlaw_logmax over the whole ranked catalogue */
} NaisGeoMix;
NAIS_API int nais_powerlaw_logmax(const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin, int64_t poi_end, float a,
                                  float b, int32_t exclude_history, float* out_logmax, nais_stream_t stream);
NAIS_API int nais_fullrank_topk_geo_planned(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                                            int64_t poi_end, int32_t k, int32_t exclude_history, int32_t precision, const void* plan,
                                            size_t plan_bytes, const NaisGeoMix* geo, uint64_t* out_keys, float* out_score,
                                            int32_t* out_id, void* workspace, size_t workspace_bytes, nais_stream_t stream);

/* Same scoring pass, but also writes every pre-sigmoid score: all_scores[n_users, poi_end-poi_begin] (history items are
 * scored with their own cell masked, like a training positive).  For parity checks of the fused path on small cases. */
NAIS_API int nais_fullrank_scores(const NaisParams* p, const NaisCatalog* cat, const NaisUsers* users, int64_t poi_begin,
                         int64_t poi_end, int32_t precision, float* all_scores, void* workspace,
                         size_t workspace_bytes, nais_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NAIS_B200_H_ */
