// Fused top-K retrieval (sm_100a): for a batch of users, score = u . v over the whole catalog, drop (or re-score) the
// items each user has already seen, and keep the K best by (score desc, item id asc). The B x nI score matrix never
// reaches global memory: scores live in registers, the running per-user top-K in shared memory.
//
// One block = TU users x one contiguous item range (a "split"). Items stream in tiles of 256, one item per thread;
// a thread scores its item against all TU users with one fp32 fma chain per score, k ascending from 0 — the canonical
// order of the evaluation kernels (eval.cu), so scores and therefore rankings are bit-identical to theirs. A candidate
// (score, item) is packed into one u64 key that orders exactly like (score desc, id asc); keys beating the user's
// current K-th best are appended to the user's candidate buffer, and a block-wide bitonic sort truncates a buffer to
// its K best whenever one could overflow on the next tile. With more than one split, recommend_merge_kernel merges the
// per-split lists.
//
// recommend_subset_kernel restricts each row to one subset of the catalog (an ascending item-id list): the same scores,
// masking and selection over the gathered ids of the row's subset, with rows grouped by subset on the device first.
//
// The _bias kernels add a per-item fp32 bias to each score after the fma chain (a CDAE output layer: z . W_o[i] + b_o[i]);
// they share their bodies with the unbiased kernels, whose code the bias does not touch.
#include <float.h>
#include <algorithm>
#include <cuda_bf16.h>
#include "common.cuh"

namespace yr {

constexpr int kRtThreads = 256;
constexpr int kRtTile = 256;         // items per tile, one per thread
constexpr int kRtEntries = 8192;     // candidate keys per block: TU users x (kRtEntries / TU)
constexpr int kRtMaxK = 1024;
constexpr int kRtMaxD = 1024;
constexpr int kRtMaxUD = 16 * 512;   // TU x d at most: wider tables take fewer users per block (see rt_users)
constexpr int kRtMinSplit = 4096;    // items per split at least: long enough for the thresholds to settle
constexpr int kRtMergeMax = 16384;   // keys one merge block sorts (128 KB of shared memory)

// (score desc, id asc) == u64 key desc. Scores map to an order-preserving u32; ids are stored complemented.
// Key 0 is never a candidate (it would be a negative NaN with id 2^32 - 1): it marks an empty slot.
__device__ __forceinline__ uint64_t rt_key(float s, uint32_t item) {
  uint32_t u = __float_as_uint(s);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((uint64_t)u << 32) | (uint64_t)(0xffffffffu - item);
}

__device__ __forceinline__ void rt_decode(uint64_t key, int64_t& id, float& s) {
  if (key == 0) { id = -1; s = -INFINITY; return; }
  uint32_t u = (uint32_t)(key >> 32);
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  s = __uint_as_float(u);
  id = (int64_t)(0xffffffffu - (uint32_t)key);
}

__device__ __forceinline__ float rt_to_float(float x) { return x; }
__device__ __forceinline__ float rt_to_float(__nv_bfloat16 x) { return __bfloat162float(x); }

// v[0..7] = p[0..7] as floats (p 16-byte aligned)
__device__ __forceinline__ void rt_load8(const float* p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void rt_load8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

// Sort each of the `segs` segments of `n` keys (n a power of two) descending; the whole block takes part.
__device__ void rt_bitonic_desc(uint64_t* keys, int segs, int n) {
  const int half = n >> 1;
  for (int size = 2; size <= n; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < segs * half; t += blockDim.x) {
        const int seg = t / half, r = t - seg * half;
        const int lo = 2 * stride * (r / stride) + (r % stride);
        uint64_t* base = keys + (size_t)seg * n;
        const uint64_t a = base[lo], b = base[lo + stride];
        const bool desc = (lo & size) == 0;
        if ((a < b) == desc) { base[lo] = b; base[lo + stride] = a; }
      }
      __syncthreads();
    }
}

// Truncate every candidate buffer to its K best; thr[u] becomes the K-th best key once a user has K candidates.
template <int TU>
__device__ void rt_compact(uint64_t* keys, int* cnt, uint64_t* thr, int K) {
  constexpr int CAP = kRtEntries / TU;
  for (int i = threadIdx.x; i < TU * CAP; i += blockDim.x)
    if ((i % CAP) >= cnt[i / CAP]) keys[i] = 0;
  __syncthreads();
  rt_bitonic_desc(keys, TU, CAP);
  if (threadIdx.x < TU) {
    const int u = threadIdx.x;
    const int c = min(cnt[u], K);
    cnt[u] = c;
    if (c == K && thr[u] != ~0ull) thr[u] = keys[(size_t)u * CAP + K - 1];
  }
  __syncthreads();
}

// acc[u] = Us[u] . vrow for the TU staged users, one fma chain each, k ascending (acc = 0 when vrow is null).
template <typename T, int TU>
__device__ __forceinline__ void rt_score(const T* __restrict__ vrow, const float* Us, int d, float (&acc)[TU]) {
#pragma unroll
  for (int u = 0; u < TU; ++u) acc[u] = 0.f;
  if (!vrow) return;
  for (int k = 0; k < d; k += 8) {
    float v[8];
    rt_load8(vrow + k, v);
#pragma unroll
    for (int u = 0; u < TU; ++u) {
      const float4 a0 = *reinterpret_cast<const float4*>(Us + u * d + k);
      const float4 a1 = *reinterpret_cast<const float4*>(Us + u * d + k + 4);
      float s = acc[u];
      s = fmaf(a0.x, v[0], s); s = fmaf(a0.y, v[1], s); s = fmaf(a0.z, v[2], s); s = fmaf(a0.w, v[3], s);
      s = fmaf(a1.x, v[4], s); s = fmaf(a1.y, v[5], s); s = fmaf(a1.z, v[6], s); s = fmaf(a1.w, v[7], s);
      acc[u] = s;
    }
  }
}

// Append (s, item) to user u's candidate buffer if it beats the user's current K-th best.
template <int TU>
__device__ __forceinline__ void rt_offer(uint64_t* keys, int* cnt, const uint64_t* thr, int u, float s, uint32_t item) {
  if (s == 0.f) s = 0.f;                       // -0 ranks like +0
  if (!(s > -INFINITY)) return;                // excluded (-inf) or NaN: never returned
  const uint64_t key = rt_key(s, item);
  if (key > thr[u]) {
    const int p = atomicAdd(cnt + u, 1);
    keys[(size_t)u * (kRtEntries / TU) + p] = key;
  }
}

// The body of recommend_topk_kernel (kBias = false) and recommend_topk_bias_kernel (kBias: score + item_bias[item]).
template <typename T, int TU, bool kBias>
__device__ __forceinline__ void
recommend_topk_body(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                    const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ seen_ptr,
                    const int32_t* __restrict__ seen_idx, int seen_by_row, float masked_score, int K, int64_t per_split,
                    uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids, float* __restrict__ out_scores,
                    int32_t* err, const float* __restrict__ item_bias) {
  constexpr int CAP = kRtEntries / TU;
  constexpr int kWords = kRtTile / 32;
  extern __shared__ __align__(16) uint64_t rt_smem[];
  uint64_t* keys = rt_smem;                                    // [TU][CAP]
  uint64_t* thr = keys + kRtEntries;                           // [TU]; ~0 = inactive row (no candidate beats it)
  float* Us = reinterpret_cast<float*>(thr + TU);              // [TU][d]
  uint32_t* bits = reinterpret_cast<uint32_t*>(Us + (size_t)TU * d);   // [TU][kWords]: seen items of the tile
  int* cnt = reinterpret_cast<int*>(bits + TU * kWords);       // [TU]
  int* mcur = cnt + TU;                                        // [TU]: next unconsumed entry of the seen list
  int* mend = mcur + TU;                                       // [TU]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t b0 = (int64_t)blockIdx.x * TU;
  const int split = blockIdx.y;
  const int64_t ib = (int64_t)split * per_split;
  const int64_t ie = min(nI, ib + per_split);

  for (int i = tid; i < TU * d; i += kRtThreads) {
    const int u = i / d, k = i - u * d;
    const int64_t b = b0 + u;
    float x = 0.f;
    if (b < B) {
      const int64_t uid = uids[b];
      if (uid >= 0 && uid < nU) x = rt_to_float(U[uid * d + k]);
    }
    Us[i] = x;
  }
  if (tid < TU) {
    const int64_t b = b0 + tid;
    bool active = false;
    int c = 0, en = 0;
    if (b < B) {
      const int64_t uid = uids[b];
      active = uid >= 0 && uid < nU;
      if (!active && err) atomicExch(err, 1);
      if (active && seen_ptr) {
        const int64_t row = seen_by_row ? b : uid;
        c = seen_ptr[row]; en = seen_ptr[row + 1];
        int lo = c, hi = en;                       // first seen entry >= ib (lists ascending)
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (seen_idx[mid] < ib) lo = mid + 1; else hi = mid;
        }
        c = lo;
      }
    }
    thr[tid] = active ? 0ull : ~0ull;
    cnt[tid] = 0;
    mcur[tid] = c; mend[tid] = en;
  }
  __syncthreads();

  for (int64_t i0 = ib; i0 < ie; i0 += kRtTile) {
    // ---- seen items of this tile -> bitmask (one warp per user, the sorted list is consumed in order) ----
    for (int i = tid; i < TU * kWords; i += kRtThreads) bits[i] = 0;
    __syncthreads();
    if (seen_ptr) {
      const int64_t tile_end = min(i0 + kRtTile, ie);
      for (int u = warp; u < TU; u += kRtThreads / 32) {
        int c = mcur[u];
        const int en = mend[u];
        while (c < en) {
          const int p = c + lane;
          const int64_t it = (p < en) ? (int64_t)seen_idx[p] : INT64_MAX;
          const bool in = it < tile_end;
          if (in && it >= i0) atomicOr(bits + u * kWords + (int)((it - i0) >> 5), 1u << ((it - i0) & 31));
          const int n = __popc(__ballot_sync(kFull, in));
          c += n;
          if (n < 32) break;
        }
        if (lane == 0) mcur[u] = c;
      }
    }
    // ---- scores of my item against every user of the tile: one fma chain each, k ascending ----
    const int64_t item = i0 + tid;
    const bool have = item < ie;
    float acc[TU];
#pragma unroll
    for (int u = 0; u < TU; ++u) acc[u] = 0.f;
    if (have) {
      const T* vrow = V + item * d;
      for (int k = 0; k < d; k += 8) {
        float v[8];
        rt_load8(vrow + k, v);
#pragma unroll
        for (int u = 0; u < TU; ++u) {
          const float4 a0 = *reinterpret_cast<const float4*>(Us + u * d + k);
          const float4 a1 = *reinterpret_cast<const float4*>(Us + u * d + k + 4);
          float s = acc[u];
          s = fmaf(a0.x, v[0], s); s = fmaf(a0.y, v[1], s); s = fmaf(a0.z, v[2], s); s = fmaf(a0.w, v[3], s);
          s = fmaf(a1.x, v[4], s); s = fmaf(a1.y, v[5], s); s = fmaf(a1.z, v[6], s); s = fmaf(a1.w, v[7], s);
          acc[u] = s;
        }
      }
    }
    __syncthreads();   // bitmask complete
    if (have) {
      float bias = 0.f;
      if constexpr (kBias) bias = __ldg(item_bias + item);
#pragma unroll
      for (int u = 0; u < TU; ++u) {
        float s = acc[u];
        if constexpr (kBias) s += bias;
        if (seen_ptr && ((bits[u * kWords + warp] >> lane) & 1u)) s = masked_score;
        if (s == 0.f) s = 0.f;                       // -0 ranks like +0
        if (!(s > -INFINITY)) continue;              // excluded (-inf) or NaN: never returned
        const uint64_t key = rt_key(s, (uint32_t)item);
        if (key > thr[u]) {
          const int p = atomicAdd(cnt + u, 1);
          keys[(size_t)u * CAP + p] = key;
        }
      }
    }
    __syncthreads();
    bool full = false;
#pragma unroll
    for (int u = 0; u < TU; ++u) full |= cnt[u] > CAP - kRtTile;   // the next tile could overflow the buffer
    if (full) rt_compact<TU>(keys, cnt, thr, K);
  }
  rt_compact<TU>(keys, cnt, thr, K);

  for (int i = tid; i < TU * K; i += kRtThreads) {
    const int u = i / K, j = i - u * K;
    const int64_t b = b0 + u;
    if (b >= B) continue;
    const uint64_t key = keys[(size_t)u * CAP + j];     // zero beyond the user's count: padding
    if (partial) {
      partial[((int64_t)split * B + b) * K + j] = key;
    } else {
      int64_t id; float s;
      rt_decode(key, id, s);
      out_ids[b * K + j] = id;
      out_scores[b * K + j] = s;
    }
  }
}

template <typename T, int TU>
__global__ void __launch_bounds__(kRtThreads)
recommend_topk_kernel(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                      const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ seen_ptr,
                      const int32_t* __restrict__ seen_idx, int seen_by_row, float masked_score, int K, int64_t per_split,
                      uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids, float* __restrict__ out_scores,
                      int32_t* err) {
  recommend_topk_body<T, TU, false>(U, nU, V, nI, d, uids, B, seen_ptr, seen_idx, seen_by_row, masked_score, K, per_split,
                                    partial, out_ids, out_scores, err, nullptr);
}

template <typename T, int TU>
__global__ void __launch_bounds__(kRtThreads)
recommend_topk_bias_kernel(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                           const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ seen_ptr,
                           const int32_t* __restrict__ seen_idx, int seen_by_row, float masked_score, int K,
                           int64_t per_split, uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids,
                           float* __restrict__ out_scores, int32_t* err, const float* __restrict__ item_bias) {
  recommend_topk_body<T, TU, true>(U, nU, V, nI, d, uids, B, seen_ptr, seen_idx, seen_by_row, masked_score, K, per_split,
                                   partial, out_ids, out_scores, err, item_bias);
}

// Row b: the K best of the S per-split lists partial[s][b][0..K).
__global__ void __launch_bounds__(kRtThreads)
recommend_merge_kernel(const uint64_t* __restrict__ partial, int S, int64_t B, int K, int P, int64_t* __restrict__ out_ids,
                       float* __restrict__ out_scores) {
  extern __shared__ __align__(16) uint64_t rt_smem[];
  const int64_t b = blockIdx.x;
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    uint64_t key = 0;
    if (i < S * K) {
      const int s = i / K, j = i - s * K;
      key = partial[((int64_t)s * B + b) * K + j];
    }
    rt_smem[i] = key;
  }
  __syncthreads();
  rt_bitonic_desc(rt_smem, 1, P);
  for (int j = threadIdx.x; j < K; j += blockDim.x) {
    int64_t id; float s;
    rt_decode(rt_smem[j], id, s);
    out_ids[b * K + j] = id;
    out_scores[b * K + j] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Subset-restricted retrieval. Row b ranks only the items of subset subset_ids[b] (an ascending id list of the subset
// CSR; -1 = the whole catalog). Rows are grouped by subset on the device so that the TU users of a block share one list;
// the block streams that list in tiles of 256 ids, gathering the item rows, and otherwise runs the path above. Groups:
// g < G the subsets, G the whole catalog, G + 1 rows with an invalid subset id (an empty list: all-padding rows).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kRsPlanThreads = 1024;

__device__ __forceinline__ int rs_group(const int64_t* subset_ids, int64_t b, int G, int32_t* err) {
  const int64_t s = subset_ids[b];
  if (s == -1) return G;
  if (s < -1 || s >= G) {
    if (err) atomicOr(err, 2);
    return G + 1;
  }
  return (int)s;
}

// One block. Counting sort of the B rows by group: order[rows_at[g] .. rows_at[g + 1]) = the rows of group g (in no
// particular order: a row's result does not depend on the rows it shares a block with), and blocks_at[g] = the first
// scoring block of group g (ceil(rows / TU) blocks per group; blocks_at[G + 2] = all of them). cursor: G + 2 ints.
__global__ void __launch_bounds__(kRsPlanThreads)
recommend_subset_plan_kernel(const int64_t* __restrict__ subset_ids, int B, int G, int TU, int32_t* __restrict__ cursor,
                             int32_t* __restrict__ rows_at, int32_t* __restrict__ blocks_at, int32_t* __restrict__ order,
                             int32_t* err) {
  __shared__ long long wsum[kRsPlanThreads / 32];
  __shared__ long long carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ng = G + 2;
  for (int g = tid; g < ng; g += kRsPlanThreads) cursor[g] = 0;
  if (tid == 0) carry = 0;
  __syncthreads();
  // histogram; lanes of a warp with the same group add once
  for (int b0 = 0; b0 < B; b0 += kRsPlanThreads) {
    const int b = b0 + tid;
    const int g = b < B ? rs_group(subset_ids, b, G, err) : -1;
    const unsigned same = __match_any_sync(kFull, g);
    if (g >= 0 && lane == __ffs(same) - 1) atomicAdd(cursor + g, __popc(same));
  }
  __syncthreads();
  // exclusive scan of (blocks << 32 | rows) over the groups
  for (int g0 = 0; g0 < ng; g0 += kRsPlanThreads) {
    const int g = g0 + tid;
    const int c = g < ng ? __ldcg(cursor + g) : 0;   // the histogram's atomics live in L2
    const long long v = ((long long)((c + TU - 1) / TU) << 32) | (long long)c;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long y = __shfl_up_sync(kFull, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      long long w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(kFull, w, o);
        if (lane >= o) w += y;
      }
      wsum[lane] = w;
    }
    __syncthreads();
    const long long ex = carry + (warp ? wsum[warp - 1] : 0) + x - v;
    if (g < ng) {
      rows_at[g] = (int32_t)(ex & 0xffffffffll);
      blocks_at[g] = (int32_t)(ex >> 32);
      cursor[g] = (int32_t)(ex & 0xffffffffll);
    }
    __syncthreads();
    if (tid == 0) carry += wsum[kRsPlanThreads / 32 - 1];
    __syncthreads();
  }
  if (tid == 0) {
    rows_at[ng] = B;
    blocks_at[ng] = (int32_t)(carry >> 32);
  }
  // scatter; groups re-read from subset_ids (err is already set)
  for (int b0 = 0; b0 < B; b0 += kRsPlanThreads) {
    const int b = b0 + tid;
    const int g = b < B ? rs_group(subset_ids, b, G, nullptr) : -1;
    const unsigned same = __match_any_sync(kFull, g);
    const int leader = __ffs(same) - 1;
    int base = 0;
    if (g >= 0 && lane == leader) base = atomicAdd(cursor + g, __popc(same));
    base = __shfl_sync(kFull, base, leader);
    if (g >= 0) order[base + __popc(same & ((1u << lane) - 1))] = b;
  }
}

// Grid (upper bound on the plan's block count, S). Block x takes TU rows of one group and split y of the group's list:
// a slice of at least kRtMinSplit ids (a multiple of the tile) so that groups shorter than the longest use fewer splits;
// a split past the end of its list writes padding keys.
// kBias: score + item_bias[item] (recommend_subset_bias_kernel).
template <typename T, int TU, bool kBias>
__device__ __forceinline__ void
recommend_subset_body(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                      const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ sub_ptr,
                      const int32_t* __restrict__ sub_idx, int G, const int32_t* __restrict__ rows_at,
                      const int32_t* __restrict__ blocks_at, const int32_t* __restrict__ order,
                      const int32_t* __restrict__ seen_ptr, const int32_t* __restrict__ seen_idx, int K, int S,
                      uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids, float* __restrict__ out_scores,
                      int32_t* err, const float* __restrict__ item_bias) {
  constexpr int CAP = kRtEntries / TU;
  constexpr int kWords = kRtTile / 32;
  extern __shared__ __align__(16) uint64_t rt_smem[];
  uint64_t* keys = rt_smem;                                    // [TU][CAP]
  uint64_t* thr = keys + kRtEntries;                           // [TU]; ~0 = inactive row (no candidate beats it)
  float* Us = reinterpret_cast<float*>(thr + TU);              // [TU][d]
  uint32_t* bits = reinterpret_cast<uint32_t*>(Us + (size_t)TU * d);   // [TU][kWords]: seen items of the tile, by position
  int* cnt = reinterpret_cast<int*>(bits + TU * kWords);       // [TU]
  int* mcur = cnt + TU;                                        // [TU]: next unconsumed entry of the seen list
  int* mend = mcur + TU;                                       // [TU]
  int* rowb = mend + TU;                                       // [TU]: batch row of each user, -1 = none
  int* sid = rowb + TU;                                        // [kRtTile]: item ids of the tile, ascending

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int blk = blockIdx.x, split = blockIdx.y;
  if (blk >= blocks_at[G + 2]) return;
  int lo = 0, hi = G + 2;                                      // group: the last g with blocks_at[g] <= blk
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (blocks_at[mid] <= blk) lo = mid + 1; else hi = mid;
  }
  const int g = lo - 1;
  const int r0 = rows_at[g] + (blk - blocks_at[g]) * TU;
  const int nr = min(TU, rows_at[g + 1] - r0);
  const int32_t* list = g < G ? sub_idx + sub_ptr[g] : nullptr;   // null: the identity (whole catalog)
  const int64_t len = g < G ? sub_ptr[g + 1] - sub_ptr[g] : g == G ? nI : 0;
  int64_t per = max((len + S - 1) / S, (int64_t)kRtMinSplit);
  per = (per + kRtTile - 1) / kRtTile * kRtTile;
  const int64_t pb = min(len, (int64_t)split * per);
  const int64_t pe = min(len, pb + per);

  if (tid < TU) {
    const int b = tid < nr ? order[r0 + tid] : -1;
    bool active = false;
    int c = 0, en = 0;
    if (b >= 0) {
      const int64_t uid = uids[b];
      active = uid >= 0 && uid < nU;
      if (!active && err) atomicOr(err, 1);
      if (active && seen_ptr && pb < pe) {
        c = seen_ptr[uid]; en = seen_ptr[uid + 1];
        const int64_t first = list ? list[pb] : pb;
        int l = c, h = en;                         // first seen entry >= the split's first id (lists ascending)
        while (l < h) {
          const int mid = (l + h) >> 1;
          if (seen_idx[mid] < first) l = mid + 1; else h = mid;
        }
        c = l;
      }
    }
    rowb[tid] = b;
    thr[tid] = active ? 0ull : ~0ull;
    cnt[tid] = 0;
    mcur[tid] = c; mend[tid] = en;
  }
  __syncthreads();
  if (pb < pe) {
    for (int i = tid; i < TU * d; i += kRtThreads) {
      const int u = i / d, k = i - u * d;
      float x = 0.f;
      if (thr[u] == 0ull) x = rt_to_float(U[uids[rowb[u]] * d + k]);
      Us[i] = x;
    }
    for (int64_t p0 = pb; p0 < pe; p0 += kRtTile) {
      const int n = (int)min((int64_t)kRtTile, pe - p0);
      for (int i = tid; i < TU * kWords; i += kRtThreads) bits[i] = 0;
      if (tid < n) sid[tid] = list ? list[p0 + tid] : (int)(p0 + tid);
      __syncthreads();
      // ---- seen items of this tile -> bitmask by tile position (one warp per user, the sorted list consumed in order) ----
      if (seen_ptr) {
        const int last = sid[n - 1];
        for (int u = warp; u < TU; u += kRtThreads / 32) {
          int c = mcur[u];
          const int en = mend[u];
          while (c < en) {
            const int p = c + lane;
            const int it = (p < en) ? seen_idx[p] : INT32_MAX;
            const bool in = it <= last;
            if (in) {
              int l = 0, h = n;                    // position of `it` among the tile's ids, if it is one
              while (l < h) {
                const int mid = (l + h) >> 1;
                if (sid[mid] < it) l = mid + 1; else h = mid;
              }
              if (l < n && sid[l] == it) atomicOr(bits + u * kWords + (l >> 5), 1u << (l & 31));
            }
            const int m = __popc(__ballot_sync(kFull, in));
            c += m;
            if (m < 32) break;
          }
          if (lane == 0) mcur[u] = c;
        }
      }
      // ---- scores of my item against every user of the block: one fma chain each, k ascending ----
      const bool have = tid < n;
      const int item = have ? sid[tid] : 0;
      float acc[TU];
      rt_score<T, TU>(have ? V + (int64_t)item * d : nullptr, Us, d, acc);
      __syncthreads();   // bitmask complete, tile ids consumed
      if (have) {
        float bias = 0.f;
        if constexpr (kBias) bias = __ldg(item_bias + item);
#pragma unroll
        for (int u = 0; u < TU; ++u) {
          if (seen_ptr && ((bits[u * kWords + warp] >> lane) & 1u)) continue;
          rt_offer<TU>(keys, cnt, thr, u, kBias ? acc[u] + bias : acc[u], (uint32_t)item);
        }
      }
      __syncthreads();
      bool full = p0 + kRtTile >= pe;              // the last tile: truncate to the K best
#pragma unroll
      for (int u = 0; u < TU; ++u) full |= cnt[u] > CAP - kRtTile;   // the next tile could overflow a buffer
      if (full) rt_compact<TU>(keys, cnt, thr, K);
    }
  }

  for (int i = tid; i < TU * K; i += kRtThreads) {
    const int u = i / K, j = i - u * K;
    const int b = rowb[u];
    if (b < 0) continue;
    const uint64_t key = pb < pe ? keys[(size_t)u * CAP + j] : 0;   // zero beyond the user's count: padding
    if (partial) {
      partial[((int64_t)split * B + b) * K + j] = key;
    } else {
      int64_t id; float s;
      rt_decode(key, id, s);
      out_ids[(int64_t)b * K + j] = id;
      out_scores[(int64_t)b * K + j] = s;
    }
  }
}

template <typename T, int TU>
__global__ void __launch_bounds__(kRtThreads, 2)   // 2 blocks an SM: up to 128 registers, no spills
recommend_subset_kernel(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                        const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ sub_ptr,
                        const int32_t* __restrict__ sub_idx, int G, const int32_t* __restrict__ rows_at,
                        const int32_t* __restrict__ blocks_at, const int32_t* __restrict__ order,
                        const int32_t* __restrict__ seen_ptr, const int32_t* __restrict__ seen_idx, int K, int S,
                        uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids, float* __restrict__ out_scores,
                        int32_t* err) {
  recommend_subset_body<T, TU, false>(U, nU, V, nI, d, uids, B, sub_ptr, sub_idx, G, rows_at, blocks_at, order, seen_ptr,
                                      seen_idx, K, S, partial, out_ids, out_scores, err, nullptr);
}

template <typename T, int TU>
__global__ void __launch_bounds__(kRtThreads, 2)
recommend_subset_bias_kernel(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int64_t nI, int d,
                             const int64_t* __restrict__ uids, int64_t B, const int32_t* __restrict__ sub_ptr,
                             const int32_t* __restrict__ sub_idx, int G, const int32_t* __restrict__ rows_at,
                             const int32_t* __restrict__ blocks_at, const int32_t* __restrict__ order,
                             const int32_t* __restrict__ seen_ptr, const int32_t* __restrict__ seen_idx, int K, int S,
                             uint64_t* __restrict__ partial, int64_t* __restrict__ out_ids,
                             float* __restrict__ out_scores, int32_t* err, const float* __restrict__ item_bias) {
  recommend_subset_body<T, TU, true>(U, nU, V, nI, d, uids, B, sub_ptr, sub_idx, G, rows_at, blocks_at, order, seen_ptr,
                                     seen_idx, K, S, partial, out_ids, out_scores, err, item_bias);
}

// ---------------------------------------------------------------------------------------------------------------------
// Radius-restricted retrieval. Row b ranks only the items i with ((c_x * p_x) + (c_y * p_y)) + (c_z * p_z) >= t_b in
// float64, every product and sum rounded on its own (__dmul_rn / __dadd_rn: no fma contraction): c = the row's centre
// (a unit vector), p = P[i] the item's unit vector, t_b = cos(radius / Earth radius), -inf for the whole Earth.
//
// Items are indexed by a grid of lat x lon cells w degrees on a side (lat band = floor((lat + 90) / w), lon band =
// floor((lon + 180) / w), both clamped to the grid; key = lat band * nlon + lon band): cell_items holds the item ids
// sorted by (key, id), cell_keys the ascending keys of the non-empty cells and cell_ptr their offsets into cell_items.
// The items of one lat band and a lon-band range are therefore one contiguous run of cell_items, and so are the items of
// a range of whole bands.
//
// recommend_geo_window_kernel gives every row a window of cells that covers its cap with one cell of margin: the lat
// bands of [lat - a - w, lat + a + w] (a = the cap's angular radius) and, per band, the lon bands of [lon - D - w,
// lon + D + w] (D = asin(sin a / cos lat), the cap's widest longitude offset), split in two at the antimeridian; every
// longitude when the cap comes within a cell of a pole, when D + w reaches 180 degrees or when the window spans more than
// kGeoMaxBands bands. The exact predicate decides membership; the window only has to be a superset. Rows are grouped by a
// hash of their window (recommend_subset_plan_kernel over the hash buckets), and recommend_geo_kernel streams each
// distinct window of its rows once for all of them.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kGeoMaxBands = 128;                  // wider windows take every longitude: one run of cell_items
constexpr int kGeoMaxSegs = 2 * kGeoMaxBands;      // runs of one window: two lon ranges per band (== kRtThreads)
constexpr int kGeoWin = 6;                         // window: lat bands [a, b], lon bands [lo0, hi0] and [lo1, hi1]
static_assert(kGeoMaxSegs <= kRtThreads, "one thread per run");

__device__ __forceinline__ int geo_band(double x, double w, int n) {   // floor(x / w) clamped to [0, n)
  const double f = floor(x / w);
  return f < 0.0 ? 0 : f >= (double)n ? n - 1 : (int)f;
}

// One thread per row: the window and its hash bucket (-1 for a non-finite centre or threshold: error bit 2, and an
// all-padding row). A zero centre or t <= -|c| takes the whole grid.
__global__ void __launch_bounds__(kRtThreads)
recommend_geo_window_kernel(const double* __restrict__ c, const double* __restrict__ t, int64_t B, double w, int nlat,
                            int nlon, int H, int32_t* __restrict__ win, int64_t* __restrict__ bucket, int32_t* err) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  constexpr double kDeg = 57.295779513082320876798;   // degrees per radian
  const double cx = c[3 * b], cy = c[3 * b + 1], cz = c[3 * b + 2], tb = t[b];
  int v[kGeoWin] = {0, nlat - 1, -1, 0, 0, -1};      // every cell; lo0 = -1: every longitude
  if (!isfinite(cx) || !isfinite(cy) || !isfinite(cz) || isnan(tb) || tb == INFINITY) {
    if (err) atomicOr(err, 2);
#pragma unroll
    for (int i = 0; i < kGeoWin; ++i) win[kGeoWin * b + i] = 0;
    bucket[b] = -1;
    return;
  }
  const double n = sqrt(cx * cx + cy * cy + cz * cz);
  if (n > 0.0 && tb / n > -1.0) {
    const double ct = fmin(tb / n, 1.0), z = fmax(-1.0, fmin(1.0, cz / n));
    const double a = acos(ct) * kDeg;
    const double lat = asin(z) * kDeg;
    const double lat_lo = lat - a - w, lat_hi = lat + a + w;
    v[0] = geo_band(lat_lo + 90.0, w, nlat);
    v[1] = geo_band(lat_hi + 90.0, w, nlat);
    if (lat_lo > -90.0 && lat_hi < 90.0 && v[1] - v[0] < kGeoMaxBands) {
      const double s = sqrt(fmax(0.0, 1.0 - ct * ct)) / sqrt(fmax(0.0, 1.0 - z * z));   // sin a / cos lat
      const double dl = s < 1.0 ? asin(s) * kDeg + w : 180.0;
      if (dl < 180.0) {
        const double lon = atan2(cy, cx) * kDeg;
        const double L = lon - dl, R = lon + dl;
        if (L >= -180.0 && R <= 180.0) {
          v[2] = geo_band(L + 180.0, w, nlon); v[3] = geo_band(R + 180.0, w, nlon);
        } else {                                     // across the antimeridian: [L', 180] and [-180, R']
          const double L2 = L < -180.0 ? L + 360.0 : L, R2 = R > 180.0 ? R - 360.0 : R;
          v[2] = geo_band(L2 + 180.0, w, nlon); v[3] = nlon - 1;
          v[4] = 0; v[5] = geo_band(R2 + 180.0, w, nlon);
          if (v[5] >= v[2]) { v[2] = -1; v[3] = 0; v[4] = 0; v[5] = -1; }   // the two ranges meet: every longitude
        }
      }
    }
  }
  uint32_t h = 2166136261u;                          // FNV-1a over the window, then a final mix
#pragma unroll
  for (int i = 0; i < kGeoWin; ++i) {
    win[kGeoWin * b + i] = v[i];
    h = (h ^ (uint32_t)v[i]) * 16777619u;
  }
  h ^= h >> 16; h *= 0x7feb352du; h ^= h >> 15;
  bucket[b] = (int64_t)(h & (uint32_t)(H - 1));
}

// First position in cell_items of the cells with key >= k.
__device__ __forceinline__ int geo_cell_lb(const int64_t* __restrict__ cell_keys, const int32_t* __restrict__ cell_ptr,
                                           int64_t nC, int64_t k) {
  int64_t lo = 0, hi = nC;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (cell_keys[mid] < k) lo = mid + 1; else hi = mid;
  }
  return cell_ptr[lo];
}

// Whether `item` is in the ascending list idx[lo, hi).
__device__ __forceinline__ bool geo_listed(const int32_t* __restrict__ idx, int lo, int hi, int item) {
  const int end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (idx[mid] < item) lo = mid + 1; else hi = mid;
  }
  return lo < end && idx[lo] == item;
}

// Grid (upper bound on the plan's block count, S), as recommend_subset_kernel: block x takes up to TU rows of one hash
// bucket (group H: rows with a non-finite centre or threshold, all padding), split y of each window. Rows of a bucket
// normally share one window; on a hash collision the block streams each distinct window of its rows in turn, and a row
// takes offers only during its own window. Window items come in cell order, not id order, so instead of the ascending
// seen cursor of the subset kernel a candidate that beats the row's current K-th best is looked up in the row's seen
// list (a binary search) before it enters the buffer: few items get that far once the thresholds settle.
// kBias: score + item_bias[item].
template <typename T, int TU, bool kBias>
__global__ void __launch_bounds__(kRtThreads, 2)   // 2 blocks an SM: up to 128 registers, no spills
recommend_geo_kernel(const T* __restrict__ U, int64_t nU, const T* __restrict__ V, int d, const int64_t* __restrict__ uids,
                     int64_t B, const int64_t* __restrict__ cell_keys, const int32_t* __restrict__ cell_ptr, int64_t nC,
                     const int32_t* __restrict__ cell_items, const double* __restrict__ P, int nlon,
                     const double* __restrict__ c, const double* __restrict__ t, const int32_t* __restrict__ win, int H,
                     const int32_t* __restrict__ rows_at, const int32_t* __restrict__ blocks_at,
                     const int32_t* __restrict__ order, const int32_t* __restrict__ seen_ptr,
                     const int32_t* __restrict__ seen_idx, int K, int S, uint64_t* __restrict__ partial,
                     int64_t* __restrict__ out_ids, float* __restrict__ out_scores, int32_t* err,
                     const float* __restrict__ item_bias) {
  constexpr int CAP = kRtEntries / TU;
  extern __shared__ __align__(16) uint64_t rt_smem[];
  uint64_t* keys = rt_smem;                                    // [TU][CAP]
  uint64_t* thr = keys + kRtEntries;                           // [TU]; ~0 = inactive row (no candidate beats it)
  double* cq = reinterpret_cast<double*>(thr + TU);            // [TU][4]: c_x, c_y, c_z, t of each row
  float* Us = reinterpret_cast<float*>(cq + 4 * TU);           // [TU][d]
  int* cnt = reinterpret_cast<int*>(Us + (size_t)TU * d);      // [TU]
  int* sb = cnt + TU;                                          // [TU]: the row's seen list, seen_idx[sb, se)
  int* se = sb + TU;                                           // [TU]
  int* rowb = se + TU;                                         // [TU]: batch row of each user, -1 = none
  int* pass = rowb + TU;                                       // [TU]: 0 to stream, 1 in the current window, 2 done
  int* wv = pass + TU;                                         // [8]: the current window
  int* seg = wv + 8;                                           // [kGeoMaxSegs]: first cell_items position of each run
  int* pref = seg + kGeoMaxSegs;                               // [kGeoMaxSegs + 1]: window position of each run
  int* misc = pref + kGeoMaxSegs + 1;                          // [16]: leader row, warp sums of the scan

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int blk = blockIdx.x, split = blockIdx.y;
  if (blk >= blocks_at[H + 2]) return;
  int lo = 0, hi = H + 2;                                      // group: the last g with blocks_at[g] <= blk
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (blocks_at[mid] <= blk) lo = mid + 1; else hi = mid;
  }
  const int g = lo - 1;
  const int r0 = rows_at[g] + (blk - blocks_at[g]) * TU;
  const int nr = min(TU, rows_at[g + 1] - r0);

  if (tid < TU) {
    const int b = tid < nr ? order[r0 + tid] : -1;
    bool active = false;
    int s0 = 0, s1 = 0;
    if (b >= 0) {
      const int64_t uid = uids[b];
      active = uid >= 0 && uid < nU;
      if (!active && err) atomicOr(err, 1);
      if (active && seen_ptr) { s0 = seen_ptr[uid]; s1 = seen_ptr[uid + 1]; }
      active = active && g < H;
      if (active) {
        cq[4 * tid] = c[3 * b]; cq[4 * tid + 1] = c[3 * b + 1]; cq[4 * tid + 2] = c[3 * b + 2]; cq[4 * tid + 3] = t[b];
      }
    }
    rowb[tid] = b;
    thr[tid] = active ? 0ull : ~0ull;
    cnt[tid] = 0;
    sb[tid] = s0; se[tid] = s1;
    pass[tid] = active ? 0 : 2;
  }
  __syncthreads();
  for (int i = tid; i < TU * d; i += kRtThreads) {
    const int u = i / d, k = i - u * d;
    float x = 0.f;
    if (thr[u] == 0ull) x = rt_to_float(U[uids[rowb[u]] * d + k]);
    Us[i] = x;
  }

  for (;;) {
    if (tid == 0) {
      int l = -1;
      for (int u = 0; u < TU && l < 0; ++u)
        if (pass[u] == 0) l = u;
      misc[0] = l;
    }
    __syncthreads();
    const int lead = misc[0];
    if (lead < 0) break;
    if (tid < kGeoWin) wv[tid] = win[(int64_t)kGeoWin * rowb[lead] + tid];
    __syncthreads();
    if (tid < TU && pass[tid] == 0) {
      bool same = true;
#pragma unroll
      for (int i = 0; i < kGeoWin; ++i) same = same && win[(int64_t)kGeoWin * rowb[tid] + i] == wv[i];
      if (same) pass[tid] = 1;
    }
    // ---- the window's runs of cell_items and their positions in the window (an exclusive scan of the lengths) ----
    const bool all_lon = wv[2] < 0;
    const int nseg = all_lon ? 1 : 2 * (wv[1] - wv[0] + 1);
    int len = 0;
    if (tid < nseg) {
      int64_t k0, k1;
      if (all_lon) {
        k0 = (int64_t)wv[0] * nlon; k1 = (int64_t)(wv[1] + 1) * nlon;
      } else {
        const int64_t band = (int64_t)(wv[0] + (tid >> 1)) * nlon;
        const int l = (tid & 1) ? wv[4] : wv[2], h = (tid & 1) ? wv[5] : wv[3];
        k0 = band + l; k1 = l <= h ? band + h + 1 : k0;
      }
      const int p0 = geo_cell_lb(cell_keys, cell_ptr, nC, k0);
      seg[tid] = p0;
      len = k1 > k0 ? geo_cell_lb(cell_keys, cell_ptr, nC, k1) - p0 : 0;
    }
    int x = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(kFull, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) misc[8 + warp] = x;
    __syncthreads();
    int base = 0;
    for (int i = 0; i < warp; ++i) base += misc[8 + i];
    if (tid < nseg) pref[tid] = base + x - len;
    if (tid == kRtThreads - 1) pref[nseg] = base + x;
    __syncthreads();
    const int64_t L = pref[nseg];
    const bool whole = L == cell_ptr[nC];          // every item: stream them in id order, no cell_items lookup
    int64_t per = max((L + S - 1) / S, (int64_t)kRtMinSplit);
    per = (per + kRtTile - 1) / kRtTile * kRtTile;
    const int64_t pb = min(L, (int64_t)split * per);
    const int64_t pe = min(L, pb + per);

    for (int64_t p0 = pb; p0 < pe; p0 += kRtTile) {
      const int64_t p = p0 + tid;
      int item = 0;
      unsigned in = 0;                             // bit u: the item is inside row u's radius (rows of this window)
      if (p < pe) {
        int l = 0, h = nseg;                       // the run holding p: the last j with pref[j] <= p
        while (!whole && h - l > 1) {
          const int mid = (l + h) >> 1;
          if (pref[mid] <= p) l = mid; else h = mid;
        }
        item = whole ? (int)p : cell_items[seg[l] + (int)(p - pref[l])];
        const double px = P[3 * (int64_t)item], py = P[3 * (int64_t)item + 1], pz = P[3 * (int64_t)item + 2];
#pragma unroll
        for (int u = 0; u < TU; ++u) {
          if (pass[u] != 1) continue;
          if (cq[4 * u + 3] == -INFINITY) { in |= 1u << u; continue; }   // every finite dot product is >= -inf
          const double dot = __dadd_rn(__dadd_rn(__dmul_rn(cq[4 * u], px), __dmul_rn(cq[4 * u + 1], py)),
                                       __dmul_rn(cq[4 * u + 2], pz));
          if (dot >= cq[4 * u + 3]) in |= 1u << u;
        }
      }
      float acc[TU];
      rt_score<T, TU>(in ? V + (int64_t)item * d : nullptr, Us, d, acc);
      if (in) {
        float bias = 0.f;
        if constexpr (kBias) bias = __ldg(item_bias + item);
#pragma unroll
        for (int u = 0; u < TU; ++u) {
          if (!((in >> u) & 1u)) continue;
          float s = kBias ? acc[u] + bias : acc[u];
          if (s == 0.f) s = 0.f;                   // -0 ranks like +0
          if (!(s > -INFINITY)) continue;          // -inf or NaN: never returned
          const uint64_t key = rt_key(s, (uint32_t)item);
          if (key <= thr[u]) continue;
          if (seen_ptr && geo_listed(seen_idx, sb[u], se[u], item)) continue;
          const int q = atomicAdd(cnt + u, 1);
          keys[(size_t)u * CAP + q] = key;
        }
      }
      __syncthreads();
      bool full = p0 + kRtTile >= pe;              // the last tile: truncate to the K best
#pragma unroll
      for (int u = 0; u < TU; ++u) full |= cnt[u] > CAP - kRtTile;   // the next tile could overflow a buffer
      if (full) rt_compact<TU>(keys, cnt, thr, K);
    }
    if (tid < TU && pass[tid] == 1) pass[tid] = 2;
    __syncthreads();
  }

  // every buffer that took an offer was truncated after its window's last tile: its first cnt keys are its K best
  for (int i = tid; i < TU * K; i += kRtThreads) {
    const int u = i / K, j = i - u * K;
    const int b = rowb[u];
    if (b < 0) continue;
    const uint64_t key = j < cnt[u] ? keys[(size_t)u * CAP + j] : 0;   // zero beyond the user's count: padding
    if (partial) {
      partial[((int64_t)split * B + b) * K + j] = key;
    } else {
      int64_t id; float s;
      rt_decode(key, id, s);
      out_ids[(int64_t)b * K + j] = id;
      out_scores[(int64_t)b * K + j] = s;
    }
  }
}

}  // namespace yr

using namespace yr;

namespace {

int rt_users_per_block(int K) { return K <= kRtEntries / 16 - kRtTile ? 16 : K <= kRtEntries / 8 - kRtTile ? 8 : 4; }

// Users per block of a launch: for d > 512 at most 8, so that the staged user rows (TU x d floats) never take more shared
// memory than 16 users at d = 512. Fewer users per block never means more item splits (rt_splits), so the workspace
// queries, which take rt_users_per_block(K), stay upper bounds.
int rt_users(int K, int d) { return d > kRtMaxUD / 16 ? std::min(rt_users_per_block(K), 8) : rt_users_per_block(K); }

// The widest d a launch with TU users per block can have.
int rt_max_d(int TU) { return std::min(kRtMaxD, kRtMaxUD / TU); }

int rt_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// Item splits: enough blocks to give every SM a few, each split at least kRtMinSplit items (a multiple of the tile), and the
// merge of S lists of K keys within one block's shared memory. TU: the users per block of the launch.
int rt_splits(int64_t B, int64_t nI, int K, int TU, int sm, int64_t* per_split) {
  const int64_t bx = (B + TU - 1) / TU;
  int64_t S = (4 * (int64_t)sm + bx - 1) / bx;
  const int64_t by_len = nI / kRtMinSplit;
  if (S > by_len) S = by_len;
  while (S > 1 && rt_pow2((int)(S * K)) > kRtMergeMax) --S;
  if (S < 1) S = 1;
  int64_t per = (nI + S - 1) / S;
  per = (per + kRtTile - 1) / kRtTile * kRtTile;
  *per_split = per;
  return (int)((nI + per - 1) / per);
}

size_t rt_smem_bytes(int TU, int d) {
  return (size_t)kRtEntries * 8 + (size_t)TU * 8 + (size_t)TU * d * 4 + (size_t)TU * (kRtTile / 32) * 4 + 3 * (size_t)TU * 4;
}

template <typename T, int TU, bool kBias>
int rt_launch(const void* U, int64_t nU, const void* V, int64_t nI, int d, const int64_t* uids, int64_t B,
              const int32_t* seen_ptr, const int32_t* seen_idx, int seen_by_row, float masked_score, int K, int S,
              int64_t per_split, uint64_t* partial, int64_t* out_ids, float* out_scores, int32_t* err,
              const float* item_bias, cudaStream_t s) {
  static AttrOnce attr;
  const size_t smem = rt_smem_bytes(TU, d);
  const int max_smem = (int)rt_smem_bytes(TU, rt_max_d(TU));
  dim3 grid((unsigned)((B + TU - 1) / TU), (unsigned)S);
  const T* Ut = reinterpret_cast<const T*>(U);
  const T* Vt = reinterpret_cast<const T*>(V);
  if constexpr (kBias) {
    int rc = attr.set(recommend_topk_bias_kernel<T, TU>, max_smem);
    if (rc) return rc;
    recommend_topk_bias_kernel<T, TU><<<grid, kRtThreads, smem, s>>>(Ut, nU, Vt, nI, d, uids, B, seen_ptr, seen_idx,
                                                                     seen_by_row, masked_score, K, per_split, partial,
                                                                     out_ids, out_scores, err, item_bias);
  } else {
    int rc = attr.set(recommend_topk_kernel<T, TU>, max_smem);
    if (rc) return rc;
    recommend_topk_kernel<T, TU><<<grid, kRtThreads, smem, s>>>(Ut, nU, Vt, nI, d, uids, B, seen_ptr, seen_idx,
                                                                seen_by_row, masked_score, K, per_split, partial, out_ids,
                                                                out_scores, err);
  }
  YR_CHECK_LAUNCH();
  return YR_OK;
}

size_t rs_smem_bytes(int TU, int d) { return rt_smem_bytes(TU, d) + (size_t)TU * 4 + (size_t)kRtTile * 4; }

template <typename T, int TU, bool kBias>
int rs_launch(const void* U, int64_t nU, const void* V, int64_t nI, int d, const int64_t* uids, int64_t B,
              const int32_t* sub_ptr, const int32_t* sub_idx, int G, const int32_t* rows_at, const int32_t* blocks_at,
              const int32_t* order, const int32_t* seen_ptr, const int32_t* seen_idx, int K, int S, uint64_t* partial,
              int64_t* out_ids, float* out_scores, int32_t* err, const float* item_bias, cudaStream_t s) {
  static AttrOnce attr;
  const int max_smem = (int)rs_smem_bytes(TU, rt_max_d(TU));
  // the plan makes sum over groups of ceil(rows / TU) blocks: at most ceil(B / TU) + one per non-empty group
  dim3 grid((unsigned)((B + TU - 1) / TU + std::min<int64_t>((int64_t)G + 2, B)), (unsigned)S);
  const size_t smem = rs_smem_bytes(TU, d);
  const T* Ut = reinterpret_cast<const T*>(U);
  const T* Vt = reinterpret_cast<const T*>(V);
  if constexpr (kBias) {
    int rc = attr.set(recommend_subset_bias_kernel<T, TU>, max_smem);
    if (rc) return rc;
    recommend_subset_bias_kernel<T, TU><<<grid, kRtThreads, smem, s>>>(Ut, nU, Vt, nI, d, uids, B, sub_ptr, sub_idx, G,
                                                                       rows_at, blocks_at, order, seen_ptr, seen_idx, K,
                                                                       S, partial, out_ids, out_scores, err, item_bias);
  } else {
    int rc = attr.set(recommend_subset_kernel<T, TU>, max_smem);
    if (rc) return rc;
    recommend_subset_kernel<T, TU><<<grid, kRtThreads, smem, s>>>(Ut, nU, Vt, nI, d, uids, B, sub_ptr, sub_idx, G,
                                                                  rows_at, blocks_at, order, seen_ptr, seen_idx, K, S,
                                                                  partial, out_ids, out_scores, err);
  }
  YR_CHECK_LAUNCH();
  return YR_OK;
}

int rs_splits(int64_t B, int64_t max_len, int K, int TU) {
  int64_t per = 0;
  return rt_splits(B, std::max<int64_t>(max_len, 1), K, TU, yr_sm_count(), &per);
}

size_t rs_partial_bytes(int S, int64_t B, int K) { return S > 1 ? (size_t)S * (size_t)B * (size_t)K * sizeof(uint64_t) : 0; }

size_t rs_plan_bytes(int64_t B, int G) { return ((size_t)3 * G + 8 + (size_t)B) * sizeof(int32_t); }

size_t geo_smem_bytes(int TU, int d) {
  return (size_t)kRtEntries * 8 + (size_t)TU * 8 + (size_t)TU * 4 * 8 + (size_t)TU * d * 4 + 5 * (size_t)TU * 4 +
         (size_t)(8 + 2 * kGeoMaxSegs + 1 + 16) * 4;
}

// Hash buckets of the row grouping: about two per row (few collisions), at most 2^16 (the plan scans them all).
int geo_buckets(int64_t B) {
  int64_t H = 64;
  while (H < 2 * B && H < (1 << 16)) H <<= 1;
  return (int)H;
}

// Workspace: per-split lists | bucket int64 [B] | plan | windows int32 [B][kGeoWin].
size_t geo_ws_bytes(int S, int64_t B, int K) {
  return rs_partial_bytes(S, B, K) + (size_t)B * 8 + rs_plan_bytes(B, geo_buckets(B)) + (size_t)B * kGeoWin * 4;
}

template <typename T, int TU, bool kBias>
int geo_launch(const void* U, int64_t nU, const void* V, int d, const int64_t* uids, int64_t B, const int64_t* cell_keys,
               const int32_t* cell_ptr, int64_t nC, const int32_t* cell_items, const double* P, int nlon, const double* c,
               const double* t, const int32_t* win, int H, const int32_t* rows_at, const int32_t* blocks_at,
               const int32_t* order, const int32_t* seen_ptr, const int32_t* seen_idx, int K, int S, uint64_t* partial,
               int64_t* out_ids, float* out_scores, int32_t* err, const float* item_bias, cudaStream_t s) {
  static AttrOnce attr;
  int rc = attr.set(recommend_geo_kernel<T, TU, kBias>, (int)geo_smem_bytes(TU, rt_max_d(TU)));
  if (rc) return rc;
  dim3 grid((unsigned)((B + TU - 1) / TU + std::min<int64_t>((int64_t)H + 2, B)), (unsigned)S);
  recommend_geo_kernel<T, TU, kBias><<<grid, kRtThreads, geo_smem_bytes(TU, d), s>>>(
      reinterpret_cast<const T*>(U), nU, reinterpret_cast<const T*>(V), d, uids, B, cell_keys, cell_ptr, nC, cell_items,
      P, nlon, c, t, win, H, rows_at, blocks_at, order, seen_ptr, seen_idx, K, S, partial, out_ids, out_scores, err,
      item_bias);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

int merge_launch(const uint64_t* partial, int S, int64_t B, int K, int64_t* out_ids, float* out_scores, cudaStream_t s) {
  const int P = rt_pow2(S * K);
  static AttrOnce attr;
  int rc = attr.set(recommend_merge_kernel, kRtMergeMax * (int)sizeof(uint64_t));
  if (rc) return rc;
  recommend_merge_kernel<<<(unsigned)B, kRtThreads, (size_t)P * sizeof(uint64_t), s>>>(partial, S, B, K, P, out_ids,
                                                                                     out_scores);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

}  // namespace

extern "C" size_t yr_recommend_ws_bytes(int64_t B, int64_t nI, int K) {
  if (B <= 0 || nI <= 0 || K <= 0 || K > kRtMaxK) return 0;
  int64_t per = 0;
  const int S = rt_splits(B, nI, K, rt_users_per_block(K), yr_sm_count(), &per);
  return rs_partial_bytes(S, B, K);
}

extern "C" int yr_recommend_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                 const int64_t* user_ids, int64_t B, const int32_t* seen_ptr, const int32_t* seen_idx,
                                 int seen_by_row, float masked_score, int K, int64_t* out_ids, float* out_scores, void* ws,
                                 size_t ws_bytes, int32_t* err, yr_stream stream) {
  return yr_recommend_topk_ex(U, nU, V, nI, d, dtype, user_ids, B, seen_ptr, seen_idx, seen_by_row, masked_score, K,
                              out_ids, out_scores, ws, ws_bytes, err, stream, nullptr);
}

extern "C" int yr_recommend_topk_ex(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                    const int64_t* user_ids, int64_t B, const int32_t* seen_ptr, const int32_t* seen_idx,
                                    int seen_by_row, float masked_score, int K, int64_t* out_ids, float* out_scores,
                                    void* ws, size_t ws_bytes, int32_t* err, yr_stream stream, const float* item_bias) {
  if (!U || !V || !out_ids || !out_scores || (B > 0 && !user_ids)) return YR_ERR_BAD_ARG;
  if ((seen_ptr == nullptr) != (seen_idx == nullptr)) return YR_ERR_BAD_ARG;
  if (B < 0 || nU <= 0 || K <= 0 || K > kRtMaxK) return YR_ERR_BAD_ARG;
  if (nI <= 0 || nI >= 0x7fffffffLL || d <= 0 || d > kRtMaxD || (d & 7) != 0) return YR_ERR_BAD_DIM;
  if (dtype != YR_DTYPE_F32 && dtype != YR_DTYPE_BF16) return YR_ERR_BAD_ARG;
  if (B == 0) return YR_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const int TU = rt_users(K, d);
  int64_t per = 0;
  const int S = rt_splits(B, nI, K, TU, yr_sm_count(), &per);
  uint64_t* partial = nullptr;
  if (S > 1) {
    if (!ws || ws_bytes < rs_partial_bytes(S, B, K)) return YR_ERR_WORKSPACE;
    partial = reinterpret_cast<uint64_t*>(ws);
  }
  int rc;
#define YR_RT_LAUNCH(T, TU_, BIAS)                                                                                        \
  rt_launch<T, TU_, BIAS>(U, nU, V, nI, d, user_ids, B, seen_ptr, seen_idx, seen_by_row, masked_score, K, S, per,        \
                          partial, out_ids, out_scores, err, item_bias, s)
#define YR_RT_TU(T, BIAS)                                                                                                 \
  (TU == 16 ? YR_RT_LAUNCH(T, 16, BIAS) : TU == 8 ? YR_RT_LAUNCH(T, 8, BIAS) : YR_RT_LAUNCH(T, 4, BIAS))
  if (dtype == YR_DTYPE_F32)
    rc = item_bias ? YR_RT_TU(float, true) : YR_RT_TU(float, false);
  else
    rc = item_bias ? YR_RT_TU(__nv_bfloat16, true) : YR_RT_TU(__nv_bfloat16, false);
#undef YR_RT_TU
#undef YR_RT_LAUNCH
  if (rc || S == 1) return rc;
  return merge_launch(partial, S, B, K, out_ids, out_scores, s);
}

extern "C" size_t yr_recommend_subset_ws_bytes(int64_t B, int G, int64_t max_subset_len, int K) {
  if (B <= 0 || G < 0 || K <= 0 || K > kRtMaxK) return 0;
  return rs_partial_bytes(rs_splits(B, max_subset_len, K, rt_users_per_block(K)), B, K) + rs_plan_bytes(B, G);
}

extern "C" int yr_recommend_subset_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                        const int64_t* user_ids, int64_t B, const int32_t* subset_ptr,
                                        const int32_t* subset_idx, int G, int64_t max_subset_len,
                                        const int64_t* subset_ids, const int32_t* seen_ptr, const int32_t* seen_idx, int K,
                                        int64_t* out_ids, float* out_scores, void* ws, size_t ws_bytes, int32_t* err,
                                        yr_stream stream) {
  return yr_recommend_subset_topk_ex(U, nU, V, nI, d, dtype, user_ids, B, subset_ptr, subset_idx, G, max_subset_len,
                                     subset_ids, seen_ptr, seen_idx, K, out_ids, out_scores, ws, ws_bytes, err, stream,
                                     nullptr);
}

extern "C" int yr_recommend_subset_topk_ex(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                           const int64_t* user_ids, int64_t B, const int32_t* subset_ptr,
                                           const int32_t* subset_idx, int G, int64_t max_subset_len,
                                           const int64_t* subset_ids, const int32_t* seen_ptr, const int32_t* seen_idx,
                                           int K, int64_t* out_ids, float* out_scores, void* ws, size_t ws_bytes,
                                           int32_t* err, yr_stream stream, const float* item_bias) {
  if (!U || !V || !out_ids || !out_scores || !subset_ptr || !subset_idx) return YR_ERR_BAD_ARG;
  if (B > 0 && (!user_ids || !subset_ids)) return YR_ERR_BAD_ARG;
  if ((seen_ptr == nullptr) != (seen_idx == nullptr)) return YR_ERR_BAD_ARG;
  if (B < 0 || B >= 0x7fffffffLL || G < 0 || G >= 0x7ffffff0 || max_subset_len < 0 || nU <= 0 || K <= 0 ||
      K > kRtMaxK)
    return YR_ERR_BAD_ARG;
  if (nI <= 0 || nI >= 0x7fffffffLL || d <= 0 || d > kRtMaxD || (d & 7) != 0) return YR_ERR_BAD_DIM;
  if (dtype != YR_DTYPE_F32 && dtype != YR_DTYPE_BF16) return YR_ERR_BAD_ARG;
  if (B == 0) return YR_OK;
  const int TU = rt_users(K, d);
  const int S = rs_splits(B, max_subset_len, K, TU);
  const size_t pbytes = rs_partial_bytes(S, B, K);
  if (!ws || ws_bytes < pbytes + rs_plan_bytes(B, G)) return YR_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  uint64_t* partial = S > 1 ? reinterpret_cast<uint64_t*>(ws) : nullptr;
  int32_t* cursor = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(ws) + pbytes);   // [G + 2]
  int32_t* rows_at = cursor + G + 2;                                                      // [G + 3]
  int32_t* blocks_at = rows_at + G + 3;                                                   // [G + 3]
  int32_t* order = blocks_at + G + 3;                                                     // [B]
  recommend_subset_plan_kernel<<<1, kRsPlanThreads, 0, s>>>(subset_ids, (int)B, G, TU, cursor, rows_at, blocks_at, order,
                                                            err);
  YR_CHECK_LAUNCH();
  int rc;
#define YR_RS_LAUNCH(T, TU_, BIAS)                                                                                        \
  rs_launch<T, TU_, BIAS>(U, nU, V, nI, d, user_ids, B, subset_ptr, subset_idx, G, rows_at, blocks_at, order, seen_ptr,  \
                          seen_idx, K, S, partial, out_ids, out_scores, err, item_bias, s)
#define YR_RS_TU(T, BIAS)                                                                                                 \
  (TU == 16 ? YR_RS_LAUNCH(T, 16, BIAS) : TU == 8 ? YR_RS_LAUNCH(T, 8, BIAS) : YR_RS_LAUNCH(T, 4, BIAS))
  if (dtype == YR_DTYPE_F32)
    rc = item_bias ? YR_RS_TU(float, true) : YR_RS_TU(float, false);
  else
    rc = item_bias ? YR_RS_TU(__nv_bfloat16, true) : YR_RS_TU(__nv_bfloat16, false);
#undef YR_RS_TU
#undef YR_RS_LAUNCH
  if (rc || S == 1) return rc;
  return merge_launch(partial, S, B, K, out_ids, out_scores, s);
}

extern "C" size_t yr_recommend_geo_ws_bytes(int64_t B, int64_t nI, int K) {
  if (B <= 0 || B >= 0x7fffffffLL || nI <= 0 || K <= 0 || K > kRtMaxK) return 0;
  return geo_ws_bytes(rs_splits(B, nI, K, rt_users_per_block(K)), B, K);
}

extern "C" int yr_recommend_geo_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                     const int64_t* user_ids, int64_t B, const int64_t* cell_keys,
                                     const int32_t* cell_ptr, int64_t num_cells, const int32_t* cell_items,
                                     const double* item_xyz, double cell_deg, int64_t num_lat, int64_t num_lon,
                                     const double* centre_xyz, const double* threshold, const int32_t* seen_ptr,
                                     const int32_t* seen_idx, int K, int64_t* out_ids, float* out_scores, void* ws,
                                     size_t ws_bytes, int32_t* err, yr_stream stream, const float* item_bias) {
  if (!U || !V || !out_ids || !out_scores || !cell_keys || !cell_ptr || !cell_items || !item_xyz) return YR_ERR_BAD_ARG;
  if (B > 0 && (!user_ids || !centre_xyz || !threshold)) return YR_ERR_BAD_ARG;
  if ((seen_ptr == nullptr) != (seen_idx == nullptr)) return YR_ERR_BAD_ARG;
  if (B < 0 || B >= 0x7fffffffLL || nU <= 0 || K <= 0 || K > kRtMaxK) return YR_ERR_BAD_ARG;
  if (!(cell_deg > 0.0) || !(cell_deg <= 360.0) || num_lat < 1 || num_lon < 1 || num_lat > 0x7fffffffLL ||
      num_lon > 0x7fffffffLL || num_cells < 0 || num_cells > nI)
    return YR_ERR_BAD_ARG;
  if (nI <= 0 || nI >= 0x7fffffffLL || d <= 0 || d > kRtMaxD || (d & 7) != 0) return YR_ERR_BAD_DIM;
  if (dtype != YR_DTYPE_F32 && dtype != YR_DTYPE_BF16) return YR_ERR_BAD_ARG;
  if (B == 0) return YR_OK;
  const int TU = rt_users(K, d);
  const int S = rs_splits(B, nI, K, TU);
  const int H = geo_buckets(B);
  if (!ws || ws_bytes < geo_ws_bytes(S, B, K)) return YR_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t pbytes = rs_partial_bytes(S, B, K);
  uint64_t* partial = S > 1 ? reinterpret_cast<uint64_t*>(ws) : nullptr;
  int64_t* bucket = reinterpret_cast<int64_t*>(reinterpret_cast<char*>(ws) + pbytes);   // [B]
  int32_t* cursor = reinterpret_cast<int32_t*>(bucket + B);                              // [H + 2]
  int32_t* rows_at = cursor + H + 2;                                                      // [H + 3]
  int32_t* blocks_at = rows_at + H + 3;                                                   // [H + 3]
  int32_t* order = blocks_at + H + 3;                                                     // [B]
  int32_t* win = order + B;                                                               // [B][kGeoWin]
  recommend_geo_window_kernel<<<(unsigned)((B + kRtThreads - 1) / kRtThreads), kRtThreads, 0, s>>>(
      centre_xyz, threshold, B, cell_deg, (int)num_lat, (int)num_lon, H, win, bucket, err);
  YR_CHECK_LAUNCH();
  recommend_subset_plan_kernel<<<1, kRsPlanThreads, 0, s>>>(bucket, (int)B, H, TU, cursor, rows_at, blocks_at, order,
                                                            err);
  YR_CHECK_LAUNCH();
  int rc;
#define YR_GEO_LAUNCH(T, TU_, BIAS)                                                                                       \
  geo_launch<T, TU_, BIAS>(U, nU, V, d, user_ids, B, cell_keys, cell_ptr, num_cells, cell_items, item_xyz, (int)num_lon, \
                           centre_xyz, threshold, win, H, rows_at, blocks_at, order, seen_ptr, seen_idx, K, S, partial,  \
                           out_ids, out_scores, err, item_bias, s)
#define YR_GEO_TU(T, BIAS)                                                                                                \
  (TU == 16 ? YR_GEO_LAUNCH(T, 16, BIAS) : TU == 8 ? YR_GEO_LAUNCH(T, 8, BIAS) : YR_GEO_LAUNCH(T, 4, BIAS))
  if (dtype == YR_DTYPE_F32)
    rc = item_bias ? YR_GEO_TU(float, true) : YR_GEO_TU(float, false);
  else
    rc = item_bias ? YR_GEO_TU(__nv_bfloat16, true) : YR_GEO_TU(__nv_bfloat16, false);
#undef YR_GEO_TU
#undef YR_GEO_LAUNCH
  if (rc || S == 1) return rc;
  return merge_launch(partial, S, B, K, out_ids, out_scores, s);
}
