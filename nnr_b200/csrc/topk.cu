// Streaming top-k merge of a news-recommendation candidate pool (scoring.CorpusScorer.recommend).
//
// The pool is scored in tiles of T candidates; after each [B, T] score tile this kernel folds the tile into a running
// per-user best list of k (score, pool position) entries.  One CTA per user row:
//   1. the row's running list (k keys) and its exclusion list (history ids) go to shared memory;
//   2. every tile entry whose key does not beat the smallest key of the list, or whose news id is excluded, is dropped;
//      the survivors are appended behind the list (shared-memory atomic counter);
//   3. list + survivors (padded with key 0 to a power of two) are bitonic-sorted in descending key order and the first
//      k keys are written back.
// Keys are unique (positions are), so the order the survivors are appended in does not change the result: the merge is
// deterministic.  No host synchronisation, no allocation: capturable in a CUDA graph.
#include "common.cuh"
#include "../../include/nnr_b200.h"

#define TOPK_THREADS 256

// Order-preserving 64-bit key, larger = ranked first.  Bits 63..32: the score's bits mapped so that unsigned order is
// numeric order, with -0.0 folded onto +0.0 (a stable sort treats them as equal) and every NaN mapped to 0, below
// -inf (0x007FFFFF): a NaN is never ranked above a number.  Bits 31..0: 0xFFFFFFFF - position, so that of two equal
// scores the smaller pool position ranks first.  Key 0 is the fill entry (score -inf, position -1); positions are
// < 2^31 - 1, so no real entry, NaN or not, has key 0.
__device__ __forceinline__ uint64_t topk_key(float s, int64_t pos) {
  const uint32_t u = __float_as_uint(s);
  uint32_t hi;
  if (s != s) hi = 0u;
  else if (s == 0.0f) hi = 0x80000000u;
  else hi = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((uint64_t)hi << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)pos);
}

__device__ __forceinline__ void topk_unkey(uint64_t key, float* s, int64_t* pos) {
  if (key == 0ull) {
    *s = -INFINITY;
    *pos = -1;
    return;
  }
  const uint32_t hi = (uint32_t)(key >> 32);
  *pos = (int64_t)(0xFFFFFFFFu - (uint32_t)key);
  if (hi == 0u) *s = __uint_as_float(0x7FC00000u);
  else *s = __uint_as_float((hi & 0x80000000u) ? (hi & 0x7FFFFFFFu) : ~hi);
}

// shared memory: key[cap] (cap = next power of two >= k + T), then the row's exclusion ids [ldx]
__global__ void __launch_bounds__(TOPK_THREADS) topk_merge_kernel(
    const float* __restrict__ scores, int64_t lds, int T, int64_t pos0, const int64_t* __restrict__ tile_ids,
    const int64_t* __restrict__ excl, const int32_t* __restrict__ excl_len, int ldx, int k, int cap, int init,
    float* __restrict__ best_score, int64_t* __restrict__ best_pos) {
  extern __shared__ uint64_t topk_smem[];
  uint64_t* key = topk_smem;
  int64_t* s_excl = reinterpret_cast<int64_t*>(topk_smem + cap);
  __shared__ unsigned long long s_thr;
  __shared__ int s_m;
  const int b = blockIdx.x, tid = threadIdx.x;
  float* bs = best_score + (size_t)b * k;
  int64_t* bp = best_pos + (size_t)b * k;
  const int nx = excl ? min(max(excl_len[b], 0), ldx) : 0;
  if (tid == 0) {
    s_thr = ~0ull;
    s_m = 0;
  }
  __syncthreads();
  for (int i = tid; i < nx; i += blockDim.x) s_excl[i] = excl[(size_t)b * ldx + i];
  for (int i = tid; i < k; i += blockDim.x) {
    const uint64_t kk = (init || bp[i] < 0) ? 0ull : topk_key(bs[i], bp[i]);
    key[i] = kk;
    atomicMin(&s_thr, (unsigned long long)kk);
  }
  __syncthreads();
  const uint64_t thr = s_thr;                                  // the k-th best so far: only keys above it can enter
  const float* row = scores + (size_t)b * lds;
  for (int j = tid; j < T; j += blockDim.x) {
    const uint64_t kk = topk_key(row[j], pos0 + j);
    if (kk <= thr) continue;
    if (nx > 0) {
      const int64_t id = tile_ids[j];
      bool hit = false;
      for (int h = 0; h < nx && !hit; ++h) hit = s_excl[h] == id;
      if (hit) continue;
    }
    key[k + atomicAdd(&s_m, 1)] = kk;
  }
  __syncthreads();
  const int m = s_m;
  if (m == 0 && !init) return;                                  // nothing beats the k-th best: the list stands
  int n = 1;
  while (n < k + m) n <<= 1;
  for (int i = k + m + tid; i < n; i += blockDim.x) key[i] = 0ull;
  __syncthreads();
  // bitonic sort of key[0, n), descending
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (n >> 1); i += blockDim.x) {
        const int lo = 2 * stride * (i / stride) + (i % stride);
        const int hi = lo + stride;
        const bool desc = (lo & size) == 0;
        const uint64_t a = key[lo], c = key[hi];
        if ((a < c) == desc) {
          key[lo] = c;
          key[hi] = a;
        }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < k; i += blockDim.x) topk_unkey(key[i], &bs[i], &bp[i]);
}

extern "C" int nnr_topk_merge(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                              const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init,
                              float* best_score, int64_t* best_pos, void* stream) {
  NNR_REQUIRE(k >= 1 && k <= NNR_TOPK_MAX_K, NNR_ERR_ARG, "nnr_topk_merge: k must be in [1, %d], got %d", NNR_TOPK_MAX_K, k);
  NNR_REQUIRE(T >= 1 && T <= NNR_TOPK_MAX_TILE, NNR_ERR_ARG, "nnr_topk_merge: T must be in [1, %d], got %d",
              NNR_TOPK_MAX_TILE, T);
  NNR_REQUIRE(B >= 0, NNR_ERR_ARG, "nnr_topk_merge: B must be >= 0, got %d", B);
  NNR_REQUIRE(scores && best_score && best_pos, NNR_ERR_ARG, "nnr_topk_merge: scores, best_score and best_pos must not be NULL");
  NNR_REQUIRE(lds >= T, NNR_ERR_ARG, "nnr_topk_merge: lds (%lld) < T (%d)", (long long)lds, T);
  NNR_REQUIRE(pos0 >= 0 && pos0 + T <= (int64_t)INT32_MAX - 1, NNR_ERR_ARG,
              "nnr_topk_merge: pool positions [%lld, %lld) outside [0, 2^31 - 1)", (long long)pos0, (long long)(pos0 + T));
  if (exclude) {
    NNR_REQUIRE(tile_ids && exclude_len, NNR_ERR_ARG, "nnr_topk_merge: an exclusion list needs tile_ids and exclude_len");
    NNR_REQUIRE(ldx >= 0 && ldx <= NNR_TOPK_MAX_EXCLUDE, NNR_ERR_ARG, "nnr_topk_merge: ldx must be in [0, %d], got %d",
                NNR_TOPK_MAX_EXCLUDE, ldx);
  }
  if (B == 0) return 0;
  int cap = 1;
  while (cap < k + T) cap <<= 1;
  const int nx = exclude ? ldx : 0;
  const size_t smem = (size_t)cap * sizeof(uint64_t) + (size_t)nx * sizeof(int64_t);
  if (smem > 48 * 1024) {
    static bool attr_set[64] = {};
    int dev = 0;
    NNR_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !attr_set[dev]) {
      const int most = (8192 + NNR_TOPK_MAX_EXCLUDE) * 8;     // cap <= 8192 for k + T <= 5120
      NNR_CUDA(cudaFuncSetAttribute((const void*)topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, most));
      if (dev < 64) attr_set[dev] = true;
    }
  }
  topk_merge_kernel<<<B, TOPK_THREADS, smem, (cudaStream_t)stream>>>(scores, lds, T, pos0, tile_ids, exclude, exclude_len,
                                                                    nx, k, cap, init, best_score, best_pos);
  NNR_LAUNCH_CHECK("topk_merge_kernel");
  return 0;
}
