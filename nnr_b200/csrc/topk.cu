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
//
// The capped variant (nnr_topk_merge_capped) keeps at most `group_cap` entries per group (news category): every key
// carries its group through the sort, and one warp then walks the sorted keys in order, keeping an entry while fewer than
// group_cap entries of its group were kept before it, until k are kept.  Why the k-entry state stays exact: DESIGN.md §4.
//
// The list variants (nnr_topk_merge_lists[_capped], LISTS) merge a [B, T] block of entries that carry their own pool
// position pos[b, j] (and group grp[b, j]) instead of pos0 + j and id_group[tile_ids[j]]: the per-rank best lists of a
// data-parallel recommend() call, folded into one.  A negative position is an empty (fill) slot and is dropped first.
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

// shared memory: key[cap] (cap = next power of two >= k + T), then the row's exclusion ids [ldx]; CAPPED adds each key's
// group grp[cap] and the per-group counters cnt[num_groups].  LISTS reads positions from list_pos [B, ldp] and groups from
// list_grp [B, ldg]; it has no exclusion list.
template <bool CAPPED, bool LISTS>
__global__ void __launch_bounds__(TOPK_THREADS) topk_merge_kernel(
    const float* __restrict__ scores, int64_t lds, int T, int64_t pos0, const int64_t* __restrict__ tile_ids,
    const int64_t* __restrict__ excl, const int32_t* __restrict__ excl_len, int ldx, int k, int cap, int init,
    float* __restrict__ best_score, int64_t* __restrict__ best_pos, const int32_t* __restrict__ id_group, int num_groups,
    int group_cap, int32_t* __restrict__ best_group, const int64_t* __restrict__ list_pos, int64_t ldp,
    const int32_t* __restrict__ list_grp, int64_t ldg) {
  extern __shared__ uint64_t topk_smem[];
  uint64_t* key = topk_smem;
  int64_t* s_excl = reinterpret_cast<int64_t*>(topk_smem + cap);
  int32_t* grp = reinterpret_cast<int32_t*>(s_excl + ldx);
  int32_t* cnt = grp + cap;
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
    if constexpr (CAPPED) grp[i] = kk ? best_group[(size_t)b * k + i] : -1;
    atomicMin(&s_thr, (unsigned long long)kk);
  }
  if constexpr (CAPPED)
    for (int g = tid; g < num_groups; g += blockDim.x) cnt[g] = 0;
  __syncthreads();
  const uint64_t thr = s_thr;                                  // the k-th best so far: only keys above it can enter
  const float* row = scores + (size_t)b * lds;
  for (int j = tid; j < T; j += blockDim.x) {
    int64_t p = pos0 + j;
    if constexpr (LISTS) {
      p = list_pos[(size_t)b * ldp + j];
      if (p < 0) continue;                                      // an empty slot of the list, not a -inf entry
    }
    const uint64_t kk = topk_key(row[j], p);
    if (kk <= thr) continue;
    if (!LISTS && nx > 0) {
      const int64_t id = tile_ids[j];
      bool hit = false;
      for (int h = 0; h < nx && !hit; ++h) hit = s_excl[h] == id;
      if (hit) continue;
    }
    const int slot = k + atomicAdd(&s_m, 1);
    key[slot] = kk;
    if constexpr (CAPPED) {
      if constexpr (LISTS) grp[slot] = list_grp[(size_t)b * ldg + j];
      else grp[slot] = id_group[tile_ids[j]];
    }
  }
  __syncthreads();
  const int m = s_m;
  if (m == 0 && !init) return;                                  // nothing beats the k-th best: the list stands
  int n = 1;
  while (n < k + m) n <<= 1;
  for (int i = k + m + tid; i < n; i += blockDim.x) {
    key[i] = 0ull;
    if constexpr (CAPPED) grp[i] = -1;
  }
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
          if constexpr (CAPPED) {
            const int32_t t = grp[lo];
            grp[lo] = grp[hi];
            grp[hi] = t;
          }
        }
      }
      __syncthreads();
    }
  }
  if constexpr (CAPPED) {
    // the cap: warp 0 walks the sorted keys 32 at a time.  A lane's rank among the chunk's lanes of its group comes from
    // __match_any_sync, the groups' counts of earlier chunks from cnt[]; kept entries are compacted in place to the front
    // (an entry moves to an index <= its own, never to one a later chunk still has to read).  Key 0 (fill, padding) ends
    // the walk, as does the k-th kept entry.  A group outside [0, num_groups) is never kept.
    __shared__ int s_kept;
    if (tid < 32) {
      const unsigned below = (1u << tid) - 1u;
      int kept = 0;
      for (int base = 0; base < n && kept < k; base += 32) {
        const int i = base + tid;
        const uint64_t kk = i < n ? key[i] : 0ull;
        const int g = i < n ? grp[i] : -1;
        const bool real = kk != 0ull && (unsigned)g < (unsigned)num_groups;
        const unsigned same = __match_any_sync(0xFFFFFFFFu, real ? g : -1);
        const int before = real ? cnt[g] : 0;
        const bool keep = real && before + __popc(same & below) < group_cap;
        const unsigned kmask = __ballot_sync(0xFFFFFFFFu, keep);
        const bool last = __ballot_sync(0xFFFFFFFFu, kk == 0ull) != 0u;
        __syncwarp();
        if (real && (same & below) == 0u) cnt[g] = before + __popc(same);
        if (keep) {
          const int o = kept + __popc(kmask & below);
          key[o] = kk;
          grp[o] = g;
        }
        kept += __popc(kmask);
        __syncwarp();
        if (last) break;
      }
      if (tid == 0) s_kept = min(kept, k);
    }
    __syncthreads();
    const int kept = s_kept;
    int32_t* bg = best_group + (size_t)b * k;
    for (int i = tid; i < k; i += blockDim.x) {
      topk_unkey(i < kept ? key[i] : 0ull, &bs[i], &bp[i]);
      bg[i] = i < kept ? grp[i] : -1;
    }
  } else {
    for (int i = tid; i < k; i += blockDim.x) topk_unkey(key[i], &bs[i], &bp[i]);
  }
}

// the checks nnr_topk_merge and nnr_topk_merge_capped share; `who` names the entry point in the message
static int topk_check(const char* who, const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                      const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, const float* best_score,
                      const int64_t* best_pos) {
  NNR_REQUIRE(k >= 1 && k <= NNR_TOPK_MAX_K, NNR_ERR_ARG, "%s: k must be in [1, %d], got %d", who, NNR_TOPK_MAX_K, k);
  NNR_REQUIRE(T >= 1 && T <= NNR_TOPK_MAX_TILE, NNR_ERR_ARG, "%s: T must be in [1, %d], got %d", who, NNR_TOPK_MAX_TILE, T);
  NNR_REQUIRE(B >= 0, NNR_ERR_ARG, "%s: B must be >= 0, got %d", who, B);
  NNR_REQUIRE(scores && best_score && best_pos, NNR_ERR_ARG, "%s: scores, best_score and best_pos must not be NULL", who);
  NNR_REQUIRE(lds >= T, NNR_ERR_ARG, "%s: lds (%lld) < T (%d)", who, (long long)lds, T);
  NNR_REQUIRE(pos0 >= 0 && pos0 + T <= (int64_t)INT32_MAX - 1, NNR_ERR_ARG,
              "%s: pool positions [%lld, %lld) outside [0, 2^31 - 1)", who, (long long)pos0, (long long)(pos0 + T));
  if (exclude) {
    NNR_REQUIRE(tile_ids && exclude_len, NNR_ERR_ARG, "%s: an exclusion list needs tile_ids and exclude_len", who);
    NNR_REQUIRE(ldx >= 0 && ldx <= NNR_TOPK_MAX_EXCLUDE, NNR_ERR_ARG, "%s: ldx must be in [0, %d], got %d", who,
                NNR_TOPK_MAX_EXCLUDE, ldx);
  }
  return 0;
}

template <bool CAPPED, bool LISTS>
static int topk_launch(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                       const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init, float* best_score,
                       int64_t* best_pos, const int32_t* id_group, int num_groups, int group_cap, int32_t* best_group,
                       const int64_t* list_pos, int64_t ldp, const int32_t* list_grp, int64_t ldg, void* stream) {
  if (B == 0) return 0;
  int cap = 1;
  while (cap < k + T) cap <<= 1;
  const int nx = exclude ? ldx : 0;
  size_t smem = (size_t)cap * sizeof(uint64_t) + (size_t)nx * sizeof(int64_t);
  if (CAPPED) smem += (size_t)cap * sizeof(int32_t) + (size_t)num_groups * sizeof(int32_t);
  if (smem > 48 * 1024) {
    static bool attr_set[64] = {};                           // one per instantiation
    int dev = 0;
    NNR_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !attr_set[dev]) {
      // cap <= 8192 for k + T <= 5120
      const int most = (8192 + NNR_TOPK_MAX_EXCLUDE) * 8 + (CAPPED ? (8192 + NNR_TOPK_MAX_GROUPS) * 4 : 0);
      NNR_CUDA(cudaFuncSetAttribute((const void*)topk_merge_kernel<CAPPED, LISTS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    most));
      if (dev < 64) attr_set[dev] = true;
    }
  }
  topk_merge_kernel<CAPPED, LISTS><<<B, TOPK_THREADS, smem, (cudaStream_t)stream>>>(
      scores, lds, T, pos0, tile_ids, exclude, exclude_len, nx, k, cap, init, best_score, best_pos, id_group, num_groups,
      group_cap, best_group, list_pos, ldp, list_grp, ldg);
  NNR_LAUNCH_CHECK(LISTS ? (CAPPED ? "topk_merge_kernel<capped, lists>" : "topk_merge_kernel<lists>")
                         : (CAPPED ? "topk_merge_kernel<capped>" : "topk_merge_kernel"));
  return 0;
}

extern "C" int nnr_topk_merge(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                              const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init,
                              float* best_score, int64_t* best_pos, void* stream) {
  const int rc = topk_check("nnr_topk_merge", scores, lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx, k, best_score,
                            best_pos);
  if (rc) return rc;
  return topk_launch<false, false>(scores, lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx, k, init, best_score,
                                   best_pos, nullptr, 0, 0, nullptr, nullptr, 0, nullptr, 0, stream);
}

extern "C" int nnr_topk_merge_capped(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                                     const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init,
                                     const int32_t* id_group, int num_groups, int cap, float* best_score,
                                     int64_t* best_pos, int32_t* best_group, void* stream) {
  const char* who = "nnr_topk_merge_capped";
  const int rc = topk_check(who, scores, lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx, k, best_score, best_pos);
  if (rc) return rc;
  NNR_REQUIRE(cap >= 1, NNR_ERR_ARG, "%s: cap must be >= 1, got %d", who, cap);
  NNR_REQUIRE(num_groups >= 1 && num_groups <= NNR_TOPK_MAX_GROUPS, NNR_ERR_ARG, "%s: num_groups must be in [1, %d], got %d",
              who, NNR_TOPK_MAX_GROUPS, num_groups);
  NNR_REQUIRE(id_group && best_group && tile_ids, NNR_ERR_ARG, "%s: id_group, best_group and tile_ids must not be NULL", who);
  return topk_launch<true, false>(scores, lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx, k, init, best_score,
                                  best_pos, id_group, num_groups, cap, best_group, nullptr, 0, nullptr, 0, stream);
}

// the checks nnr_topk_merge_lists and nnr_topk_merge_lists_capped share (those of topk_check for a tile at position 0
// without exclusion list, plus pos and ldp)
static int topk_lists_check(const char* who, const float* scores, int64_t lds, int B, int T, const int64_t* pos, int64_t ldp,
                            int k, const float* best_score, const int64_t* best_pos) {
  const int rc = topk_check(who, scores, lds, B, T, 0, nullptr, nullptr, nullptr, 0, k, best_score, best_pos);
  if (rc) return rc;
  NNR_REQUIRE(pos, NNR_ERR_ARG, "%s: pos must not be NULL", who);
  NNR_REQUIRE(ldp >= T, NNR_ERR_ARG, "%s: ldp (%lld) < T (%d)", who, (long long)ldp, T);
  return 0;
}

extern "C" int nnr_topk_merge_lists(const float* scores, int64_t lds, int B, int T, const int64_t* pos, int64_t ldp, int k,
                                    int init, float* best_score, int64_t* best_pos, void* stream) {
  const int rc = topk_lists_check("nnr_topk_merge_lists", scores, lds, B, T, pos, ldp, k, best_score, best_pos);
  if (rc) return rc;
  return topk_launch<false, true>(scores, lds, B, T, 0, nullptr, nullptr, nullptr, 0, k, init, best_score, best_pos, nullptr,
                                  0, 0, nullptr, pos, ldp, nullptr, 0, stream);
}

extern "C" int nnr_topk_merge_lists_capped(const float* scores, int64_t lds, int B, int T, const int64_t* pos, int64_t ldp,
                                           const int32_t* grp, int64_t ldg, int num_groups, int cap, int k, int init,
                                           float* best_score, int64_t* best_pos, int32_t* best_group, void* stream) {
  const char* who = "nnr_topk_merge_lists_capped";
  const int rc = topk_lists_check(who, scores, lds, B, T, pos, ldp, k, best_score, best_pos);
  if (rc) return rc;
  NNR_REQUIRE(grp && best_group, NNR_ERR_ARG, "%s: grp and best_group must not be NULL", who);
  NNR_REQUIRE(ldg >= T, NNR_ERR_ARG, "%s: ldg (%lld) < T (%d)", who, (long long)ldg, T);
  NNR_REQUIRE(cap >= 1, NNR_ERR_ARG, "%s: cap must be >= 1, got %d", who, cap);
  NNR_REQUIRE(num_groups >= 1 && num_groups <= NNR_TOPK_MAX_GROUPS, NNR_ERR_ARG, "%s: num_groups must be in [1, %d], got %d",
              who, NNR_TOPK_MAX_GROUPS, num_groups);
  return topk_launch<true, true>(scores, lds, B, T, 0, nullptr, nullptr, nullptr, 0, k, init, best_score, best_pos, nullptr,
                                 num_groups, cap, best_group, pos, ldp, grp, ldg, stream);
}
