// Factored cluster tail of SUE for top-k recommendation (nnr_cluster_tail_scores; scoring.CorpusScorer.recommend(exact=False)).
//
// The exact tail (cluster_intra_fwd_kernel, the clusterFeatureAffine GEMM with EPI_BIAS_RELU_RES, attn_pool mode 1, rowdot)
// materialises C1 D-wide cluster features per (user, candidate) pair and multiplies each by the D x D affine.  The
// intra-cluster weights of a non-empty cluster sum to 1 and an empty cluster's feature is 0, so the affine commutes with the
// weighted sum:  W intra_c + b = sum_{h in c} alpha_h (W g_h) + b.  With Wg = g W^T computed once per user, a pair needs
// only two scalars per cluster, f_c . qk2 and f_c . cand, where f_c = relu(sum_{h in c} alpha_h Wg_h + b) + intra_c.
//
// One CTA per (user, slice of TC = 2 * NT candidates); thread tid owns candidates tid and tid + NT of the slice.
//   1. the user's H slots are counting-sorted by cluster (stable), as in cluster_intra_fwd_kernel;
//   2. intra-cluster logits s[e][t] = Kp[perm[e]] . Qp[t], over chunks of TAIL_KC features of Au staged in shared memory;
//   3. per candidate, a max-shifted softmax over each cluster's slots turns scale * s into alpha, in place;
//   4. per step of DD features: for each non-empty cluster, y = sum alpha Wg and i = sum alpha g over the cluster's slots
//      (registers: DD features x 2 candidates), then f = relu(y + b) + i is dotted with the candidate's qk2 and cand rows and
//      the two partial dots are added to per-(cluster, candidate) accumulators in shared memory.  Every empty cluster has
//      f = relu(b); its two dots are accumulated once per candidate;
//   5. per candidate: beta = softmax over clusters of scale * (f_c . qk2), -1e9 for masked clusters (attn_pool's rule),
//      score = sum_c beta_c (f_c . cand).
// Every sum runs in a fixed order and every accumulator has one owner thread: the result is deterministic.  After phase 2
// a thread reads only its own candidates' columns, so phases 3-5 need no barrier.
//
// nnr_cluster_tail_scores_packed (evaluate(exact=False)) runs the same phases (tail_cta) on per-user candidate lists
// stored back to back, one CTA per (user, slice of TAIL_PC candidates).  A MIND list has ~37 candidates, too few to hide
// the latency of phase 4's loads with one warp, so W warps split the slots, the clusters and the feature steps, and the
// partial dots of a round of W steps are added in step order: the scores equal the pool kernel's bit for bit.
//
// nnr_cluster_tail_explain_packed (CorpusScorer.explain(exact=False)) is the packed kernel with EX = true: phase 3 also
// stores each slot's alpha at its history position, phase 5 each cluster's beta and beta * (f . cand).  The score is
// summed by the same instructions, so it equals the packed kernel's bit for bit.
#include "common.cuh"
#include "../../include/nnr_b200.h"

#define TAIL_MAXH 256          // the limits of cluster_intra_fwd_kernel (sue.cu: CI_MAXH, CI_MAXC)
#define TAIL_MAXC 72
#define TAIL_KC 16             // Au features per staged chunk of the logits
#define TAIL_TT 2              // candidates per thread
#define TAIL_PC 64             // candidates per CTA of the packed kernel: MIND lists are ~37 long

__device__ __forceinline__ void tail_load(float* dst, const float* src, int n4) {
#pragma unroll
  for (int i = 0; i < n4; ++i) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    dst[4 * i] = v.x; dst[4 * i + 1] = v.y; dst[4 * i + 2] = v.z; dst[4 * i + 3] = v.w;
  }
}

// the dots of relu(b) (every empty cluster's feature) with features [d0, d0 + DD) of the candidates' qk2 and cand rows,
// accumulated into eq / ec; candidate j of the thread is column col + j * CS of the CTA's slice
template <int CS, int DD>
__device__ __forceinline__ void tail_empty_dots(int d0, const float* __restrict__ qk2, const float* __restrict__ cand,
                                                const float* __restrict__ bias, int D, int T, int t0, int col,
                                                float (&q)[TAIL_TT][DD], float (&x)[TAIL_TT][DD], float (&bv)[DD],
                                                float* eq, float* ec) {
#pragma unroll
  for (int j = 0; j < TAIL_TT; ++j) {
    const int t = t0 + col + j * CS;
    if (t < T) {
      tail_load(q[j], qk2 + (size_t)t * D + d0, DD / 4);
      tail_load(x[j], cand + (size_t)t * D + d0, DD / 4);
    } else {
#pragma unroll
      for (int k = 0; k < DD; ++k) q[j][k] = x[j][k] = 0.f;
    }
  }
  tail_load(bv, bias + d0, DD / 4);
#pragma unroll
  for (int j = 0; j < TAIL_TT; ++j)
#pragma unroll
    for (int k = 0; k < DD; ++k) {
      const float f = fmaxf(bv[k], 0.f);
      eq[j] = fmaf(f, q[j][k], eq[j]);
      ec[j] = fmaf(f, x[j][k], ec[j]);
    }
}

// phase 4 for features [d0, d0 + DD) of the thread's candidates.  ADD: add each non-empty cluster's two partial dots to
// acc (the running per-(cluster, candidate) sums); otherwise store them there (one step's partials, summed in step order
// by the caller)
template <int CS, int DD, bool ADD>
__device__ __forceinline__ void tail_step(int d0, const float* __restrict__ gb, const float* __restrict__ wb,
                                          const float* __restrict__ qk2, const float* __restrict__ cand,
                                          const float* __restrict__ bias, const float* s_al, float* acc,
                                          const int* s_perm, const int* s_start, int C1, int D, int T, int t0, int col,
                                          float* eq, float* ec) {
  constexpr int TC = CS * TAIL_TT;
  float q[TAIL_TT][DD], x[TAIL_TT][DD], bv[DD];
  tail_empty_dots<CS, DD>(d0, qk2, cand, bias, D, T, t0, col, q, x, bv, eq, ec);
  for (int c = 0; c < C1; ++c) {
    const int lo = s_start[c], hi = s_start[c + 1];
    if (lo == hi) continue;
    float y[TAIL_TT][DD], z[TAIL_TT][DD];
#pragma unroll
    for (int j = 0; j < TAIL_TT; ++j)
#pragma unroll
      for (int k = 0; k < DD; ++k) y[j][k] = z[j][k] = 0.f;
#pragma unroll 2
    for (int e = lo; e < hi; ++e) {
      const int h = s_perm[e];
      float wv[DD], gv[DD], a[TAIL_TT];
      tail_load(wv, wb + (size_t)h * D + d0, DD / 4);
      tail_load(gv, gb + (size_t)h * D + d0, DD / 4);
#pragma unroll
      for (int j = 0; j < TAIL_TT; ++j) a[j] = s_al[e * TC + col + j * CS];
#pragma unroll
      for (int j = 0; j < TAIL_TT; ++j)
#pragma unroll
        for (int k = 0; k < DD; ++k) {
          y[j][k] = fmaf(a[j], wv[k], y[j][k]);
          z[j][k] = fmaf(a[j], gv[k], z[j][k]);
        }
    }
#pragma unroll
    for (int j = 0; j < TAIL_TT; ++j) {
      float pq = 0.f, pc = 0.f;
#pragma unroll
      for (int k = 0; k < DD; ++k) {
        const float f = fmaxf(y[j][k] + bv[k], 0.f) + z[j][k];
        pq = fmaf(f, q[j][k], pq);
        pc = fmaf(f, x[j][k], pc);
      }
      float* aq = acc + c * TC + col + j * CS;
      float* ac = acc + (C1 + c) * TC + col + j * CS;
      if (ADD) { *aq += pq; *ac += pc; } else { *aq = pq; *ac = pc; }
    }
  }
}

// phases 1-5 of one CTA: candidates [t0, min(t0 + TC, T)) of user b, whose candidate rows start at Qp, qk2 and cand;
// candidate t's score goes to srow[t].  Shared by the pool and the packed kernel, so that both sum in the same order.
// NT = CS * W threads: thread tid owns the candidate columns col + j * CS (col = tid % CS, j < TAIL_TT) of the slice for
// the slots e, the clusters c and the feature steps s with e, c, s = grp (mod W) (grp = tid / CS).  W = 1 (the pool
// kernel): one thread does all of a candidate's work, and phases 3-5 need no barrier.  W > 1: the W groups take turns
// over the feature steps; the W partial dots of a round are stored in s_part and added to the running sums in step
// order, so every sum runs in the order of W = 1.
// EX: candidate t's alpha goes to ex.alpha[t * H + h] (h: the slot's history position), its beta and beta * (f . cand)
// to ex.beta[t * C1 + c] and ex.contrib[t * C1 + c].
// One struct parameter rather than three pointers: with three, even unused, ptxas allocates the EX = false kernels'
// registers differently.
struct TailEx { float* alpha; float* beta; float* contrib; };

template <int CS, int W, bool EX = false>
__device__ __forceinline__ void tail_cta(const float* __restrict__ Kp, const float* __restrict__ g,
                                         const float* __restrict__ Wg, const int64_t* __restrict__ idx,
                                         const uint8_t* __restrict__ cmask, const float* __restrict__ Qp,
                                         const float* __restrict__ qk2, const float* __restrict__ cand,
                                         const float* __restrict__ bias, int b, int H, int Au, int D, int C1, int T, int t0,
                                         float scale, float* __restrict__ srow, TailEx ex = {}) {
  constexpr int NT = CS * W, TC = CS * TAIL_TT;
  extern __shared__ __align__(16) float sm[];
  float* s_al = sm;                                   // [H][TC]: logits, then alpha (slots in cluster order)
  float* s_acc = sm + (size_t)H * TC;                 // [2][C1][TC]: f . qk2, f . cand of the non-empty clusters
  float* s_q = s_acc;                                 // phase 2 only: Qp chunk [TAIL_KC][TC + 1] and Kp chunk [H][TAIL_KC]
  float* s_k = s_acc + TAIL_KC * (TC + 1);
  __shared__ int s_idx[TAIL_MAXH];
  __shared__ int s_perm[TAIL_MAXH];
  __shared__ int s_start[TAIL_MAXC + 1];
  const int tid = threadIdx.x, col = W == 1 ? tid : tid % CS, grp = W == 1 ? 0 : tid / CS;

  // 1. stable counting sort of the slots by cluster
  for (int h = tid; h < H; h += NT) { const int c = (int)idx[(size_t)b * H + h]; s_idx[h] = min(max(c, 0), C1 - 1); }
  __syncthreads();
  for (int c = tid; c <= C1; c += NT) {
    int pos = 0;
    for (int h = 0; h < H; ++h) pos += (s_idx[h] < c);
    s_start[c] = pos;
  }
  __syncthreads();
  for (int h = tid; h < H; h += NT) {
    const int c = s_idx[h];
    int pos = s_start[c];
    for (int j = 0; j < h; ++j) pos += (s_idx[j] == c);
    s_perm[pos] = h;
  }
  __syncthreads();

  // 2. logits, accumulated over the chunks of Au in order
  const float* Kb = Kp + (size_t)b * H * Au;
  for (int a0 = 0; a0 < Au; a0 += TAIL_KC) {
    for (int i = tid; i < TC * TAIL_KC; i += NT) {
      const int t = i / TAIL_KC, a = i % TAIL_KC;
      s_q[a * (TC + 1) + t] = (t0 + t < T && a0 + a < Au) ? __ldg(Qp + (size_t)(t0 + t) * Au + a0 + a) : 0.f;
    }
    for (int i = tid; i < H * TAIL_KC; i += NT) {
      const int e = i / TAIL_KC, a = i % TAIL_KC;
      s_k[i] = (a0 + a < Au) ? __ldg(Kb + (size_t)s_perm[e] * Au + a0 + a) : 0.f;
    }
    __syncthreads();
    float q[TAIL_TT][TAIL_KC];
#pragma unroll
    for (int j = 0; j < TAIL_TT; ++j)
#pragma unroll
      for (int a = 0; a < TAIL_KC; ++a) q[j][a] = s_q[a * (TC + 1) + col + j * CS];
    for (int e = grp; e < H; e += W) {
      const float4* kr = reinterpret_cast<const float4*>(s_k + e * TAIL_KC);
      float v[TAIL_TT] = {};
#pragma unroll
      for (int a4 = 0; a4 < TAIL_KC / 4; ++a4) {
        const float4 k4 = kr[a4];
#pragma unroll
        for (int j = 0; j < TAIL_TT; ++j) {
          v[j] = fmaf(k4.x, q[j][4 * a4], v[j]);
          v[j] = fmaf(k4.y, q[j][4 * a4 + 1], v[j]);
          v[j] = fmaf(k4.z, q[j][4 * a4 + 2], v[j]);
          v[j] = fmaf(k4.w, q[j][4 * a4 + 3], v[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < TAIL_TT; ++j) {
        float* p = s_al + e * TC + col + j * CS;
        *p = (a0 == 0) ? v[j] : *p + v[j];
      }
    }
    __syncthreads();                                  // the next chunk (or phase 4's accumulators) reuses the staging
  }

  // 3. softmax within each cluster (max-shifted, like torch_scatter.scatter_softmax)
#pragma unroll
  for (int j = 0; j < TAIL_TT; ++j) {
    float* col_j = s_al + col + j * CS;
    if (W == 1)
      for (int e = 0; e < H; ++e) col_j[e * TC] *= scale;
    else
      for (int c = grp; c < C1; c += W)
        for (int e = s_start[c]; e < s_start[c + 1]; ++e) col_j[e * TC] *= scale;
    for (int c = grp; c < C1; c += W) {
      const int lo = s_start[c], hi = s_start[c + 1];
      if (lo == hi) continue;
      float m = -INFINITY;
      for (int e = lo; e < hi; ++e) m = fmaxf(m, col_j[e * TC]);
      float sum = 0.f;
      for (int e = lo; e < hi; ++e) sum += expf(col_j[e * TC] - m);
      for (int e = lo; e < hi; ++e) {
        col_j[e * TC] = expf(col_j[e * TC] - m) / sum;
        if constexpr (EX)
          if (t0 + col + j * CS < T) ex.alpha[(size_t)(t0 + col + j * CS) * H + s_perm[e]] = col_j[e * TC];
      }
    }
    for (int c = grp; c < C1; c += W) s_acc[c * TC + col + j * CS] = s_acc[(C1 + c) * TC + col + j * CS] = 0.f;
  }

  // 4. the two dots of every cluster feature, DD features at a time (D % 4 == 0)
  const float* gb = g + (size_t)b * H * D;
  const float* wb = Wg + (size_t)b * H * D;
  float eq[TAIL_TT] = {}, ec[TAIL_TT] = {};
  if (W == 1) {
    int d0 = 0;
    for (; d0 + 8 <= D; d0 += 8)
      tail_step<CS, 8, true>(d0, gb, wb, qk2, cand, bias, s_al, s_acc, s_perm, s_start, C1, D, T, t0, col, eq, ec);
    if (d0 < D) tail_step<CS, 4, true>(d0, gb, wb, qk2, cand, bias, s_al, s_acc, s_perm, s_start, C1, D, T, t0, col, eq, ec);
  } else {
    float* s_part = s_acc + (size_t)2 * C1 * TC;      // [W][2][C1][TC]: one round's partial dots (past the staging)
    __syncthreads();                                  // alpha and the zeroed sums of the other groups
    const int steps = (D + 7) / 8;
    for (int r0 = 0; r0 < steps; r0 += W) {
      const int d0 = 8 * (r0 + grp);
      float* part = s_part + (size_t)grp * 2 * C1 * TC;
      float dq[TAIL_TT] = {}, dc[TAIL_TT] = {};       // the empty-cluster dots are summed by group 0 alone, below
      if (d0 + 8 <= D)
        tail_step<CS, 8, false>(d0, gb, wb, qk2, cand, bias, s_al, part, s_perm, s_start, C1, D, T, t0, col, dq, dc);
      else if (d0 < D)
        tail_step<CS, 4, false>(d0, gb, wb, qk2, cand, bias, s_al, part, s_perm, s_start, C1, D, T, t0, col, dq, dc);
      __syncthreads();
      const int nw = min(W, steps - r0);
      for (int c = grp; c < C1; c += W) {
        if (s_start[c] == s_start[c + 1]) continue;
#pragma unroll
        for (int j = 0; j < TAIL_TT; ++j)
          for (int w = 0; w < nw; ++w) {
            s_acc[c * TC + col + j * CS] += s_part[((size_t)w * 2 * C1 + c) * TC + col + j * CS];
            s_acc[(C1 + c) * TC + col + j * CS] += s_part[((size_t)w * 2 * C1 + C1 + c) * TC + col + j * CS];
          }
      }
      __syncthreads();
    }
    if (grp != 0) return;
    int d0 = 0;
    float q[TAIL_TT][8], x[TAIL_TT][8], bv[8];
    for (; d0 + 8 <= D; d0 += 8) tail_empty_dots<CS, 8>(d0, qk2, cand, bias, D, T, t0, col, q, x, bv, eq, ec);
    if (d0 < D) {
      float q4[TAIL_TT][4], x4[TAIL_TT][4], bv4[4];
      tail_empty_dots<CS, 4>(d0, qk2, cand, bias, D, T, t0, col, q4, x4, bv4, eq, ec);
    }
  }

  // 5. inter-cluster attention and the click score
  const uint8_t* cm = cmask + (size_t)b * C1;
#pragma unroll
  for (int j = 0; j < TAIL_TT; ++j) {
    const int tl = col + j * CS;
    if (t0 + tl >= T) continue;
    float m = -INFINITY;
    for (int c = 0; c < C1; ++c) {
      const float l = cm[c] ? scale * (s_start[c] < s_start[c + 1] ? s_acc[c * TC + tl] : eq[j]) : -1e9f;
      m = fmaxf(m, l);
    }
    float sum = 0.f;
    for (int c = 0; c < C1; ++c) {
      const float l = cm[c] ? scale * (s_start[c] < s_start[c + 1] ? s_acc[c * TC + tl] : eq[j]) : -1e9f;
      sum += expf(l - m);
    }
    const float inv = 1.0f / sum;
    float out = 0.f;
    for (int c = 0; c < C1; ++c) {
      const bool full = s_start[c] < s_start[c + 1];
      const float l = cm[c] ? scale * (full ? s_acc[c * TC + tl] : eq[j]) : -1e9f;
      const float beta = expf(l - m) * inv, dot = full ? s_acc[(C1 + c) * TC + tl] : ec[j];
      out = fmaf(beta, dot, out);
      if constexpr (EX) {
        ex.beta[(size_t)(t0 + tl) * C1 + c] = beta;
        ex.contrib[(size_t)(t0 + tl) * C1 + c] = beta * dot;
      }
    }
    srow[t0 + tl] = out;
  }
}

template <int NT>
__global__ void __launch_bounds__(NT) cluster_tail_scores_kernel(
    const float* __restrict__ Kp, const float* __restrict__ g, const float* __restrict__ Wg, const int64_t* __restrict__ idx,
    const uint8_t* __restrict__ cmask, const float* __restrict__ Qp, const float* __restrict__ qk2,
    const float* __restrict__ cand, const float* __restrict__ bias, int H, int Au, int D, int C1, int T, float scale,
    float* __restrict__ scores, int64_t lds) {
  const int b = blockIdx.x;
  tail_cta<NT, 1>(Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias, b, H, Au, D, C1, T, blockIdx.y * NT * TAIL_TT, scale,
               scores + (size_t)b * lds);
}

// packed candidate lists: CTA x = (user b, slice s) of ns slices of TAIL_PC candidates, W warps; user b's candidates are
// rows [row_off[b], row_off[b + 1]) of Qp / qk2 / cand.  The offsets come from the device unchecked: the count is clamped
// to [0, n_max] and the rows to [0, rows), and a CTA whose slice starts past the count exits before it reads anything else.
// EX: also the explanation of every score, [B, lds, H] alpha_out and [B, lds, C1] beta_out / contrib_out (tail_cta).
template <int W, bool EX>
__global__ void __launch_bounds__(32 * W) cluster_tail_scores_packed_kernel(
    const float* __restrict__ Kp, const float* __restrict__ g, const float* __restrict__ Wg, const int64_t* __restrict__ idx,
    const uint8_t* __restrict__ cmask, const int32_t* __restrict__ row_off, int64_t rows, const float* __restrict__ Qp,
    const float* __restrict__ qk2, const float* __restrict__ cand, const float* __restrict__ bias, int ns, int H, int Au,
    int D, int C1, int n_max, float scale, float* __restrict__ scores, int64_t lds, float* __restrict__ alpha_out,
    float* __restrict__ beta_out, float* __restrict__ contrib_out) {
  const int b = blockIdx.x / ns, t0 = (blockIdx.x % ns) * TAIL_PC;
  const int64_t lo = min(max((int64_t)row_off[b], (int64_t)0), rows);
  const int64_t hi = min(max((int64_t)row_off[b + 1], lo), rows);
  const int T = (int)min(hi - lo, (int64_t)n_max);
  if (t0 >= T) return;
  if constexpr (EX)
    tail_cta<32, W, true>(Kp, g, Wg, idx, cmask, Qp + lo * Au, qk2 + lo * D, cand + lo * D, bias, b, H, Au, D, C1, T, t0,
                          scale, scores + (size_t)b * lds,
                          TailEx{alpha_out + (size_t)b * lds * H, beta_out + (size_t)b * lds * C1,
                                 contrib_out + (size_t)b * lds * C1});
  else
    tail_cta<32, W>(Kp, g, Wg, idx, cmask, Qp + lo * Au, qk2 + lo * D, cand + lo * D, bias, b, H, Au, D, C1, T, t0, scale,
                    scores + (size_t)b * lds);
}

// dynamic shared memory of a CTA of TC candidates: the logits / alpha and the larger of the accumulators and the staging
// (W > 1: and W rounds of partial dots after the accumulators)
static size_t tail_smem(int H, int C1, int TC, int W = 1) {
  const size_t acc = (size_t)2 * C1 * TC * (W > 1 ? 1 + W : 1), stage = (size_t)TAIL_KC * (TC + 1) + (size_t)H * TAIL_KC;
  return ((size_t)H * TC + (acc > stage ? acc : stage)) * sizeof(float);
}

// raise a kernel's dynamic shared memory limit to ``most`` bytes, once per device
static int tail_smem_attr(const void* fn, size_t most, bool* attr_set) {
  int dev = 0;
  NNR_CUDA(cudaGetDevice(&dev));
  if (dev >= 64 || !attr_set[dev]) {
    NNR_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
    if (dev < 64) attr_set[dev] = true;
  }
  return 0;
}

template <int NT>
static int tail_launch(const float* Kp, const float* g, const float* Wg, const int64_t* idx, const uint8_t* cmask,
                       const float* Qp, const float* qk2, const float* cand, const float* bias, int B, int H, int Au, int D,
                       int C1, int T, float scale, float* scores, int64_t lds, size_t smem, size_t most, void* stream) {
  static bool attr_set[64] = {};                                // one per instantiation and device
  if (int rc = tail_smem_attr((const void*)cluster_tail_scores_kernel<NT>, most, attr_set)) return rc;
  constexpr int TC = NT * TAIL_TT;
  cluster_tail_scores_kernel<NT><<<dim3(B, (T + TC - 1) / TC), NT, smem, (cudaStream_t)stream>>>(
      Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias, H, Au, D, C1, T, scale, scores, lds);
  NNR_LAUNCH_CHECK(NT == 128 ? "cluster_tail_scores_kernel<128>" : "cluster_tail_scores_kernel<64>");
  return 0;
}

// the 256-candidate CTA when its shared memory fits next to a second CTA's on the SM (the default H = 50, C1 = 19 needs
// 90 KB), the 128-candidate CTA otherwise: at H = 256, C1 = 72 it needs 200 KB
#define TAIL_SMEM_PAIR (113 * 1024)

extern "C" int nnr_cluster_tail_scores(const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                                       const uint8_t* cmask, const float* Qp, const float* qk2, const float* cand,
                                       const float* bias, int B, int H, int Au, int D, int C1, int T, float scale,
                                       float* scores, int64_t lds, void* stream) {
  const char* who = "nnr_cluster_tail_scores";
  NNR_REQUIRE(Kp && g && Wg && idx && cmask && Qp && qk2 && cand && bias && scores, NNR_ERR_ARG,
              "%s: Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias and scores must not be NULL", who);
  NNR_REQUIRE(B >= 0 && H >= 1 && Au >= 1 && D >= 1 && C1 >= 1, NNR_ERR_ARG,
              "%s: bad sizes B=%d H=%d Au=%d D=%d C1=%d (B >= 0, the others >= 1)", who, B, H, Au, D, C1);
  NNR_REQUIRE(T >= 1 && T <= NNR_TOPK_MAX_TILE, NNR_ERR_ARG, "%s: T must be in [1, %d], got %d", who, NNR_TOPK_MAX_TILE, T);
  NNR_REQUIRE(lds >= T, NNR_ERR_ARG, "%s: lds (%lld) < T (%d)", who, (long long)lds, T);
  NNR_REQUIRE(H <= TAIL_MAXH && C1 <= TAIL_MAXC, NNR_ERR_UNSUPPORTED, "%s: needs H <= %d and C1 <= %d, got H=%d C1=%d", who,
              TAIL_MAXH, TAIL_MAXC, H, C1);
  NNR_REQUIRE(D % 4 == 0 && nnr_aligned16(g) && nnr_aligned16(Wg) && nnr_aligned16(qk2) && nnr_aligned16(cand) &&
                  nnr_aligned16(bias),
              NNR_ERR_UNSUPPORTED, "%s: needs D %% 4 == 0 (got %d) and 16-byte aligned g, Wg, qk2, cand and bias", who, D);
  if (B == 0) return 0;
  const size_t wide = tail_smem(H, C1, 128 * TAIL_TT);
  if (wide <= TAIL_SMEM_PAIR)
    return tail_launch<128>(Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias, B, H, Au, D, C1, T, scale, scores, lds, wide, TAIL_SMEM_PAIR,
                           stream);
  return tail_launch<64>(Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias, B, H, Au, D, C1, T, scale, scores, lds,
                         tail_smem(H, C1, 64 * TAIL_TT), tail_smem(TAIL_MAXH, TAIL_MAXC, 64 * TAIL_TT), stream);
}

template <int W, bool EX>
static int tail_packed_launch(const float* Kp, const float* g, const float* Wg, const int64_t* idx, const uint8_t* cmask,
                              const int32_t* row_off, int64_t rows, const float* Qp, const float* qk2, const float* cand,
                              const float* bias, int B, int H, int Au, int D, int C1, int n_max, float scale, float* scores,
                              int64_t lds, float* alpha_out, float* beta_out, float* contrib_out, size_t smem, size_t most,
                              void* stream) {
  static bool attr_set[64] = {};
  if (int rc = tail_smem_attr((const void*)cluster_tail_scores_packed_kernel<W, EX>, most, attr_set)) return rc;
  const int ns = (n_max + TAIL_PC - 1) / TAIL_PC;
  cluster_tail_scores_packed_kernel<W, EX><<<(unsigned)((int64_t)B * ns), 32 * W, smem, (cudaStream_t)stream>>>(
      Kp, g, Wg, idx, cmask, row_off, rows, Qp, qk2, cand, bias, ns, H, Au, D, C1, n_max, scale, scores, lds, alpha_out,
      beta_out, contrib_out);
  NNR_LAUNCH_CHECK(EX ? (W == 8 ? "cluster_tail_scores_packed_kernel<8, explain>" : "cluster_tail_scores_packed_kernel<2, explain>")
                      : (W == 8 ? "cluster_tail_scores_packed_kernel<8>" : "cluster_tail_scores_packed_kernel<2>"));
  return 0;
}

// the checks and the launch of nnr_cluster_tail_scores_packed / nnr_cluster_tail_explain_packed (EX), past the NULL checks
template <bool EX>
static int tail_packed(const char* who, const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                       const uint8_t* cmask, const int32_t* row_off, int64_t rows, const float* Qp, const float* qk2,
                       const float* cand, const float* bias, int B, int H, int Au, int D, int C1, int n_max, float scale,
                       float* scores, int64_t lds, float* alpha_out, float* beta_out, float* contrib_out, void* stream) {
  NNR_REQUIRE(B >= 0 && H >= 1 && Au >= 1 && D >= 1 && C1 >= 1, NNR_ERR_ARG,
              "%s: bad sizes B=%d H=%d Au=%d D=%d C1=%d (B >= 0, the others >= 1)", who, B, H, Au, D, C1);
  NNR_REQUIRE(n_max >= 1 && n_max <= lds, NNR_ERR_ARG, "%s: n_max must be in [1, lds = %lld], got %d", who, (long long)lds,
              n_max);
  NNR_REQUIRE(rows >= 0 && rows < ((int64_t)1 << 31), NNR_ERR_ARG, "%s: rows must be in [0, 2^31), got %lld", who,
              (long long)rows);
  NNR_REQUIRE((int64_t)B * ((n_max + TAIL_PC - 1) / TAIL_PC) < ((int64_t)1 << 31), NNR_ERR_ARG,
              "%s: bad sizes: B (%d) x n_max (%d) needs more than 2^31 - 1 CTAs", who, B, n_max);
  NNR_REQUIRE(H <= TAIL_MAXH && C1 <= TAIL_MAXC, NNR_ERR_UNSUPPORTED, "%s: needs H <= %d and C1 <= %d, got H=%d C1=%d", who,
              TAIL_MAXH, TAIL_MAXC, H, C1);
  NNR_REQUIRE(D % 4 == 0 && nnr_aligned16(g) && nnr_aligned16(Wg) && nnr_aligned16(qk2) && nnr_aligned16(cand) &&
                  nnr_aligned16(bias),
              NNR_ERR_UNSUPPORTED, "%s: needs D %% 4 == 0 (got %d) and 16-byte aligned g, Wg, qk2, cand and bias", who, D);
  if (B == 0) return 0;
  // 8 warps when two CTAs fit on an SM (the default H = 50, C1 = 19 needs 98 KB), 2 otherwise (176 KB at H = 256, C1 = 72)
  const size_t wide = tail_smem(H, C1, TAIL_PC, 8);
  if (wide <= TAIL_SMEM_PAIR)
    return tail_packed_launch<8, EX>(Kp, g, Wg, idx, cmask, row_off, rows, Qp, qk2, cand, bias, B, H, Au, D, C1, n_max,
                                     scale, scores, lds, alpha_out, beta_out, contrib_out, wide, TAIL_SMEM_PAIR, stream);
  return tail_packed_launch<2, EX>(Kp, g, Wg, idx, cmask, row_off, rows, Qp, qk2, cand, bias, B, H, Au, D, C1, n_max, scale,
                                   scores, lds, alpha_out, beta_out, contrib_out, tail_smem(H, C1, TAIL_PC, 2),
                                   tail_smem(TAIL_MAXH, TAIL_MAXC, TAIL_PC, 2), stream);
}

extern "C" int nnr_cluster_tail_scores_packed(const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                                              const uint8_t* cmask, const int32_t* row_off, int64_t rows, const float* Qp,
                                              const float* qk2, const float* cand, const float* bias, int B, int H, int Au,
                                              int D, int C1, int n_max, float scale, float* scores, int64_t lds,
                                              void* stream) {
  const char* who = "nnr_cluster_tail_scores_packed";
  NNR_REQUIRE(Kp && g && Wg && idx && cmask && row_off && Qp && qk2 && cand && bias && scores, NNR_ERR_ARG,
              "%s: Kp, g, Wg, idx, cmask, row_off, Qp, qk2, cand, bias and scores must not be NULL", who);
  return tail_packed<false>(who, Kp, g, Wg, idx, cmask, row_off, rows, Qp, qk2, cand, bias, B, H, Au, D, C1, n_max, scale,
                            scores, lds, nullptr, nullptr, nullptr, stream);
}

extern "C" int nnr_cluster_tail_explain_packed(const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                                               const uint8_t* cmask, const int32_t* row_off, int64_t rows, const float* Qp,
                                               const float* qk2, const float* cand, const float* bias, int B, int H, int Au,
                                               int D, int C1, int n_max, float scale, float* scores, int64_t lds,
                                               float* alpha_out, float* beta_out, float* contrib_out, void* stream) {
  const char* who = "nnr_cluster_tail_explain_packed";
  NNR_REQUIRE(Kp && g && Wg && idx && cmask && row_off && Qp && qk2 && cand && bias && scores && alpha_out && beta_out &&
                  contrib_out,
              NNR_ERR_ARG,
              "%s: Kp, g, Wg, idx, cmask, row_off, Qp, qk2, cand, bias, scores, alpha_out, beta_out and contrib_out must "
              "not be NULL", who);
  return tail_packed<true>(who, Kp, g, Wg, idx, cmask, row_off, rows, Qp, qk2, cand, bias, B, H, Au, D, C1, n_max, scale,
                           scores, lds, alpha_out, beta_out, contrib_out, stream);
}
