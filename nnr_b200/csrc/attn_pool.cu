// Fused masked attention pooling over segments (scores -> masked softmax -> weighted sum in one
// kernel), forward and backward.  Replaces the chain of Linear/tanh/masked_fill/softmax/bmm calls of
// layers.py:167-175 (Attention) and layers.py:196-203 (ScaledDotProduct_CandidateAttention).
//
// One CTA per segment (a news item's tokens, or the 19 clusters of one (user, candidate) pair).
// The feature rows of the segment are read once for the scores and once for the weighted sum
// (second read is an L2 hit: a segment is <= 128 x 1.6 KB); HBM-bound by design.
//   mode 0: score = w2 . U[p]                 (U = tanh(W1 x + b1) produced by nnr_gemm's epilogue)
//   mode 1: score = scale * X[p] . qvec[s]    (K folded onto the query: (K x).(q) == x.(K^T q))
#include "common.cuh"
#include "../../include/nnr_b200.h"

#define POOL_THREADS 128       // backward kernels
#ifndef POOL_FWD_THREADS
#define POOL_FWD_THREADS 256   // forward kernel (sweep on B200, fwd / bwd ms per step: 64 threads 0.417 / 0.399, 128: 0.256 / 0.305,
                               // 256: 0.207 / 0.344, 512: 0.250 / -)
#endif

__global__ void __launch_bounds__(POOL_FWD_THREADS) attn_pool_fwd_kernel(nnr_pool_args a) {
  extern __shared__ float sc[];  // [max_len]
  __shared__ float red[POOL_FWD_THREADS / 32];
  const int s = a.seg_order ? a.seg_order[blockIdx.x] : blockIdx.x;
  const int beg = a.seg_off ? a.seg_off[s] : s * a.fixed_len;
  const int n = a.seg_off ? (a.seg_off[s + 1] - beg) : a.fixed_len;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = POOL_FWD_THREADS / 32;
  // scores: a warp takes two rows per iteration so that both rows' loads are in flight before the shuffle reductions
  {
    const float* src = (a.mode == 0) ? a.U : a.X;
    const int64_t lds = (a.mode == 0) ? a.ldu : a.ldx;
    const float* wv = (a.mode == 0) ? a.w2 : a.qvec + (size_t)s * a.ldq;
    const int nv = (a.mode == 0) ? a.A : a.D;
    for (int t = w; t < n; t += 2 * nw) {
      const int t1 = t + nw;
      const bool two = t1 < n;
      const float* r0 = src + ((size_t)beg + t) * lds;
      const float* r1 = two ? src + ((size_t)beg + t1) * lds : r0;
      float v0 = 0.f, v1 = 0.f;
      for (int k = lane; k < nv; k += 32) { const float wk = wv[k]; v0 += r0[k] * wk; v1 += r1[k] * wk; }
      v0 = warp_sum(v0);
      v1 = warp_sum(v1);
      if (a.mode == 1) { v0 *= a.scale; v1 *= a.scale; }
      if (a.mask) {
        if (a.mask[(size_t)beg + t] == 0) v0 = -1e9f;
        if (two && a.mask[(size_t)beg + t1] == 0) v1 = -1e9f;
      }
      if (lane == 0) { sc[t] = v0; if (two) sc[t1] = v1; }
    }
  }
  __syncthreads();
  // softmax over the segment
  float m = -INFINITY;
  for (int t = tid; t < n; t += POOL_FWD_THREADS) m = fmaxf(m, sc[t]);
  m = warp_max(m);
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = red[0];
  for (int i = 1; i < nw; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float sum = 0.f;
  for (int t = tid; t < n; t += POOL_FWD_THREADS) { float e = expf(sc[t] - m); sc[t] = e; sum += e; }
  sum = warp_sum(sum);
  if (lane == 0) red[w] = sum;
  __syncthreads();
  sum = 0.f;
  for (int i = 0; i < nw; ++i) sum += red[i];
  const float inv = 1.0f / sum;
  for (int t = tid; t < n; t += POOL_FWD_THREADS) {
    float al = sc[t] * inv;
    sc[t] = al;
    if (a.alpha) a.alpha[(size_t)beg + t] = al;
  }
  __syncthreads();
  for (int d = tid; d < a.D; d += POOL_FWD_THREADS) {
    // four independent partial sums keep four loads in flight; combined in a fixed order
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    const float* x = a.X + (size_t)beg * a.ldx + d;
    int t = 0;
    for (; t + 4 <= n; t += 4) {
      a0 += sc[t] * x[(size_t)t * a.ldx];
      a1 += sc[t + 1] * x[(size_t)(t + 1) * a.ldx];
      a2 += sc[t + 2] * x[(size_t)(t + 2) * a.ldx];
      a3 += sc[t + 3] * x[(size_t)(t + 3) * a.ldx];
    }
    for (; t < n; ++t) a0 += sc[t] * x[(size_t)t * a.ldx];
    a.pooled[(size_t)s * a.ldp + d] = (a0 + a1) + (a2 + a3);
  }
}

__global__ void __launch_bounds__(POOL_THREADS) attn_pool_bwd_kernel(nnr_pool_args a) {
  extern __shared__ float sm[];  // [2*max_len]: alpha, da
  __shared__ float red[POOL_THREADS / 32];
  const int s = a.seg_order ? a.seg_order[blockIdx.x] : blockIdx.x;
  const int beg = a.seg_off ? a.seg_off[s] : s * a.fixed_len;
  const int n = a.seg_off ? (a.seg_off[s + 1] - beg) : a.fixed_len;
  float* al = sm;
  float* da = sm + a.max_len;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = POOL_THREADS / 32;
  const float* dp = a.dpooled + (size_t)s * a.lddp;
  // dalpha[t] = dpooled . X[p]
  for (int t = w; t < n; t += nw) {
    const float* x = a.X + ((size_t)beg + t) * a.ldx;
    float v = 0.f;
    for (int d = lane; d < a.D; d += 32) v += dp[d] * x[d];
    v = warp_sum(v);
    if (lane == 0) { da[t] = v; al[t] = a.alpha[(size_t)beg + t]; }
  }
  __syncthreads();
  float dot = 0.f;
  for (int t = tid; t < n; t += POOL_THREADS) dot += al[t] * da[t];
  dot = warp_sum(dot);
  if (lane == 0) red[w] = dot;
  __syncthreads();
  dot = 0.f;
  for (int i = 0; i < nw; ++i) dot += red[i];
  __syncthreads();
  for (int t = tid; t < n; t += POOL_THREADS) {
    float v = al[t] * (da[t] - dot);           // dL/dscore (masked rows have alpha == 0 -> 0)
    if (a.mode == 1) v *= a.scale;
    da[t] = v;
  }
  __syncthreads();
  // dX and (mode 1) dqvec.  Loads of four tokens are issued before the first store (the compiler cannot move a load
  // across a store through a possibly aliasing pointer), so four rows are in flight per thread.
  const float* __restrict__ Xr = a.X;
  float* __restrict__ dXw = a.dX;
  for (int d = tid; d < a.D; d += POOL_THREADS) {
    const float g = dp[d];
    const float q = (a.mode == 1) ? a.qvec[(size_t)s * a.ldq + d] : 0.f;
    float accq = 0.f;
    int t = 0;
    for (; t + 4 <= n; t += 4) {
      float xv[4] = {0.f, 0.f, 0.f, 0.f}, old[4] = {0.f, 0.f, 0.f, 0.f};
      if (a.mode == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) xv[j] = Xr[((size_t)beg + t + j) * a.ldx + d];
      }
      if (a.accumulate_dx) {
#pragma unroll
        for (int j = 0; j < 4; ++j) old[j] = dXw[((size_t)beg + t + j) * a.lddx + d];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = al[t + j] * g;
        if (a.mode == 1) { v += da[t + j] * q; accq += da[t + j] * xv[j]; }
        dXw[((size_t)beg + t + j) * a.lddx + d] = old[j] + v;
      }
    }
    for (; t < n; ++t) {
      const size_t p = (size_t)beg + t;
      float v = al[t] * g;
      if (a.mode == 1) { v += da[t] * q; accq += da[t] * Xr[p * a.ldx + d]; }
      float* o = dXw + p * a.lddx + d;
      *o = a.accumulate_dx ? (*o + v) : v;
    }
    if (a.mode == 1 && a.dqvec) a.dqvec[(size_t)s * a.lddq + d] = accq;
  }
  if (a.mode == 0) {
    const float* __restrict__ Ur = a.U;
    float* __restrict__ dUw = a.dU;
    for (int k = tid; k < a.A; k += POOL_THREADS) {
      const float wk = a.w2[k];
      float accw = 0.f;
      int t = 0;
      for (; t + 4 <= n; t += 4) {
        float u[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) u[j] = Ur[((size_t)beg + t + j) * a.ldu + k];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          dUw[((size_t)beg + t + j) * a.lddu + k] = da[t + j] * wk * (1.f - u[j] * u[j]);
          accw += da[t + j] * u[j];
        }
      }
      for (; t < n; ++t) {
        const size_t p = (size_t)beg + t;
        const float u = Ur[p * a.ldu + k];
        dUw[p * a.lddu + k] = da[t] * wk * (1.f - u * u);
        accw += da[t] * u;
      }
      a.dw2_partial[(size_t)s * a.A + k] = accw;
    }
  }
}

// Row-parallel backward (the default when D and A are multiples of 4, <= 1024, and the rows are 16-byte aligned): the
// column-per-thread kernel above walks ALL rows of the segment serially in every thread (128 rows x 4 column passes for
// the longest news bodies -- the launch lasted as long as its longest CTA).  Here a warp owns whole rows (t = w, w + nw,
// ...), lanes cover the row in 16-byte pieces, so the rows of a segment are independent streams; the two per-segment
// reductions over rows (dqvec in mode 1, dw2_partial in mode 0) are kept per warp in registers and combined across
// the warps in warp order at the end (fixed order -> deterministic).
#define POOL_K4 8            // 16-byte column groups per lane: D, A <= 32 * 4 * POOL_K4 = 1024 (K4 = 4 when they are <= 512)
template <int K4>
__global__ void __launch_bounds__(POOL_THREADS) attn_pool_bwd_rows_kernel(nnr_pool_args a, int ml4) {
  extern __shared__ __align__(16) float sm[];   // alpha[ml4], da[ml4], dpooled[D], qvec[D] (mode 1), red[nw][max(D, A)]
  __shared__ float red[POOL_THREADS / 32];
  const int s = a.seg_order ? a.seg_order[blockIdx.x] : blockIdx.x;
  const int beg = a.seg_off ? a.seg_off[s] : s * a.fixed_len;
  const int n = a.seg_off ? (a.seg_off[s + 1] - beg) : a.fixed_len;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = POOL_THREADS / 32;
  const int D4 = a.D >> 2, A4 = a.A >> 2;
  float* al = sm;
  float* da = al + ml4;
  float4* s_dp = reinterpret_cast<float4*>(da + ml4);
  float4* s_q = s_dp + D4;
  float4* s_red = s_q + (a.mode == 1 ? D4 : 0);
  const int R4 = (a.mode == 1) ? D4 : A4;
  {
    const float4* dp4 = reinterpret_cast<const float4*>(a.dpooled + (size_t)s * a.lddp);
    for (int c = tid; c < D4; c += POOL_THREADS) s_dp[c] = dp4[c];
    if (a.mode == 1) {
      const float4* q4 = reinterpret_cast<const float4*>(a.qvec + (size_t)s * a.ldq);
      for (int c = tid; c < D4; c += POOL_THREADS) s_q[c] = q4[c];
    }
  }
  __syncthreads();
  // dalpha[t] = dpooled . X[t]
  for (int t = w; t < n; t += nw) {
    const float4* x4 = reinterpret_cast<const float4*>(a.X + ((size_t)beg + t) * a.ldx);
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < K4; ++k) {
      const int c = lane + 32 * k;
      if (c < D4) { const float4 x = __ldg(x4 + c); const float4 g = s_dp[c]; v += x.x * g.x + x.y * g.y + x.z * g.z + x.w * g.w; }
    }
    v = warp_sum(v);
    if (lane == 0) { da[t] = v; al[t] = a.alpha[(size_t)beg + t]; }
  }
  __syncthreads();
  float dot = 0.f;
  for (int t = tid; t < n; t += POOL_THREADS) dot += al[t] * da[t];
  dot = warp_sum(dot);
  if (lane == 0) red[w] = dot;
  __syncthreads();
  dot = 0.f;
  for (int i = 0; i < nw; ++i) dot += red[i];
  __syncthreads();
  for (int t = tid; t < n; t += POOL_THREADS) {
    float v = al[t] * (da[t] - dot);           // dL/dscore (masked rows have alpha == 0 -> 0)
    if (a.mode == 1) v *= a.scale;
    da[t] = v;
  }
  __syncthreads();
  float4 acc[K4];                         // per-warp partial of dqvec (mode 1) / dw2 (mode 0)
#pragma unroll
  for (int k = 0; k < K4; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  // dX rows
  for (int t = w; t < n; t += nw) {
    const float alt = al[t], dat = da[t];
    const size_t p = (size_t)beg + t;
    const float4* x4 = reinterpret_cast<const float4*>(a.X + p * a.ldx);
    float4* o4 = reinterpret_cast<float4*>(a.dX + p * a.lddx);
    float4 xv[K4], old[K4];
#pragma unroll
    for (int k = 0; k < K4; ++k) {
      const int c = lane + 32 * k;
      xv[k] = make_float4(0.f, 0.f, 0.f, 0.f); old[k] = xv[k];
      if (c < D4) {
        if (a.mode == 1) xv[k] = __ldg(x4 + c);
        if (a.accumulate_dx) old[k] = o4[c];
      }
    }
#pragma unroll
    for (int k = 0; k < K4; ++k) {
      const int c = lane + 32 * k;
      if (c < D4) {
        const float4 g = s_dp[c];
        float4 v = make_float4(alt * g.x, alt * g.y, alt * g.z, alt * g.w);
        if (a.mode == 1) {
          const float4 q = s_q[c];
          v.x += dat * q.x; v.y += dat * q.y; v.z += dat * q.z; v.w += dat * q.w;
          acc[k].x += dat * xv[k].x; acc[k].y += dat * xv[k].y; acc[k].z += dat * xv[k].z; acc[k].w += dat * xv[k].w;
        }
        o4[c] = make_float4(old[k].x + v.x, old[k].y + v.y, old[k].z + v.z, old[k].w + v.w);
      }
    }
  }
  if (a.mode == 0) {
    const float4* w4 = reinterpret_cast<const float4*>(a.w2);
    for (int t = w; t < n; t += nw) {
      const float dat = da[t];
      const size_t p = (size_t)beg + t;
      const float4* u4 = reinterpret_cast<const float4*>(a.U + p * a.ldu);
      float4* o4 = reinterpret_cast<float4*>(a.dU + p * a.lddu);
#pragma unroll
      for (int k = 0; k < K4; ++k) {
        const int c = lane + 32 * k;
        if (c < A4) {
          const float4 u = __ldg(u4 + c), wk = __ldg(w4 + c);
          o4[c] = make_float4(dat * wk.x * (1.f - u.x * u.x), dat * wk.y * (1.f - u.y * u.y), dat * wk.z * (1.f - u.z * u.z),
                              dat * wk.w * (1.f - u.w * u.w));
          acc[k].x += dat * u.x; acc[k].y += dat * u.y; acc[k].z += dat * u.z; acc[k].w += dat * u.w;
        }
      }
    }
  }
  // per-segment reductions over rows: warp partials combined in warp order
  float* outv = (a.mode == 1) ? (a.dqvec ? a.dqvec + (size_t)s * a.lddq : nullptr) : a.dw2_partial + (size_t)s * a.A;
  if (outv) {
#pragma unroll
    for (int k = 0; k < K4; ++k) {
      const int c = lane + 32 * k;
      if (c < R4) s_red[w * R4 + c] = acc[k];
    }
    __syncthreads();
    for (int c = tid; c < R4; c += POOL_THREADS) {
      float4 t4 = s_red[c];
      for (int ww = 1; ww < nw; ++ww) { const float4 o = s_red[ww * R4 + c]; t4.x += o.x; t4.y += o.y; t4.z += o.z; t4.w += o.w; }
      reinterpret_cast<float4*>(outv)[c] = t4;
    }
  }
}

static int pool_validate(const nnr_pool_args* a, bool bwd) {
  NNR_REQUIRE(a && a->X && a->S > 0 && a->D > 0 && a->max_len > 0, NNR_ERR_ARG, "nnr_attn_pool: bad arguments");
  NNR_REQUIRE(a->seg_off || a->fixed_len > 0, NNR_ERR_ARG, "nnr_attn_pool: need seg_off or fixed_len");
  NNR_REQUIRE(!(a->seg_off == nullptr && a->fixed_len > a->max_len), NNR_ERR_ARG, "nnr_attn_pool: fixed_len > max_len");
  NNR_REQUIRE(a->mode == 0 || a->mode == 1, NNR_ERR_ARG, "nnr_attn_pool: bad mode");
  if (a->mode == 0) NNR_REQUIRE(a->U && a->w2 && a->A > 0, NNR_ERR_ARG, "nnr_attn_pool: mode 0 needs U, w2");
  else NNR_REQUIRE(a->qvec, NNR_ERR_ARG, "nnr_attn_pool: mode 1 needs qvec");
  NNR_REQUIRE(a->max_len <= 4096, NNR_ERR_UNSUPPORTED, "nnr_attn_pool: max_len > 4096");
  if (!bwd) NNR_REQUIRE(a->pooled, NNR_ERR_ARG, "nnr_attn_pool_fwd: pooled is null");
  else {
    NNR_REQUIRE(a->dpooled && a->dX && a->alpha, NNR_ERR_ARG, "nnr_attn_pool_bwd: dpooled/dX/alpha null");
    if (a->mode == 0) NNR_REQUIRE(a->dU && a->dw2_partial, NNR_ERR_ARG, "nnr_attn_pool_bwd: mode 0 needs dU, dw2_partial");
  }
  return 0;
}

extern "C" int nnr_attn_pool_fwd(const nnr_pool_args* a, void* stream) {
  int rc = pool_validate(a, false);
  if (rc) return rc;
  attn_pool_fwd_kernel<<<a->S, POOL_FWD_THREADS, a->max_len * sizeof(float), (cudaStream_t)stream>>>(*a);
  NNR_LAUNCH_CHECK("attn_pool_fwd_kernel");
  return 0;
}
extern "C" int nnr_attn_pool_bwd(const nnr_pool_args* a, void* stream) {
  int rc = pool_validate(a, true);
  if (rc) return rc;
  const bool al = nnr_aligned16(a->X) && nnr_aligned16(a->dX) && nnr_aligned16(a->dpooled) && a->ldx % 4 == 0 && a->lddx % 4 == 0 &&
                  a->lddp % 4 == 0 && a->D % 4 == 0 && a->D <= 128 * POOL_K4;
  const bool al0 = a->mode != 0 || (nnr_aligned16(a->U) && nnr_aligned16(a->dU) && nnr_aligned16(a->w2) && nnr_aligned16(a->dw2_partial) &&
                                    a->ldu % 4 == 0 && a->lddu % 4 == 0 && a->A % 4 == 0 && a->A <= 128 * POOL_K4);
  const bool al1 = a->mode != 1 || (nnr_aligned16(a->qvec) && a->ldq % 4 == 0 && (!a->dqvec || (nnr_aligned16(a->dqvec) && a->lddq % 4 == 0)));
  if (al && al0 && al1) {
    const int ml4 = (a->max_len + 3) / 4 * 4;
    const int R = a->mode == 1 ? a->D : a->A;
    const size_t smem = ((size_t)2 * ml4 + a->D + (a->mode == 1 ? a->D : 0) + (size_t)(POOL_THREADS / 32) * R) * sizeof(float);
    if (smem <= 48 * 1024) {
      if (a->D <= 512 && (a->mode != 0 || a->A <= 512)) attn_pool_bwd_rows_kernel<4><<<a->S, POOL_THREADS, smem, (cudaStream_t)stream>>>(*a, ml4);
      else attn_pool_bwd_rows_kernel<8><<<a->S, POOL_THREADS, smem, (cudaStream_t)stream>>>(*a, ml4);
      NNR_LAUNCH_CHECK("attn_pool_bwd_rows_kernel");
      return 0;
    }
  }
  attn_pool_bwd_kernel<<<a->S, POOL_THREADS, 2 * a->max_len * sizeof(float), (cudaStream_t)stream>>>(*a);
  NNR_LAUNCH_CHECK("attn_pool_bwd_kernel");
  return 0;
}
