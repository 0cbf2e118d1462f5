// SUE user-encoder kernels: history-graph construction (bit-exact integer/fp32 work), dense graph ->
// compressed neighbour lists, deterministic GCN aggregation, intra-cluster (segment) attention.
//
// Replaces: MIND_corpus.py:162-216 (numpy preprocessing), torch.bmm(graph, feature) at layers.py:286,
// and torch_scatter.scatter_softmax / scatter_sum at userEncoders.py:88-89.
#include "common.cuh"
#include "../../include/nnr_b200.h"

// ------------------------------------------------------------------------------------------------
// nnr_sue_graph_build : one CTA per behaviour
// ------------------------------------------------------------------------------------------------
#define GB_MAXC 64
#define GB_MAXH 256
// flags (MIND_corpus.py:179-182,203-213): bit 0 = no_self_connection, bit 1 = no_adjacent_normalization,
// bit 2 = gcn_normalization_type == 'asymmetric' (D^-1 A instead of D^-1/2 A D^-1/2)
__global__ void sue_graph_build_kernel(const int32_t* __restrict__ categories, const int32_t* __restrict__ history_len,
                                       int H, int C, int flags, float* __restrict__ graph, uint8_t* __restrict__ cmask,
                                       int64_t* __restrict__ cidx) {
  __shared__ int s_cat[GB_MAXH];     // category of slot, or C for padding
  __shared__ int s_cnt[GB_MAXC];
  __shared__ float s_d[GB_MAXH + GB_MAXC];
  __shared__ int s_P;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int G = H + C;
  const bool self_conn = !(flags & NNR_GRAPH_NO_SELF_CONNECTION);
  const bool asym = (flags & NNR_GRAPH_ASYMMETRIC) != 0;
  int hl = history_len[b];
  hl = min(max(hl, 0), H);
  // the reference normalises only inside `if len(history.strip()) > 0` (MIND_corpus.py:185,203)
  const bool normalize = !(flags & NNR_GRAPH_NO_NORMALIZATION) && hl > 0;
  for (int i = tid; i < H; i += blockDim.x) {
    int c = (i < hl) ? categories[(size_t)b * H + i] : C;
    if (c < 0 || c > C) c = C;
    s_cat[i] = c;
  }
  for (int c = tid; c < C; c += blockDim.x) s_cnt[c] = 0;
  __syncthreads();
  if (tid < C) {   // counts (integer, order independent)
    int n = 0;
    for (int i = 0; i < hl; ++i) n += (s_cat[i] == tid);
    s_cnt[tid] = n;
  }
  __syncthreads();
  if (tid == 0) {
    int P = 0;
    for (int c = 0; c < C; ++c) P += (s_cnt[c] > 0);
    s_P = P;
  }
  __syncthreads();
  const int P = s_P;
  // row sums are exact small integers; symmetric: d = sqrt(1/deg), asymmetric: d = 1/deg, both in fp32, correctly rounded
  // like numpy (MIND_corpus.py:207,212)
  const int sc = self_conn ? 1 : 0;
  for (int v = tid; v < G; v += blockDim.x) {
    int deg;
    if (v < H) deg = (v < hl) ? (s_cnt[s_cat[v]] + sc) : sc;
    else { int c = v - H; deg = (s_cnt[c] > 0) ? (sc + s_cnt[c] + (P - 1)) : sc; }
    const float inv = __fdiv_rn(1.0f, (float)deg);          // deg == 0 only without self connections (rejected with normalisation)
    s_d[v] = asym ? inv : __fsqrt_rn(inv);
  }
  __syncthreads();
  if (cidx) for (int i = tid; i < H; i += blockDim.x) cidx[(size_t)b * H + i] = (int64_t)s_cat[i];
  if (cmask) for (int c = tid; c <= C; c += blockDim.x) cmask[(size_t)b * (C + 1) + c] = (c < C && s_cnt[c] > 0) ? 1 : 0;
  if (graph) {
    float* g = graph + (size_t)b * G * G;
    for (int e = tid; e < G * G; e += blockDim.x) {
      int i = e / G, j = e - i * G;
      bool edge;
      if (i == j) edge = self_conn;
      else if (i < H && j < H) edge = (i < hl && j < hl && s_cat[i] == s_cat[j]);
      else if (i < H) edge = (i < hl && s_cat[i] == j - H);
      else if (j < H) edge = (j < hl && s_cat[j] == i - H);
      else edge = (s_cnt[i - H] > 0 && s_cnt[j - H] > 0);
      // symmetric: (D A) D with A in {0,1} = fl(fl(d_i * 1) * d_j); asymmetric: D A = d_i; none: A
      float v = 0.0f;
      if (edge) v = !normalize ? 1.0f : (asym ? s_d[i] : __fmul_rn(s_d[i], s_d[j]));
      g[e] = v;
    }
  }
}

extern "C" int nnr_sue_graph_build_ex(const int32_t* categories, const int32_t* history_len, int B, int H, int C, int flags,
                                      float* graph, uint8_t* category_mask, int64_t* category_indices, void* stream) {
  NNR_REQUIRE(categories && history_len && B > 0 && H > 0 && C > 0, NNR_ERR_ARG, "nnr_sue_graph_build: bad arguments");
  NNR_REQUIRE(H <= GB_MAXH && C <= GB_MAXC, NNR_ERR_UNSUPPORTED, "nnr_sue_graph_build: H<=%d, C<=%d", GB_MAXH, GB_MAXC);
  NNR_REQUIRE((flags & ~7) == 0, NNR_ERR_ARG, "nnr_sue_graph_build: unknown flags 0x%x", flags);
  // config.py:111: adjacent normalisation is only defined with self connections (rows without edges would divide by 0)
  NNR_REQUIRE(!((flags & NNR_GRAPH_NO_SELF_CONNECTION) && !(flags & NNR_GRAPH_NO_NORMALIZATION)), NNR_ERR_ARG,
              "nnr_sue_graph_build: no_self_connection requires no_adjacent_normalization (reference config.py:111)");
  sue_graph_build_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(categories, history_len, H, C, flags, graph, category_mask,
                                                            category_indices);
  NNR_LAUNCH_CHECK("sue_graph_build_kernel");
  return 0;
}
extern "C" int nnr_sue_graph_build(const int32_t* categories, const int32_t* history_len, int B, int H, int C, float* graph,
                                   uint8_t* category_mask, int64_t* category_indices, void* stream) {
  return nnr_sue_graph_build_ex(categories, history_len, B, H, C, 0, graph, category_mask, category_indices, stream);
}

// ------------------------------------------------------------------------------------------------
// nnr_graph_to_csr : one warp per graph row, ballot compaction (ascending column order)
// ------------------------------------------------------------------------------------------------
__global__ void graph_to_csr_kernel(const float* __restrict__ graph, int BG, int G, int transpose, int32_t* __restrict__ nnz,
                                    int32_t* __restrict__ col, float* __restrict__ val) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= BG) return;
  int b = row / G, i = row - b * G;
  const float* g = graph + (size_t)b * G * G;
  int cnt = 0;
  for (int j0 = 0; j0 < G; j0 += 32) {
    int j = j0 + lane;
    float v = 0.f;
    if (j < G) v = transpose ? g[(size_t)j * G + i] : g[(size_t)i * G + j];
    bool nz = (v != 0.0f);
    unsigned m = __ballot_sync(0xffffffffu, nz);
    if (nz) {
      int pos = cnt + __popc(m & ((1u << lane) - 1));
      col[(size_t)row * G + pos] = j;
      val[(size_t)row * G + pos] = v;
    }
    cnt += __popc(m);
  }
  if (lane == 0) nnz[row] = cnt;
}
extern "C" int nnr_graph_to_csr(const float* graph, int B, int G, int transpose, int32_t* nnz, int32_t* col, float* val,
                                void* stream) {
  NNR_REQUIRE(graph && nnz && col && val && B > 0 && G > 0, NNR_ERR_ARG, "nnr_graph_to_csr: bad arguments");
  int rows = B * G;
  graph_to_csr_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(graph, rows, G, transpose, nnz, col, val);
  NNR_LAUNCH_CHECK("graph_to_csr_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// nnr_gcn_aggregate : out[b,i,:] = sum_e val[e] * x[b,col[e],:]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gcn_aggregate_kernel(const int32_t* __restrict__ nnz, const int32_t* __restrict__ col,
                                                            const float* __restrict__ val, const float* __restrict__ x, int G,
                                                            int D, const float* __restrict__ add, float* __restrict__ out) {
  extern __shared__ unsigned char smraw[];
  int* s_col = reinterpret_cast<int*>(smraw);
  float* s_val = reinterpret_cast<float*>(smraw + sizeof(int) * G);
  const int row = blockIdx.x;
  const int b = row / G;
  const int n = nnz[row];
  for (int e = threadIdx.x; e < n; e += blockDim.x) { s_col[e] = col[(size_t)row * G + e]; s_val[e] = val[(size_t)row * G + e]; }
  __syncthreads();
  const float* xb = x + (size_t)b * G * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float acc = 0.f;
    int e = 0;
    for (; e + 8 <= n; e += 8) {            // eight neighbour rows in flight, accumulated in edge order
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = xb[(size_t)s_col[e + j] * D + d];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = fmaf(s_val[e + j], v[j], acc);
    }
    for (; e < n; ++e) acc = fmaf(s_val[e], xb[(size_t)s_col[e] * D + d], acc);
    out[(size_t)row * D + d] = add ? acc + add[(size_t)row * D + d] : acc;     // + residual branch of the backward
  }
}
// D % 4 == 0: a thread owns 4 consecutive features (16-byte loads), one pass over the neighbour list per thread
__global__ void __launch_bounds__(256) gcn_aggregate_vec_kernel(const int32_t* __restrict__ nnz, const int32_t* __restrict__ col,
                                                                const float* __restrict__ val, const float* __restrict__ x, int G,
                                                                int D, const float* __restrict__ add, float* __restrict__ out) {
  extern __shared__ unsigned char smraw[];
  int* s_col = reinterpret_cast<int*>(smraw);
  float* s_val = reinterpret_cast<float*>(smraw + sizeof(int) * G);
  const int row = blockIdx.x;
  const int b = row / G;
  const int n = nnz[row];
  for (int e = threadIdx.x; e < n; e += blockDim.x) { s_col[e] = col[(size_t)row * G + e]; s_val[e] = val[(size_t)row * G + e]; }
  __syncthreads();
  const int D4 = D >> 2;
  const float4* xb = reinterpret_cast<const float4*>(x + (size_t)b * G * D);
  for (int d = threadIdx.x; d < D4; d += blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int e = 0;
    for (; e + 8 <= n; e += 8) {            // eight neighbour rows in flight, accumulated in edge order
      float4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldg(xb + (size_t)s_col[e + j] * D4 + d);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float w = s_val[e + j];
        acc.x = fmaf(w, v[j].x, acc.x); acc.y = fmaf(w, v[j].y, acc.y); acc.z = fmaf(w, v[j].z, acc.z); acc.w = fmaf(w, v[j].w, acc.w);
      }
    }
    for (; e < n; ++e) {
      const float w = s_val[e];
      const float4 v = __ldg(xb + (size_t)s_col[e] * D4 + d);
      acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y); acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
    }
    if (add) {
      const float4 r = __ldg(reinterpret_cast<const float4*>(add + (size_t)row * D) + d);
      acc.x += r.x; acc.y += r.y; acc.z += r.z; acc.w += r.w;
    }
    reinterpret_cast<float4*>(out + (size_t)row * D)[d] = acc;
  }
}
static int gcn_aggregate_launch(const int32_t* nnz, const int32_t* col, const float* val, const float* x, int B, int G, int D,
                                const float* add, float* out, void* stream, const char* who) {
  NNR_REQUIRE(nnz && col && val && x && out && B > 0 && G > 0 && D > 0, NNR_ERR_ARG, "%s: bad arguments", who);
  const size_t smem = (sizeof(int) + sizeof(float)) * G;
  if (D % 4 == 0 && nnr_aligned16(x) && nnr_aligned16(out) && (!add || nnr_aligned16(add))) {
    const int threads = ((D / 4 + 31) / 32 * 32) < 256 ? ((D / 4 + 31) / 32 * 32) : 256;
    gcn_aggregate_vec_kernel<<<B * G, threads, smem, (cudaStream_t)stream>>>(nnz, col, val, x, G, D, add, out);
  } else {
    gcn_aggregate_kernel<<<B * G, 256, smem, (cudaStream_t)stream>>>(nnz, col, val, x, G, D, add, out);
  }
  NNR_LAUNCH_CHECK("gcn_aggregate_kernel");
  return 0;
}
extern "C" int nnr_gcn_aggregate(const int32_t* nnz, const int32_t* col, const float* val, const float* x, int B, int G, int D,
                                 float* out, void* stream) {
  return gcn_aggregate_launch(nnz, col, val, x, B, G, D, nullptr, out, stream, "nnr_gcn_aggregate");
}
// out = A x + add (the residual term of the GCN backward, layers.py:320-322 differentiated); add must not alias out
extern "C" int nnr_gcn_aggregate_add(const int32_t* nnz, const int32_t* col, const float* val, const float* x, int B, int G,
                                     int D, const float* add, float* out, void* stream) {
  NNR_REQUIRE(add && add != out, NNR_ERR_ARG, "nnr_gcn_aggregate_add: add must be given and must not alias out");
  return gcn_aggregate_launch(nnz, col, val, x, B, G, D, add, out, stream, "nnr_gcn_aggregate_add");
}

// ------------------------------------------------------------------------------------------------
// intra-cluster attention (segment softmax by category + segment weighted sum)
// ------------------------------------------------------------------------------------------------
#define CI_MAXH 256
__device__ __forceinline__ bool dev_al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }
#define CI_MAXC 72
__global__ void __launch_bounds__(256) cluster_intra_fwd_kernel(const float* __restrict__ Kp, const float* __restrict__ Qp,
                                                                const float* __restrict__ g, const int64_t* __restrict__ idx,
                                                                int n, int H, int Au, int D, int C1, float scale,
                                                                float* __restrict__ alpha, float* __restrict__ intra) {
  __shared__ float s_a[CI_MAXH];
  __shared__ int s_idx[CI_MAXH];
  __shared__ int s_perm[CI_MAXH];
  __shared__ int s_start[CI_MAXC + 1];
  const int bk = blockIdx.x, b = bk / n;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int h = tid; h < H; h += 256) { int c = (int)idx[(size_t)b * H + h]; s_idx[h] = min(max(c, 0), C1 - 1); }
  const float* q = Qp + (size_t)bk * Au;
  for (int h = w; h < H; h += 8) {
    const float* kp = Kp + ((size_t)b * H + h) * Au;
    float v = 0.f;
    for (int a = lane; a < Au; a += 32) v += kp[a] * q[a];
    v = warp_sum(v);
    if (lane == 0) s_a[h] = v * scale;
  }
  __syncthreads();
  // stable counting sort of the H slots by cluster, one thread per cluster start and one per slot
  if (tid <= C1) {
    int pos = 0;
    for (int h = 0; h < H; ++h) pos += (s_idx[h] < tid);
    s_start[tid] = pos;
  }
  __syncthreads();
  if (tid < H) {
    const int c = s_idx[tid];
    int pos = s_start[c];
    for (int h = 0; h < tid; ++h) pos += (s_idx[h] == c);
    s_perm[pos] = tid;
  }
  __syncthreads();
  // per-slot softmax within its cluster (max-shifted, like torch_scatter.scatter_softmax)
  float my_alpha = 0.f;
  if (tid < H) {
    int c = s_idx[tid];
    float m = -INFINITY;
    for (int e = s_start[c]; e < s_start[c + 1]; ++e) m = fmaxf(m, s_a[s_perm[e]]);
    float sum = 0.f;
    for (int e = s_start[c]; e < s_start[c + 1]; ++e) sum += expf(s_a[s_perm[e]] - m);
    my_alpha = expf(s_a[tid] - m) / sum;
    alpha[(size_t)bk * H + tid] = my_alpha;
  }
  __syncthreads();
  if (tid < H) s_a[tid] = my_alpha;
  __syncthreads();
  const float* gb = g + (size_t)b * H * D;
  float* ob = intra + (size_t)bk * C1 * D;
  if ((D & 3) == 0 && dev_al16(g) && dev_al16(intra)) {
    // 16-byte version of the loop below: a thread owns four features
    const int D4 = D >> 2;
    const float4* gb4 = reinterpret_cast<const float4*>(gb);
    float4* ob4 = reinterpret_cast<float4*>(ob);
    for (int d = tid; d < D4; d += 256) {
      int c = 0;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int e0 = 0; e0 < H; e0 += 8) {
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (e0 + j < H) ? __ldg(gb4 + (size_t)s_perm[e0 + j] * D4 + d) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int e = e0 + j;
          if (e < H) {
            while (e == s_start[c + 1]) { ob4[(size_t)c * D4 + d] = acc; acc = make_float4(0.f, 0.f, 0.f, 0.f); ++c; }
            const float al = s_a[s_perm[e]];
            acc.x += al * v[j].x; acc.y += al * v[j].y; acc.z += al * v[j].z; acc.w += al * v[j].w;
          }
        }
      }
      for (; c < C1; ++c) { ob4[(size_t)c * D4 + d] = acc; acc = make_float4(0.f, 0.f, 0.f, 0.f); }
    }
    return;
  }
  for (int d = tid; d < D; d += 256) {
    // one pass over the slots in cluster order, eight feature rows in flight; a cluster's sum is stored when the
    // next cluster starts (empty clusters store 0); same summation order as a per-cluster loop
    int c = 0;
    float acc = 0.f;
    for (int e0 = 0; e0 < H; e0 += 8) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (e0 + j < H) ? gb[(size_t)s_perm[e0 + j] * D + d] : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int e = e0 + j;
        if (e < H) {
          while (e == s_start[c + 1]) { ob[(size_t)c * D + d] = acc; acc = 0.f; ++c; }
          acc += s_a[s_perm[e]] * v[j];
        }
      }
    }
    for (; c < C1; ++c) { ob[(size_t)c * D + d] = acc; acc = 0.f; }
  }
}

// A: per (b,k): da (scaled) -> da_ws, dQp
__global__ void __launch_bounds__(256) cluster_intra_bwd_a_kernel(const float* __restrict__ dintra, const float* __restrict__ Kp,
                                                                  const float* __restrict__ g, const int64_t* __restrict__ idx,
                                                                  const float* __restrict__ alpha, int n, int H, int Au, int D,
                                                                  int C1, float scale, float* __restrict__ da_ws,
                                                                  float* __restrict__ dQp) {
  __shared__ float s_da[CI_MAXH];
  __shared__ float s_al[CI_MAXH];
  __shared__ int s_idx[CI_MAXH];
  const int bk = blockIdx.x, b = bk / n;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int h = tid; h < H; h += 256) {
    int c = (int)idx[(size_t)b * H + h];
    s_idx[h] = min(max(c, 0), C1 - 1);
    s_al[h] = alpha[(size_t)bk * H + h];
  }
  __syncthreads();
  for (int h = w; h < H; h += 8) {
    const float* di = dintra + ((size_t)bk * C1 + s_idx[h]) * D;
    const float* gh = g + ((size_t)b * H + h) * D;
    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;          // four independent partial sums (fixed combination order)
    int d = lane;
    if ((D & 3) == 0 && dev_al16(dintra) && dev_al16(g)) {      // 16-byte loads, lane partials per component
      const float4* di4 = reinterpret_cast<const float4*>(di);
      const float4* gh4 = reinterpret_cast<const float4*>(gh);
      for (int q = lane; q < (D >> 2); q += 32) {
        const float4 x = __ldg(di4 + q), y = __ldg(gh4 + q);
        v0 += x.x * y.x; v1 += x.y * y.y; v2 += x.z * y.z; v3 += x.w * y.w;
      }
      d = D;
    }
    for (; d + 96 < D; d += 128) {
      v0 += di[d] * gh[d]; v1 += di[d + 32] * gh[d + 32]; v2 += di[d + 64] * gh[d + 64]; v3 += di[d + 96] * gh[d + 96];
    }
    for (; d < D; d += 32) v0 += di[d] * gh[d];
    float v = warp_sum((v0 + v1) + (v2 + v3));
    if (lane == 0) s_da[h] = v;   // dL/dalpha
  }
  __syncthreads();
  float out = 0.f;
  if (tid < H) {
    int c = s_idx[tid];
    float dot = 0.f;
    for (int h = 0; h < H; ++h) if (s_idx[h] == c) dot += s_al[h] * s_da[h];
    out = s_al[tid] * (s_da[tid] - dot) * scale;
  }
  __syncthreads();
  if (tid < H) { s_da[tid] = out; da_ws[(size_t)bk * H + tid] = out; }
  __syncthreads();
  for (int a = tid; a < Au; a += 256) {
    float acc = 0.f;
    int h = 0;
    for (; h + 8 <= H; h += 8) {             // eight rows of Kp in flight, accumulated in slot order
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = Kp[((size_t)b * H + h + j) * Au + a];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc += s_da[h + j] * v[j];
    }
    for (; h < H; ++h) acc += s_da[h] * Kp[((size_t)b * H + h) * Au + a];
    dQp[(size_t)bk * Au + a] = acc;
  }
}
// B: per (b,h): dKp, dg
__global__ void __launch_bounds__(256) cluster_intra_bwd_b_kernel(const float* __restrict__ dintra, const float* __restrict__ Qp,
                                                                  const int64_t* __restrict__ idx, const float* __restrict__ alpha,
                                                                  const float* __restrict__ da_ws, int n, int H, int Au, int D,
                                                                  int C1, float* __restrict__ dKp, float* __restrict__ dg,
                                                                  int accumulate_dg) {
  const int bh = blockIdx.x, b = bh / H, h = bh - b * H;
  const int tid = threadIdx.x;
  int c = (int)idx[bh];
  c = min(max(c, 0), C1 - 1);
  for (int a = tid; a < Au; a += 256) {
    float acc = 0.f;
    for (int k = 0; k < n; ++k) acc += da_ws[((size_t)b * n + k) * H + h] * Qp[((size_t)b * n + k) * Au + a];
    dKp[(size_t)bh * Au + a] = acc;
  }
  if ((D & 3) == 0 && dev_al16(dintra) && dev_al16(dg)) {
    const int D4 = D >> 2;
    for (int d = tid; d < D4; d += 256) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < n; ++k) {
        const float al = alpha[((size_t)b * n + k) * H + h];
        const float4 v = __ldg(reinterpret_cast<const float4*>(dintra + (((size_t)b * n + k) * C1 + c) * D) + d);
        acc.x += al * v.x; acc.y += al * v.y; acc.z += al * v.z; acc.w += al * v.w;
      }
      float4* o = reinterpret_cast<float4*>(dg + (size_t)bh * D) + d;
      if (accumulate_dg) { const float4 p = *o; acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w; }
      *o = acc;
    }
    return;
  }
  for (int d = tid; d < D; d += 256) {
    float acc = 0.f;
    for (int k = 0; k < n; ++k)
      acc += alpha[((size_t)b * n + k) * H + h] * dintra[(((size_t)b * n + k) * C1 + c) * D + d];
    float* o = dg + (size_t)bh * D + d;
    *o = accumulate_dg ? (*o + acc) : acc;
  }
}

extern "C" int nnr_cluster_intra_fwd(const float* Kp, const float* Qp, const float* g, const int64_t* idx, int B, int n, int H,
                                     int Au, int D, int C1, float scale, float* alpha, float* intra, void* stream) {
  NNR_REQUIRE(Kp && Qp && g && idx && alpha && intra && B > 0 && n > 0 && H > 0 && Au > 0 && D > 0 && C1 > 0, NNR_ERR_ARG,
              "nnr_cluster_intra_fwd: bad arguments");
  NNR_REQUIRE(H <= CI_MAXH && C1 <= CI_MAXC, NNR_ERR_UNSUPPORTED, "nnr_cluster_intra_fwd: H<=%d C1<=%d", CI_MAXH, CI_MAXC);
  cluster_intra_fwd_kernel<<<B * n, 256, 0, (cudaStream_t)stream>>>(Kp, Qp, g, idx, n, H, Au, D, C1, scale, alpha, intra);
  NNR_LAUNCH_CHECK("cluster_intra_fwd_kernel");
  return 0;
}
extern "C" int nnr_cluster_intra_bwd(const float* dintra, const float* Kp, const float* Qp, const float* g, const int64_t* idx,
                                     const float* alpha, int B, int n, int H, int Au, int D, int C1, float scale, float* da_ws,
                                     float* dKp, float* dQp, float* dg, int accumulate_dg, void* stream) {
  NNR_REQUIRE(dintra && Kp && Qp && g && idx && alpha && da_ws && dKp && dQp && dg && B > 0 && n > 0 && H > 0, NNR_ERR_ARG,
              "nnr_cluster_intra_bwd: bad arguments");
  NNR_REQUIRE(H <= CI_MAXH && C1 <= CI_MAXC, NNR_ERR_UNSUPPORTED, "nnr_cluster_intra_bwd: H<=%d C1<=%d", CI_MAXH, CI_MAXC);
  cudaStream_t st = (cudaStream_t)stream;
  cluster_intra_bwd_a_kernel<<<B * n, 256, 0, st>>>(dintra, Kp, g, idx, alpha, n, H, Au, D, C1, scale, da_ws, dQp);
  NNR_LAUNCH_CHECK("cluster_intra_bwd_a_kernel");
  cluster_intra_bwd_b_kernel<<<B * H, 256, 0, st>>>(dintra, Qp, idx, alpha, da_ws, n, H, Au, D, C1, dKp, dg, accumulate_dg);
  NNR_LAUNCH_CHECK("cluster_intra_bwd_b_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// GCN layer with layer normalisation (flag gcn_layer_norm; layers.py:286-292):
//   y = W (A X) + b  (nnr_gemm, EPI_BIAS);  n = LN(y) * gamma + beta;  r = relu(n);  out = dropout(r + res)
// forward : a warp per row, the row lives in registers (D <= 1024), biased variance like nn.LayerNorm
// backward: same mapping; a CTA's rows are accumulated per lane for dgamma / dbeta, warps combined in warp order, the
//           per-CTA partials are summed by nnr_colsum (fixed order -> deterministic)
// Dropout counter = r * D + c (regenerated in the backward), the convention of the EPI_BIAS_RELU_RES epilogue.
// ------------------------------------------------------------------------------------------------
#define LN_MAXPL 32          // columns per lane: D <= 1024
#define LN_WARPS 8
#define LN_ROWS_PER_CTA 32   // rows per CTA in the backward (4 per warp)
__global__ void __launch_bounds__(LN_WARPS * 32) ln_relu_res_fwd_kernel(const float* __restrict__ y, const float* __restrict__ gamma,
                                                                       const float* __restrict__ beta, const float* __restrict__ res,
                                                                       int R, int D, float eps, float p, float inv_keep, uint64_t seed,
                                                                       float* __restrict__ out, float* __restrict__ relu_out,
                                                                       float* __restrict__ mean, float* __restrict__ rstd) {
  const int row = blockIdx.x * LN_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= R) return;
  if (p > 0.f) seed = nnr_resolve_seed(seed);
  float v[LN_MAXPL];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < LN_MAXPL; ++j) {
    const int c = lane + 32 * j;
    v[j] = c < D ? y[(size_t)row * D + c] : 0.f;
    s += v[j];
  }
  const float mu = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < LN_MAXPL; ++j) {
    const int c = lane + 32 * j;
    const float d = c < D ? v[j] - mu : 0.f;
    q += d * d;
  }
  const float rs = rsqrtf(warp_sum(q) / (float)D + eps);
  if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
#pragma unroll
  for (int j = 0; j < LN_MAXPL; ++j) {
    const int c = lane + 32 * j;
    if (c < D) {
      const float n = (v[j] - mu) * rs * gamma[c] + beta[c];
      const float r = fmaxf(n, 0.f);
      relu_out[(size_t)row * D + c] = r;
      float o = res ? r + res[(size_t)row * D + c] : r;
      if (p > 0.f) o *= dropout_scale(seed, (uint64_t)row * (uint64_t)D + c, p, inv_keep);
      out[(size_t)row * D + c] = o;
    }
  }
}

__global__ void __launch_bounds__(LN_WARPS * 32) ln_relu_res_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ y,
                                                                       const float* __restrict__ gamma, const float* __restrict__ relu_out,
                                                                       const float* __restrict__ mean, const float* __restrict__ rstd,
                                                                       int R, int D, float p, float inv_keep, uint64_t seed,
                                                                       float* __restrict__ dout_dropped, float* __restrict__ dy,
                                                                       float* __restrict__ part_g, float* __restrict__ part_b) {
  __shared__ float s_g[LN_WARPS][32], s_b[LN_WARPS][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (p > 0.f) seed = nnr_resolve_seed(seed);
  float ag[LN_MAXPL], ab[LN_MAXPL];
#pragma unroll
  for (int j = 0; j < LN_MAXPL; ++j) { ag[j] = 0.f; ab[j] = 0.f; }
  for (int k = 0; k < LN_ROWS_PER_CTA / LN_WARPS; ++k) {
    const int row = blockIdx.x * LN_ROWS_PER_CTA + k * LN_WARPS + warp;
    if (row >= R) break;
    const float mu = mean[row], rs = rstd[row];
    float dxh[LN_MAXPL], xh[LN_MAXPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < LN_MAXPL; ++j) {
      const int c = lane + 32 * j;
      dxh[j] = 0.f; xh[j] = 0.f;
      if (c < D) {
        const size_t o = (size_t)row * D + c;
        float g = dout[o];
        if (p > 0.f) g *= dropout_scale(seed, (uint64_t)row * (uint64_t)D + c, p, inv_keep);
        if (dout_dropped) dout_dropped[o] = g;
        const float dn = relu_out[o] > 0.f ? g : 0.f;
        xh[j] = (y[o] - mu) * rs;
        dxh[j] = dn * gamma[c];
        ag[j] += dn * xh[j];
        ab[j] += dn;
        s1 += dxh[j];
        s2 += dxh[j] * xh[j];
      }
    }
    const float m1 = warp_sum(s1) / (float)D, m2 = warp_sum(s2) / (float)D;
#pragma unroll
    for (int j = 0; j < LN_MAXPL; ++j) {
      const int c = lane + 32 * j;
      if (c < D) dy[(size_t)row * D + c] = rs * (dxh[j] - m1 - xh[j] * m2);
    }
  }
  // per-CTA column partials: warps combined in warp order, 32 columns at a time
  for (int j = 0; j < LN_MAXPL; ++j) {
    if (32 * j >= D) break;
    __syncthreads();
    s_g[warp][lane] = ag[j]; s_b[warp][lane] = ab[j];
    __syncthreads();
    if (warp == 0) {
      const int c = lane + 32 * j;
      if (c < D) {
        float tg = 0.f, tb = 0.f;
#pragma unroll
        for (int w = 0; w < LN_WARPS; ++w) { tg += s_g[w][lane]; tb += s_b[w][lane]; }
        part_g[(size_t)blockIdx.x * D + c] = tg;
        part_b[(size_t)blockIdx.x * D + c] = tb;
      }
    }
  }
}

extern "C" int nnr_ln_relu_res_fwd(const float* y, const float* gamma, const float* beta, const float* res, int R, int D, float eps,
                                   float p_drop, uint64_t seed, float* out, float* relu_out, float* mean, float* rstd, void* stream) {
  NNR_REQUIRE(y && gamma && beta && out && relu_out && mean && rstd && R > 0 && D > 0, NNR_ERR_ARG, "nnr_ln_relu_res_fwd: bad arguments");
  NNR_REQUIRE(D <= 32 * LN_MAXPL, NNR_ERR_UNSUPPORTED, "nnr_ln_relu_res_fwd: D <= %d", 32 * LN_MAXPL);
  NNR_REQUIRE(p_drop >= 0.f && p_drop < 1.f, NNR_ERR_ARG, "nnr_ln_relu_res_fwd: p_drop=%f", p_drop);
  ln_relu_res_fwd_kernel<<<(R + LN_WARPS - 1) / LN_WARPS, LN_WARPS * 32, 0, (cudaStream_t)stream>>>(
      y, gamma, beta, res, R, D, eps, p_drop, 1.0f / (1.0f - p_drop), seed, out, relu_out, mean, rstd);
  NNR_LAUNCH_CHECK("ln_relu_res_fwd_kernel");
  return 0;
}

extern "C" size_t nnr_colsum_workspace_bytes(int M, int N);
extern "C" int nnr_colsum(const float* X, int64_t ldx, int M, int N, const int32_t* m_dev, float* out, int accumulate, void* workspace,
                          size_t workspace_bytes, void* stream);
static size_t ln_up256(size_t x) { return (x + 255) / 256 * 256; }
extern "C" size_t nnr_ln_relu_res_bwd_workspace_bytes(int R, int D) {
  if (R <= 0 || D <= 0) return 0;
  const int nb = (R + LN_ROWS_PER_CTA - 1) / LN_ROWS_PER_CTA;
  return 2 * ln_up256((size_t)nb * D * sizeof(float)) + ln_up256(nnr_colsum_workspace_bytes(nb, D));
}
extern "C" int nnr_ln_relu_res_bwd(const float* dout, const float* y, const float* gamma, const float* relu_out, const float* mean,
                                   const float* rstd, int R, int D, float p_drop, uint64_t seed, float* dout_dropped, float* dy,
                                   float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, void* stream) {
  NNR_REQUIRE(dout && y && gamma && relu_out && mean && rstd && dy && dgamma && dbeta && workspace && R > 0 && D > 0, NNR_ERR_ARG,
              "nnr_ln_relu_res_bwd: bad arguments");
  NNR_REQUIRE(D <= 32 * LN_MAXPL, NNR_ERR_UNSUPPORTED, "nnr_ln_relu_res_bwd: D <= %d", 32 * LN_MAXPL);
  NNR_REQUIRE(p_drop >= 0.f && p_drop < 1.f, NNR_ERR_ARG, "nnr_ln_relu_res_bwd: p_drop=%f", p_drop);
  NNR_REQUIRE(workspace_bytes >= nnr_ln_relu_res_bwd_workspace_bytes(R, D), NNR_ERR_WORKSPACE, "nnr_ln_relu_res_bwd: workspace too small");
  NNR_REQUIRE(dout_dropped != dout, NNR_ERR_ARG, "nnr_ln_relu_res_bwd: dout_dropped must not alias dout");
  const int nb = (R + LN_ROWS_PER_CTA - 1) / LN_ROWS_PER_CTA;
  char* ws = (char*)workspace;
  float* pg = (float*)ws;
  float* pb = (float*)(ws + ln_up256((size_t)nb * D * sizeof(float)));
  void* cws = ws + 2 * ln_up256((size_t)nb * D * sizeof(float));
  const size_t cws_bytes = ln_up256(nnr_colsum_workspace_bytes(nb, D));
  ln_relu_res_bwd_kernel<<<nb, LN_WARPS * 32, 0, (cudaStream_t)stream>>>(dout, y, gamma, relu_out, mean, rstd, R, D, p_drop,
                                                                        1.0f / (1.0f - p_drop), seed, dout_dropped, dy, pg, pb);
  NNR_LAUNCH_CHECK("ln_relu_res_bwd_kernel");
  int rc = nnr_colsum(pg, D, nb, D, nullptr, dgamma, 0, cws, cws_bytes, stream);
  if (rc) return rc;
  return nnr_colsum(pb, D, nb, D, nullptr, dbeta, 0, cws, cws_bytes, stream);
}
