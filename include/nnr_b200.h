/* nnr_b200 -- C ABI of the B200-native CNE+SUE hot path.
 *
 * Every entry point is a plain `extern "C"` function over raw DEVICE pointers, sizes and a
 * `cudaStream_t` (passed as void*).  No torch types cross this boundary.  The reference
 * (Veason-silverbullet/NNR) is pure PyTorch, so what each function replaces is a span of
 * library calls in the reference's Python; the span is cited as file:line next to each entry.
 *
 * Conventions (SURVEY.md section 8b)
 *   - return 0 on success, a negative NNR_ERR_* on argument / alignment / workspace errors, a
 *     positive cudaError_t when a launch fails; `nnr_last_error()` returns a thread-local message.
 *   - the caller owns every buffer (inputs, outputs, stashes, workspaces); the library never
 *     allocates, frees or retains a pointer beyond the call; outputs are fully overwritten
 *     unless the argument is called `accumulate`.
 *   - launches go only to the passed stream; entry points are re-entrant.
 *   - fp32 everywhere unless the name says otherwise; token ids int32; masks uint8 (torch.bool).
 *   - dropout `seed` arguments: a value below 2^62 is the seed itself.  With bit 62 set (NNR_SEED_INDIRECT) the seed is
 *     indirect: bits 0..47 = device address of a uint64 base the caller advances on the device between steps, bits
 *     48..61 = a site id; the kernels use hash(base + site).  This is what lets a whole training step be captured in a
 *     CUDA graph and replayed with fresh masks (kernel arguments are frozen at capture).
 *
 * Token layout.  A CNE call sees N news rows with up to L tokens each.  `nnr_seq_prepare` turns
 * the [N,L] prefix mask into len[N], off[N+1] (exclusive prefix sum) and tok_row[N*L]; every
 * per-token tensor is then PACKED: the token t of row r lives at row off[r]+t of a
 * [N*L (capacity), dim] matrix, and off[N] is the number of valid tokens (read on the device, so
 * no host synchronisation is needed).
 */
#ifndef NNR_B200_H
#define NNR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNR_ABI_VERSION 11
#define NNR_SEED_INDIRECT (1ULL << 62)

const char* nnr_last_error(void);
int nnr_abi_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t nnr_launch_count(void);
/* kernel-level timing of the kernels inside the composite nnr_gemm op (CUDA events on the launching stream).
 * tags: 0 gemm_tc_kernel, 1 tc_split_kernel, 2 tc_splitk_reduce_kernel, 3 gemm_simt_kernel.
 * nnr_profile_read synchronises the device, fills out[3*tag + {0: ms, 1: launches, 2: reserved}] and clears the log. */
int nnr_profile_enable(int on);
int nnr_profile_read(double* out, int ntags);

/* ---- sequence bookkeeping: newsEncoders.py:106-111 (mask[:,0]=1 in place, lengths) ---------- */
int nnr_seq_prepare(uint8_t* mask, int N, int L, int32_t* len, int32_t* off, int32_t* tok_row,
                    void* stream);

/* ---- word-embedding gather + dropout: newsEncoders.py:117-118 (nn.Embedding + nn.Dropout) ---
 * out[off[r]+t, :] = table[ids[r,t], :] * keep(seed, (r*L+t)*E+e) / (1-p)                       */
int nnr_embed_gather_fwd(const float* table, const int32_t* ids, const int32_t* len,
                         const int32_t* off, int N, int L, int E, int V, float* out, float p_drop,
                         uint64_t seed, void* stream);
/* the same gather + dropout written directly as operand planes of the tensor-core GEMM (layout of nnr_tc_split for a
 * [cap, E] matrix, rows [ntok, round_up(ntok, 64)) zeroed): bit-identical to nnr_embed_gather_fwd followed by
 * nnr_tc_split.  The consumer passes A = NULL / B = NULL with A_planes / B_planes to nnr_gemm.  E % 4 == 0.   */
int nnr_embed_gather_planes_fwd(const float* table, const int32_t* ids, const int32_t* len,
                                const int32_t* off, int N, int L, int E, int V, int cap, float p_drop,
                                uint64_t seed, int algo, void* planes, size_t planes_bytes, void* stream);
/* autograd of the above (ATen embedding_dense_backward): deterministic sort-by-id + segment
 * reduce into the dense [V,E] table gradient.  `dout` is packed [tokens,E].                      */
size_t nnr_embed_gather_bwd_workspace_bytes(int N, int L);
int nnr_embed_gather_bwd(const float* dout, const int32_t* ids, const int32_t* len,
                         const int32_t* off, int N, int L, int E, int V, float p_drop,
                         uint64_t seed, float* dtable, int accumulate, void* workspace,
                         size_t workspace_bytes, void* stream);

/* ---- GEMM with fused epilogues: every nn.Linear on the path (newsEncoders.py:122-129,
 *      layers.py:168,197,286; userEncoders.py:85-86,91) and their autograd ----------------------
 * C[M,N] = epi( op(A)[M,K] * op(B)[K,N] ),  op(A)[m,k] = transA ? A[k*lda+m] : A[m*lda+k],
 *                                           op(B)[k,n] = transB ? B[n*ldb+k] : B[k*ldb+n].       */
enum {
  NNR_EPI_NONE = 0,          /* C = acc                                                         */
  NNR_EPI_BIAS = 1,          /* C = acc + bias[n]                                               */
  NNR_EPI_BIAS_TANH = 2,     /* C = tanh(acc + bias[n])                                         */
  NNR_EPI_BIAS_RELU_RES = 3, /* r = relu(acc+bias[n]); aux_out = r; C = (r + aux[m,n]) * drop   */
  NNR_EPI_GATE = 4,          /* g = sigmoid(acc + rowbias[rowmap[m], n]); aux_out = g; C = aux*g */
  NNR_EPI_ADD_AUX = 5        /* C = acc + aux[m,n]                                              */
};
enum {
  NNR_GEMM_AUTO = 0,
  NNR_GEMM_SIMT_FP32 = 1,    /* exact fp32 FFMA tiles                                           */
  NNR_GEMM_TC_TF32X3 = 2,    /* tcgen05 kind::tf32, hi/lo split (3 MMAs), fp32-grade accuracy   */
  NNR_GEMM_TC_BF16 = 3,      /* tcgen05 kind::f16 bf16 operands, fp32 accumulate                */
  NNR_GEMM_TC_BF16X3 = 4     /* tcgen05 kind::f16, bf16 hi/lo split (3 MMAs): ~2^-17 operand error, half the bytes */
};
typedef struct {
  const float* A; int64_t lda; int32_t transA;
  const float* B; int64_t ldb; int32_t transB;
  float* C; int64_t ldc;
  int32_t M, N, K;
  const int32_t* m_dev;      /* optional device scalar: rows >= *m_dev are skipped             */
  const int32_t* k_dev;      /* optional device scalar: contraction stops at *k_dev            */
  int32_t epilogue;
  int32_t accumulate;        /* C += epi(...) instead of C = epi(...)                          */
  const float* bias;
  const float* aux; int64_t ldaux;
  float* aux_out; int64_t ldaux_out;
  const float* rowbias; int64_t ldrowbias; const int32_t* rowmap;
  float p_drop; uint64_t seed;
  int32_t algo;
  void* workspace; size_t workspace_bytes;   /* operand planes + split-K partials (see nnr_gemm_workspace_bytes) */
  /* optional: operands already split by nnr_tc_split (tensor-core backend only; A / B may then be NULL --
   * an operand that exists only as planes makes nnr_gemm fail if the exact-fp32 kernel would have to run).
   * X_planes points at the first plane of the (possibly column-sliced) stored matrix, pitch in elements,
   * plane_rows = rows of the full planes (plane stride = plane_rows * pitch). */
  const void* A_planes; int64_t a_planes_pitch; int64_t a_planes_rows;
  const void* B_planes; int64_t b_planes_pitch; int64_t b_planes_rows;
  /* optional (bf16 tensor-core algos, N % 8 == 0, epilogue operands 16-byte aligned, no split-K): the result is ALSO written
   * as the operand planes nnr_tc_split(C, ..., m_dev) would produce -- [hi|lo][c_planes_rows][pitch] bf16, rows
   * [M_eff, round_up(M_eff, 64)) zero-filled -- so that a GEMM whose output feeds further GEMMs needs no split pass
   * (newsEncoders.py:128-131: the gated states feed the attention projections).  NNR_ERR_UNSUPPORTED otherwise. */
  void* C_planes; int64_t c_planes_pitch; int64_t c_planes_rows;
} nnr_gemm_args;
size_t nnr_gemm_workspace_bytes(const nnr_gemm_args* args);
int nnr_gemm(const nnr_gemm_args* args, void* stream);
/* Split a row-major fp32 matrix X[R,C] (ld) into the operand planes of the tensor-core backend so that several
 * GEMMs can share them: 3xTF32 -> fp32 [hi|lo][R][pitch], BF16 -> bf16 [1][R][pitch]; pitch = C rounded up to 16
 * bytes.  With r_dev, rows [*r_dev, round_up(*r_dev, 64)) are zero-filled (contraction tail) and later rows
 * are left untouched.  algo = NNR_GEMM_TC_TF32X3 or NNR_GEMM_TC_BF16 (NNR_GEMM_AUTO = the library default). */
int64_t nnr_tc_split_pitch(int C, int algo);
size_t nnr_tc_split_bytes(int R, int C, int algo);
int nnr_tc_split(const float* X, int64_t ld, int R, int C, const int32_t* r_dev, int algo, void* planes,
                 size_t planes_bytes, void* stream);
/* nnr_tc_split of many matrices in ONE launch (e.g. every weight matrix right after the optimizer step).
 * `descs` is a DEVICE array of n descriptors; planes = [hi|lo][rows][pitch] with pitch = nnr_tc_split_pitch(cols). */
typedef struct nnr_split_desc {
  const float* src; int64_t ld; int32_t rows, cols;
  void* planes; int64_t pitch;
} nnr_split_desc;
int nnr_tc_split_many(const nnr_split_desc* descs, int n, int algo, void* stream);

/* Stable descending sort of small integer keys (the sequence lengths of newsEncoders.py:112,114):
 * sorted_idx[rank] = original index, ties in ascending original index (= torch.sort on CUDA).  N <= 8192,
 * 0 <= key <= max_key <= 1024 (keys are clamped). */
int nnr_length_sort_desc(const int64_t* keys, int N, int max_key, int64_t* sorted_idx, void* stream);

/* nnr_tc_split plus the column sums of X (rows < *r_dev) in the same pass: a bias gradient (trainer-side
 * `dy.sum(0)`, i.e. the bias part of every nn.Linear / nn.LSTM backward) is the column sum of the dL/dy whose planes feed
 * the dgrad / wgrad GEMMs.  Deterministic (fixed partial order).  colsum[C] is overwritten, or added to if accumulate. */
size_t nnr_tc_split_colsum_workspace_bytes(int R, int C, int algo);
int nnr_tc_split_colsum(const float* X, int64_t ld, int R, int C, const int32_t* r_dev, int algo, void* planes,
                        size_t planes_bytes, float* colsum, int accumulate, void* workspace, size_t workspace_bytes,
                        void* stream);
/* Backward of "dropout -> relu -> Linear" (GCN layer layers.py:286-289, cluster affine userEncoders.py:91) in the same
 * pass: x = dy * keep(seed, r*C + c)/(1-p) (the mask of nnr_dropout; x is also stored to dy_dropped when given -- it
 * feeds the residual branch; must not alias dy), z = x * (relu_out > 0); planes(z) and colsum[c] = sum_r z[r,c].
 * Bit-identical to nnr_dropout + the elementwise product + nnr_tc_split_colsum.                                  */
int nnr_relu_bwd_split_colsum(const float* dy, const float* relu_out, int64_t ld, int R, int C, float p_drop,
                              uint64_t seed, float* dy_dropped, int algo, void* planes, size_t planes_bytes,
                              float* colsum, int accumulate, void* workspace, size_t workspace_bytes,
                              void* stream);
/* the algorithm NNR_GEMM_AUTO resolves to (env NNR_GEMM_ALGO = simt | tf32x3 | bf16 | bf16x3; default bf16x3) */
int nnr_gemm_default_algo(void);

/* column sums: out[n] (+)= sum_m X[m,n]   (bias gradients; deterministic two-stage)            */
size_t nnr_colsum_workspace_bytes(int M, int N);
int nnr_colsum(const float* X, int64_t ldx, int M, int N, const int32_t* m_dev, float* out,
               int accumulate, void* workspace, size_t workspace_bytes, void* stream);
/* per-row (segment) column sums over packed tokens: out[r,:] = sum_t X[off[r]+t,:]              */
int nnr_segment_colsum(const float* X, int64_t ldx, const int32_t* off, int N, int D, float* out,
                       int64_t ldo, void* stream);

/* ---- bidirectional LSTM recurrence: nn.LSTM at newsEncoders.py:66-67,122-127 ----------------
 * Persistent thread-block-cluster kernel; W_hh stays on chip for all time steps.
 * Hidden sizes: 0 < H <= 200 with H % 4 == 0 (tensor-core kernels, clusters of max(2, ceil(H / 40)) CTAs); the exact-fp32
 * FFMA kernels (NNR_LSTM_ALGO=ffma) take H = 200 only.  Any other H returns NNR_ERR_UNSUPPORTED before a CUDA call, with the
 * rule in nnr_last_error().
 *   gx      [tokens, 2, 4H]  in: x_t W_ih^T + b_ih + b_hh (gate order i,f,g,o per direction)
 *                            out: the activated gates (stash for the backward pass)
 *   w_hh    [2, 4H, H]       forward / reverse recurrent weights
 *   order   [N]              rows sorted by length, longest first (tile homogeneity only)
 *   h_out   [tokens, 2H]     h_t, forward | reverse
 *   c_stash [tokens, 2, H]   c_t for the backward pass
 *   c_n     [N, 2H]          final cell state per row (forward | reverse)  (newsEncoders.py:124)
 *   tile_counters [2] int32  scratch for the dynamic (longest-tile-first) scheduler; zeroed by the call */
int nnr_lstm_fwd(float* gx, const float* w_hh, const int32_t* len, const int32_t* off,
                 const int32_t* order, int N, int L, int H, float* h_out, float* c_stash,
                 float* c_n, int32_t* tile_counters, void* stream);
/* BPTT.  gates (the stash written by nnr_lstm_fwd) is overwritten IN PLACE with dL/d(pre-
 * activation) = dL/d(gx).  dh [tokens,2H] and dcn [N,2H] are the upstream gradients.            */
int nnr_lstm_bwd(float* gates, const float* c_stash, const float* w_hh, const int32_t* len,
                 const int32_t* off, const int32_t* order, int N, int L, int H, const float* dh,
                 const float* dcn, int32_t* tile_counters, void* stream);
/* nnr_lstm_fwd whose h ALSO leaves as the operand planes nnr_tc_split(h, cap, 2H, ntok) would produce ([hi|lo][cap][2H] bf16,
 * rows [tokens, round_up(tokens, 64)) zeroed): h feeds the selective-gate GEMM and two weight-gradient GEMMs
 * (newsEncoders.py:128-131), the split pass over it is skipped.  bf16 tensor-core algos, H = 200. */
int nnr_lstm_fwd_planes_supported(int H, int algo);
int nnr_lstm_fwd_planes(float* gx, const float* w_hh, const int32_t* len, const int32_t* off, const int32_t* order,
                        int N, int L, int H, float* h_out, float* c_stash, float* c_n, int32_t* tile_counters, int cap,
                        int algo, void* planes, size_t planes_bytes, void* stream);
/* The same BPTT with dL/d(gx) written as the operand planes of the tensor-core GEMM (layout of nnr_tc_split for a
 * [cap, 8H] matrix, rows [tokens, round_up(tokens, 64)) zeroed) and db[8H] = its column sums over the tokens (the bias
 * gradient; per-tile partials added in tile order, run-to-run identical).  dL/d(gx) feeds only GEMMs and that column
 * sum, so the fp32 tensor is never written; `gates` is left untouched.  Bit-identical to nnr_lstm_bwd followed by
 * nnr_tc_split (planes); db differs from nnr_colsum only by fp32 summation order.
 * nnr_lstm_bwd_planes_supported: H == 200, tensor-core recurrence (NNR_LSTM_ALGO != ffma), algo BF16 / BF16X3.        */
int nnr_lstm_bwd_planes_supported(int H, int algo);
size_t nnr_lstm_bwd_planes_workspace_bytes(int N, int H);
int nnr_lstm_bwd_planes(const float* gates, const float* c_stash, const float* w_hh, const int32_t* len,
                        const int32_t* off, const int32_t* order, int N, int L, int H, const float* dh,
                        const float* dcn, int32_t* tile_counters, int cap, int algo, void* dz_planes,
                        size_t planes_bytes, float* db, void* workspace, size_t workspace_bytes, void* stream);
/* hprev[p, 0:H] = h[p-1, 0:H] (0 at t=0); hprev[p, H:2H] = h[p+1, H:2H] (0 at t=len-1): the
 * recurrent input of every step, needed for dW_hh = dgates^T hprev.                             */
int nnr_lstm_shift_h(const float* h, const int32_t* len, const int32_t* off,
                     const int32_t* tok_row, int N, int L, int H, float* hprev, void* stream);
/* the same shifted states written directly as operand planes ([cap, 2H] layout of nnr_tc_split, zeroed row tail):
 * bit-identical to nnr_lstm_shift_h followed by nnr_tc_split; hprev is only the B operand of dW_hh = dgates^T hprev. */
int nnr_lstm_shift_h_planes(const float* h, const int32_t* len, const int32_t* off,
                            const int32_t* tok_row, int N, int L, int H, int cap, int algo, void* planes,
                            size_t planes_bytes, void* stream);
/* dz = dhg*h*g*(1-g), dh0 = dhg*g : elementwise part of the selective-gate backward
 * (newsEncoders.py:128-131)                                                                     */
int nnr_gate_bwd_pre(const float* dhg, const float* h, const float* g, int64_t n_max,
                     const int32_t* n_dev, int D, float* dz, float* dh0, void* stream);
/* nnr_gate_bwd_pre + nnr_tc_split(dz) + nnr_segment_colsum(dz) in one pass: dz leaves as operand planes ([cap, D] layout
 * of nnr_tc_split, zeroed row tail), dmproj[r, :] = sum of dz over the tokens of news r (token order), dh0 stays fp32.
 * Bit-identical to the three separate calls.                                                                      */
int nnr_gate_bwd_planes(const float* dhg, const float* h, const float* g, const int32_t* off, int N, int D,
                        int cap, int algo, void* dz_planes, size_t planes_bytes, float* dh0, float* dmproj,
                        int64_t lddm, void* stream);

/* ---- fused masked attention pooling over segments: layers.py:167-175 and :196-203 -----------
 * Segment s covers rows [seg_off[s], seg_off[s+1]) of X (or s*fixed_len.. when seg_off == NULL).
 *   mode 0 (additive):    score[p] = dot(U[p,:A], w2)            U = tanh(W1 x + b1) precomputed
 *   mode 1 (scaled dot):  score[p] = scale * dot(X[p,:], qvec[s,:])   qvec = K^T (Q q + b) folded
 * mask (optional, per row of X): 0 -> score = -1e9.  Outputs pooled[S,D], alpha[rows].          */
typedef struct {
  const float* X; int64_t ldx; int32_t D;
  const int32_t* seg_off; int32_t S; int32_t fixed_len; int32_t max_len;
  int32_t mode;
  const float* U; int64_t ldu; int32_t A; const float* w2;
  const float* qvec; int64_t ldq; float scale;
  const uint8_t* mask;
  float* pooled; int64_t ldp;
  float* alpha;
  /* backward only */
  const float* dpooled; int64_t lddp;
  float* dX; int64_t lddx; int32_t accumulate_dx;
  float* dU; int64_t lddu;        /* mode 0: dL/d(pre-tanh) = da * w2 * (1 - U^2)               */
  float* dw2_partial;             /* mode 0: [S, A] per-segment partials (reduce with colsum)   */
  float* dqvec; int64_t lddq;     /* mode 1: [S, D]                                              */
  const int32_t* seg_order;       /* optional [S]: block b processes segment seg_order[b] (e.g. longest first, so the
                                     long segments do not form the tail of the launch); NULL = identity          */
} nnr_pool_args;
int nnr_attn_pool_fwd(const nnr_pool_args* args, void* stream);
int nnr_attn_pool_bwd(const nnr_pool_args* args, void* stream);

/* ---- news vector assembly: newsEncoders.py:50-54,138 ----------------------------------------
 * out[r] = [ts+tc | cs+cc | drop(cat_table[cat[r]]) | drop(sub_table[sub[r]])]                  */
/* c_self = NULL (fwd) / d_b = NULL (bwd): single-modality encoders, layout [self | category | subCategory]
 * (variantEncoders.py:14-99). */
int nnr_news_fuse_fwd(const float* t_self, const float* t_cross, const float* c_self,
                      const float* c_cross, const float* cat_table, const float* sub_table,
                      const int32_t* cat, const int32_t* sub, int N, int D2, int Ec, int Es,
                      float p_drop, uint64_t seed, float* out, void* stream);
/* backward: d_a[N,D2] = dout[:, :D2], d_b[N,D2] = dout[:, D2:2*D2]; dense table grads
 * (deterministic: one block per table row scanning the N rows in order).  dcat_table == dsub_table == NULL: only the
 * activation split; the table gradients -- leaves of the backward pass -- can then be taken by
 * nnr_news_fuse_tables_bwd on another stream (col0 = first category column of dout = 2*D2, or D2 for one modality). */
int nnr_news_fuse_bwd(const float* dout, const int32_t* cat, const int32_t* sub, int N, int D2,
                      int Ec, int Es, int n_cat, int n_sub, float p_drop, uint64_t seed,
                      float* d_a, float* d_b, float* dcat_table, float* dsub_table,
                      int accumulate, void* stream);
int nnr_news_fuse_tables_bwd(const float* dout, const int32_t* cat, const int32_t* sub, int N, int Dout, int col0,
                             int Ec, int Es, int n_cat, int n_sub, float p_drop, uint64_t seed,
                             float* dcat_table, float* dsub_table, int accumulate, void* stream);

/* ---- SUE graph: MIND_corpus.py:162-216 (structure), layers.py:286 (aggregation) --------------
 * Build graph / mask / cluster indices on the device from per-slot categories (bit-exact with
 * the reference's numpy: fp32 1/deg, sqrt, two roundings).  Any output pointer may be NULL.     */
int nnr_sue_graph_build(const int32_t* categories, const int32_t* history_len, int B, int H,
                        int C, float* graph, uint8_t* category_mask, int64_t* category_indices,
                        void* stream);
/* the same with the reference's graph flags (config.py:56-58, MIND_corpus.py:179-182,203-213); a bit set = flag on.
 * no_self_connection without no_adjacent_normalization is rejected like config.py:111 does.     */
enum {
  NNR_GRAPH_NO_SELF_CONNECTION = 1, /* adjacency starts from zeros instead of the identity       */
  NNR_GRAPH_NO_NORMALIZATION = 2,   /* keep the 0/1 adjacency                                     */
  NNR_GRAPH_ASYMMETRIC = 4          /* D^-1 A instead of D^-1/2 A D^-1/2                          */
};
int nnr_sue_graph_build_ex(const int32_t* categories, const int32_t* history_len, int B, int H,
                           int C, int flags, float* graph, uint8_t* category_mask,
                           int64_t* category_indices, void* stream);
/* GCN layer with layer normalisation (flag gcn_layer_norm, layers.py:286-292).  y [R,D] is the output of
 * nnr_gemm(EPI_BIAS) = W (A X) + b.  forward: n = LayerNorm(y) * gamma + beta (biased variance, eps), r = relu(n)
 * -> relu_out, out = dropout(r + res) (res may be NULL; dropout counter = row * D + col), mean / rstd [R] are the
 * backward stash.  backward: dout_dropped (optional) = dout * mask (the residual branch's gradient),
 * dy = dL/dy, dgamma / dbeta [D] (deterministic).  D <= 1024.                                   */
int nnr_ln_relu_res_fwd(const float* y, const float* gamma, const float* beta, const float* res,
                        int R, int D, float eps, float p_drop, uint64_t seed, float* out,
                        float* relu_out, float* mean, float* rstd, void* stream);
size_t nnr_ln_relu_res_bwd_workspace_bytes(int R, int D);
int nnr_ln_relu_res_bwd(const float* dout, const float* y, const float* gamma, const float* relu_out,
                        const float* mean, const float* rstd, int R, int D, float p_drop,
                        uint64_t seed, float* dout_dropped, float* dy, float* dgamma, float* dbeta,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Dense (caller-supplied) graph -> per-row compressed neighbour lists (row-compressed with a fixed
 * row capacity of G entries).  transpose=1 emits the lists of A^T (for the backward pass).
 * nnz [B*G], col/val [B*G, G]; entries of a row are in ascending column order.                  */
int nnr_graph_to_csr(const float* graph, int B, int G, int transpose, int32_t* nnz, int32_t* col,
                     float* val, void* stream);
/* out[b,i,:] = sum_{e < nnz[b,i]} val[b,i,e] * x[b,col[b,i,e],:]   (fixed order: deterministic) */
int nnr_gcn_aggregate(const int32_t* nnz, const int32_t* col, const float* val, const float* x,
                      int B, int G, int D, float* out, void* stream);
/* out = A x + add: the aggregation of the GCN backward with its residual term in the same pass (add != out) */
int nnr_gcn_aggregate_add(const int32_t* nnz, const int32_t* col, const float* val, const float* x, int B,
                          int G, int D, const float* add, float* out, void* stream);

/* ---- intra-cluster attention: userEncoders.py:85-89 (torch_scatter softmax + sum) -----------
 *   Kp [B,H,Au], Qp [B,n,Au], g [B,H,D], idx [B,H] int64 in [0,C1)
 *   alpha[b,k,h] = segment_softmax_h( Kp[b,h].Qp[b,k] * scale ; idx[b,h] )
 *   intra[b,k,c,:] = sum_{h: idx=c} alpha[b,k,h] g[b,h,:]   (ascending h: deterministic)        */
int nnr_cluster_intra_fwd(const float* Kp, const float* Qp, const float* g, const int64_t* idx,
                          int B, int n, int H, int Au, int D, int C1, float scale, float* alpha,
                          float* intra, void* stream);
int nnr_cluster_intra_bwd(const float* dintra, const float* Kp, const float* Qp, const float* g,
                          const int64_t* idx, const float* alpha, int B, int n, int H, int Au,
                          int D, int C1, float scale, float* da_ws /* [B,n,H] scratch */,
                          float* dKp, float* dQp, float* dg, int accumulate_dg, void* stream);
/* Factored cluster tail for top-k recommendation: click scores of T pool candidates, shared by the B users, without the
 * per-(user, candidate) cluster features.  The weights of a non-empty cluster's softmax sum to 1 and an empty cluster's
 * feature is 0, so the cluster affine commutes with the weighted sum (W intra_c + b = sum_{h in c} alpha_h Wg_h + b):
 *   Kp [B,H,Au] (intra-cluster keys), g [B,H,D], Wg [B,H,D] = g W^T (clusterFeatureAffine.weight, no bias), idx [B,H]
 *   int64 (clamped to [0,C1)), cmask [B,C1] uint8, Qp [T,Au], qk2 [T,D], cand [T,D] (one row per candidate), bias [D]
 *   alpha[b,t,h] = segment_softmax_h(scale * Kp[b,h].Qp[t] ; idx[b,h])   (every slot takes part, max-shifted)
 *   f[b,t,c,:]   = relu(sum_{h: idx=c} alpha Wg[b,h] + bias) + sum_{h: idx=c} alpha g[b,h]   (empty cluster: relu(bias))
 *   beta[b,t,c]  = softmax_c(cmask[b,c] ? scale * f.qk2[t] : -1e9)
 *   scores[b*lds + t] = sum_c beta * (f . cand[t])
 * = cluster_intra_fwd + the EPI_BIAS_RELU_RES affine + attn_pool mode 1 + rowdot in real arithmetic, not bit for bit.
 * Deterministic (fixed summation order, no atomics), no allocation, no host synchronisation (graph-capturable).
 * Limits: H <= 256, C1 <= 72, 1 <= T <= NNR_TOPK_MAX_TILE, lds >= T (NNR_ERR_ARG / NNR_ERR_UNSUPPORTED before any CUDA
 * call otherwise); D % 4 == 0 and 16-byte aligned g, Wg, qk2, cand, bias (NNR_ERR_UNSUPPORTED).                       */
int nnr_cluster_tail_scores(const float* Kp, const float* g, const float* Wg, const int64_t* idx, const uint8_t* cmask,
                            const float* Qp, const float* qk2, const float* cand, const float* bias, int B, int H, int Au,
                            int D, int C1, int T, float scale, float* scores, int64_t lds, void* stream);
/* The same factored tail for per-user candidate lists stored back to back (dev/test evaluation;
 * scoring.CorpusScorer.evaluate(exact=False)): user b's candidates are rows [row_off[b], row_off[b+1]) of Qp [rows,Au],
 * qk2 [rows,D] and cand [rows,D]; the score of its j-th candidate goes to scores[b*lds + j], and entries j >= its count
 * are not written.  Kp, g, Wg, idx, cmask and bias are as above.  Given the same rows, every score equals
 * nnr_cluster_tail_scores' bit for bit (one shared per-candidate code path).  The work follows the sum of the counts, not
 * B * n_max: a CTA holds a slice of one user's list, and a slice past the count exits at once.
 * row_off [B+1] int32 lives on the device and is not checked by the host: each count is clamped to [0, n_max] and each
 * row to [0, rows), so bad offsets read and write nothing out of bounds.
 * Deterministic (no atomics), no allocation, no host synchronisation (graph-capturable).
 * Limits: B >= 0, 1 <= n_max <= lds, 0 <= rows < 2^31, H <= 256, C1 <= 72 (NNR_ERR_ARG / NNR_ERR_UNSUPPORTED before any
 * CUDA call otherwise); D % 4 == 0 and 16-byte aligned g, Wg, qk2, cand, bias (NNR_ERR_UNSUPPORTED).                  */
int nnr_cluster_tail_scores_packed(const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                                   const uint8_t* cmask, const int32_t* row_off, int64_t rows, const float* Qp,
                                   const float* qk2, const float* cand, const float* bias, int B, int H, int Au, int D,
                                   int C1, int n_max, float scale, float* scores, int64_t lds, void* stream);
/* nnr_cluster_tail_scores_packed that also explains every score it writes (scoring.CorpusScorer.explain(exact=False)):
 * for user b's j-th candidate (t = b*lds + j, j below its count)
 *   alpha_out[t*H + h]     = alpha[b,j,h], slot h's weight in its cluster's softmax (history order; sums to 1 over the
 *                            slots of each non-empty cluster)
 *   beta_out[t*C1 + c]     = beta[b,j,c] (exactly 0 for a masked cluster)
 *   contrib_out[t*C1 + c]  = beta[b,j,c] * (f[b,j,c,:] . cand), whose sum over c is the score up to fp32 rounding
 * The scores are those of nnr_cluster_tail_scores_packed on the same arguments, bit for bit.  Entries past a user's
 * count are not written, in any of the four outputs.  The arguments, checks, error codes and limits are those of
 * nnr_cluster_tail_scores_packed; alpha_out, beta_out and contrib_out must not be NULL either (NNR_ERR_ARG).         */
int nnr_cluster_tail_explain_packed(const float* Kp, const float* g, const float* Wg, const int64_t* idx,
                                    const uint8_t* cmask, const int32_t* row_off, int64_t rows, const float* Qp,
                                    const float* qk2, const float* cand, const float* bias, int B, int H, int Au, int D,
                                    int C1, int n_max, float scale, float* scores, int64_t lds, float* alpha_out,
                                    float* beta_out, float* contrib_out, void* stream);

/* ---- click predictor: model.py:127 ---------------------------------------------------------- */
int nnr_rowdot_fwd(const float* a, const float* b, int R, int D, float* out, void* stream);
/* da = dout[r]*b (+= if accumulate_a), db likewise */
int nnr_rowdot_bwd(const float* dout, const float* a, const float* b, int R, int D, float* da,
                   int accumulate_a, float* db, int accumulate_b, void* stream);

/* ---- streaming top-k over a candidate pool (news recommendation; scoring.CorpusScorer.recommend) ----------------
 * Merges one score tile scores[B, T] (row stride lds) into a running per-row best list best_score[B, k] (fp32) /
 * best_pos[B, k] (int64 pool positions), in place.  Tile entry j of row b has pool position pos0 + j.
 * Order: score descending; equal scores by ascending position (= a stable descending sort of the whole row); a NaN
 * ranks below every number, -inf included.  Entries whose news id tile_ids[j] is among exclude[b, 0:exclude_len[b]]
 * (exclude [B, ldx] int64, lengths clamped to [0, ldx]) are skipped; exclude = NULL skips nothing (tile_ids may then be
 * NULL).  The list is left sorted best first; slots no candidate has reached hold the fill entry (-inf, -1), which
 * every real entry, -inf or NaN, ranks before.  init != 0 ignores the list's previous content (the first tile of a
 * pool); otherwise the list must be as a previous call left it.
 * Entries that do not beat the current k-th best are dropped before anything is sorted.  Deterministic, no host
 * synchronisation, no allocation (graph-capturable).  Limits: 1 <= k <= NNR_TOPK_MAX_K, 1 <= T <= NNR_TOPK_MAX_TILE,
 * ldx <= NNR_TOPK_MAX_EXCLUDE, 0 <= pos0 and pos0 + T < 2^31 - 1; NNR_ERR_ARG before any CUDA call otherwise.       */
#define NNR_TOPK_MAX_K 1024
#define NNR_TOPK_MAX_TILE 4096
#define NNR_TOPK_MAX_EXCLUDE 1024
int nnr_topk_merge(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                   const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init,
                   float* best_score, int64_t* best_pos, void* stream);
/* The same merge with at most `cap` entries per group (a news category): tile entry j belongs to group
 * id_group[tile_ids[j]] (id_group: int32 per news id, values in [0, num_groups); an entry of another group is never kept),
 * and best_group[B, k] (int32) holds each list entry's group next to best_score / best_pos (-1 for the fill).  The list is
 * the first k entries of the eligible entries seen so far, taken in the order above, each taken unless `cap` entries of its
 * group were already taken; the fill entry counts toward nothing.  With cap >= k the result equals nnr_topk_merge's.
 * Rejects, besides what nnr_topk_merge rejects: cap < 1, num_groups outside [1, NNR_TOPK_MAX_GROUPS], NULL id_group,
 * best_group or tile_ids.                                                                                             */
#define NNR_TOPK_MAX_GROUPS 1024
int nnr_topk_merge_capped(const float* scores, int64_t lds, int B, int T, int64_t pos0, const int64_t* tile_ids,
                          const int64_t* exclude, const int32_t* exclude_len, int ldx, int k, int init,
                          const int32_t* id_group, int num_groups, int cap, float* best_score, int64_t* best_pos,
                          int32_t* best_group, void* stream);
/* The same merges of entries that carry their own pool positions: entry j of row b has score scores[b*lds + j] and
 * position pos[b*ldp + j] (int64), and in the capped variant group grp[b*ldg + j] (int32), instead of pos0 + j and
 * id_group[tile_ids[j]].  A negative position is an empty slot (the fill entry of a best list) and is dropped before
 * anything else; a real entry scoring -inf is kept.  No exclusion list.  Used to fold the per-rank best lists of a
 * data-parallel CorpusScorer.recommend() into one: positions of different calls' entries must be distinct (keys are
 * unique), and must be < 2^31 - 1.  Order, state, determinism and limits are those of nnr_topk_merge[_capped]; a best
 * list of k entries fits T = k.  Rejects, besides what nnr_topk_merge[_capped] rejects: NULL pos, ldp < T, and in the
 * capped variant NULL grp or best_group and ldg < T.                                                                 */
int nnr_topk_merge_lists(const float* scores, int64_t lds, int B, int T, const int64_t* pos, int64_t ldp,
                         int k, int init, float* best_score, int64_t* best_pos, void* stream);
int nnr_topk_merge_lists_capped(const float* scores, int64_t lds, int B, int T, const int64_t* pos, int64_t ldp,
                                const int32_t* grp, int64_t ldg, int num_groups, int cap, int k, int init,
                                float* best_score, int64_t* best_pos, int32_t* best_group, void* stream);

/* elementwise dropout with the library's counter RNG (proxy nodes / cluster features /
 * GCN inter-layer dropout): y = x * keep(seed, i)/(1-p); the same call applies the backward.   */
int nnr_dropout(const float* x, int64_t n, float p_drop, uint64_t seed, float* y, void* stream);

/* ---- optimizer: trainer.py:118-120 (clip_grad_norm_(4) + Adam) over one flat buffer ---------
 * norm_out[0] receives the pre-clip global L2 norm.  step is 1-based.                           */
size_t nnr_flat_clip_adam_workspace_bytes(int64_t n);
int nnr_flat_clip_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                       int64_t n, float lr, float beta1, float beta2, float eps, float max_norm,
                       float grad_scale, int32_t step, float* norm_out, void* workspace,
                       size_t workspace_bytes, void* stream);
/* the same with Adam's step counter on the device: the call increments *step_dev (int32, starts at 0) and derives the
 * bias corrections from it, so a CUDA graph that captured the call advances the step on every replay.               */
int nnr_flat_clip_adam_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                           int64_t n, float lr, float beta1, float beta2, float eps, float max_norm,
                           float grad_scale, int32_t* step_dev, float* norm_out, void* workspace,
                           size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NNR_B200_H */
