// Bidirectional LSTM recurrence, forward and backward-through-time, as persistent thread-block
// cluster kernels (sm_100a).  Replaces cuDNN's RNN behind nn.LSTM at newsEncoders.py:66-67,119-127.
//
// Design
//   * One cluster of CL = 4 CTAs owns a tile of sequences and one direction.  CTA r of the cluster owns
//     hidden units [r*H/4, (r+1)*H/4): the i,f,g,o rows of those units, i.e. a [4*H/4, H] slice of
//     W_hh = 160 KB fp32 for H = 200, which stays in shared memory for every time step of every tile the
//     cluster processes (the kernel is persistent over tiles).
//   * forward step (32-row tiles): z = gx_t + h_{t-1} W_slice^T, register tiled FFMA (2 units x 4 gates x
//     4 rows per thread), fused sigmoid/tanh/cell update with c_t kept in registers, then the new h slice is
//     broadcast into all four CTAs' (double-buffered) h tiles through distributed shared memory and one
//     barrier.cluster per step publishes it.  (A 64-row single-buffer variant was measured: better FFMA
//     efficiency but a longer per-step latency, which loses on MIND-like length distributions where the
//     longest sequences set the critical path.)
//   * backward step (32-row tiles): each CTA turns dh_t (+ recurrent part) into d(pre-activations) for its
//     own units, multiplies them with its W slice to get a PARTIAL dh_{t-1} over all H units, and
//     reduce-scatters the partials to the owning CTAs through DSMEM (fixed summation order ->
//     deterministic).
//   * the per-step exchange uses st.async into the peers' shared memory with mbarrier transaction counts
//     (and, in BPTT, a "recv is free" barrier fed by remote arrives) - no barrier.cluster inside the time loop.
//   * variable lengths: rows are tiled in length-sorted order; a row is active for its own `len` steps only
//     (packed-sequence semantics); the reverse direction walks t = len-1 .. 0.
//   * the input projection gx (a dense GEMM) is computed outside (nnr_gemm); the activated gates
//     overwrite gx in place as the stash for BPTT, and BPTT overwrites them with dL/dgx.
#include "lstm_common.cuh"
#include "../../include/nnr_b200.h"
#include <stdlib.h>
#include <string.h>

template <int HID_, int CL_, int MT_, int UPT_, int RPT_ = 4>   // hidden, cluster size, rows per tile, units / rows per thread
struct LCfg {
  static constexpr int HID = HID_, CL = CL_, MT = MT_, UPT = UPT_, RPT = RPT_;
  static constexpr int UPC = HID / CL;        // hidden units per CTA
  static constexpr int COLS = 4 * UPC;        // gate columns per CTA
  static constexpr int UG = UPC / UPT;        // unit groups
  static constexpr int RG = MT / RPT;         // row groups (one warp each)
  static constexpr int NT = RG * 32;          // one warp per row group; lanes [0, UG) work (warp-aligned: no
                                              // shared-memory bank conflicts between row groups, h loads broadcast)
  static_assert(UG <= 32, "unit groups must fit one warp");
  static_assert(HID % CL == 0 && UPC % UPT == 0 && MT % RPT == 0 && RPT % 4 == 0 && HID % 4 == 0, "unsupported LSTM geometry");
  static constexpr size_t FWD_SMEM = sizeof(float) * ((size_t)HID * COLS + 2 * (size_t)HID * MT) + 3 * MT * sizeof(int);
  static constexpr size_t BWD_SMEM = sizeof(float) * ((size_t)COLS * HID + (size_t)COLS * MT + (size_t)CL * UPC * MT) + 3 * MT * sizeof(int);
};

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <class C>
__global__ void __launch_bounds__(C::NT, 1)
lstm_fwd_kernel(float* __restrict__ gx, const float* __restrict__ w_hh, const int32_t* __restrict__ len,
                const int32_t* __restrict__ off, const int32_t* __restrict__ order, int N, int ntiles,
                float* __restrict__ h_out, float* __restrict__ c_stash, float* __restrict__ c_n, int* __restrict__ tile_counter) {
  constexpr int HID = C::HID, CL = C::CL, MT = C::MT, UPC = C::UPC, COLS = C::COLS, UP = C::UG;
  constexpr int RPT = C::RPT;                  // rows per thread (register tile: 2 units x 4 gates x RPT rows)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Wt = reinterpret_cast<float*>(smem_raw);                 // [HID][COLS]
  float* hT = Wt + (size_t)HID * COLS;                            // [2][HID][MT]
  int* s_row = reinterpret_cast<int*>(hT + 2 * (size_t)HID * MT); // [MT]
  int* s_len = s_row + MT;
  int* s_off = s_len + MT;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cluster_id = blockIdx.x / CL;
  const int nclusters = gridDim.x / CL;
  const int dir = cluster_id & 1;
  const int tid = threadIdx.x;
  const int up = tid & 31, rg = tid >> 5;      // lane = unit pair, warp = row group
  const bool worker = up < UP;
  const int j0 = 2 * min(up, UP - 1);          // local unit of this thread (and j0+1)
  const int unit0 = rank * UPC + j0;           // global hidden unit

  // W slice -> smem, transposed to k-major: Wt[k][g*UPC + j] = W_hh[dir][g*HID + rank*UPC + j][k]
  {
    const float* W = w_hh + (size_t)dir * 4 * HID * HID;
    for (int idx = tid; idx < COLS * HID; idx += C::NT) {
      int c = idx / HID, k = idx - c * HID;
      int g = c / UPC, j = c - g * UPC;
      Wt[(size_t)k * COLS + c] = W[(size_t)(g * HID + rank * UPC + j) * HID + k];
    }
  }
  __shared__ __align__(8) uint64_t hfull[2];        // "all of h for the next step has landed in buffer b"
  uint32_t remote_hT[CL], remote_bar[CL];
#pragma unroll
  for (int d = 0; d < CL; ++d) {
    remote_hT[d] = mapa_u32(smem_addr_u32(hT), d);
    remote_bar[d] = mapa_u32(smem_addr_u32(&hfull[0]), d);
  }
  if (tid == 0) {
    lbar_init(&hfull[0], 1);
    lbar_init(&hfull[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  cluster_arrive();      // every CTA of the cluster runs before a peer writes into its shared memory
  cluster_wait();
  uint32_t hph[2] = {0u, 0u};                       // phase parity per buffer (identical in every thread)

  const size_t GS = (size_t)2 * 4 * HID;  // gx row stride (both directions)
  // dynamic tile scheduling: tiles are sorted longest-first, so handing the next tile to whichever cluster
  // becomes free is longest-processing-time-first list scheduling (one atomic per tile, broadcast via DSMEM)
  __shared__ int s_tile;
  int* remote_tile[CL];
#pragma unroll
  for (int d = 0; d < CL; ++d) remote_tile[d] = cluster.map_shared_rank(&s_tile, d);
  (void)nclusters;
  for (;;) {
    if (rank == 0 && tid == 0) {
      int t = atomicAdd(&tile_counter[dir], 1);
#pragma unroll
      for (int d = 0; d < CL; ++d) *remote_tile[d] = t;
    }
    cluster_arrive();
    cluster_wait();
    const int tile = s_tile;
    if (tile >= ntiles) break;
    __syncthreads();
    if (tid < MT) {
      int i = tile * MT + tid;
      int r = (i < N) ? order[i] : -1;
      s_row[tid] = r;
      s_len[tid] = (r >= 0) ? len[r] : 0;
      s_off[tid] = (r >= 0) ? off[r] : 0;
    }
    for (int idx = tid; idx < HID * MT; idx += C::NT) hT[idx] = 0.f;   // h_0 = 0 in buffer 0
    __syncthreads();
    int maxlen = 0;
    for (int i = 0; i < MT; ++i) maxlen = max(maxlen, s_len[i]);

    int rlen[RPT], roff[RPT], rrow[RPT];
    float cst[2][RPT], hst[2][RPT];
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      rlen[i] = worker ? s_len[RPT * rg + i] : 0;
      roff[i] = worker ? s_off[RPT * rg + i] : 0;
      rrow[i] = worker ? s_row[RPT * rg + i] : -1;
      cst[0][i] = cst[1][i] = hst[0][i] = hst[1][i] = 0.f;
    }
    // prefetch gx for step 0
    float2 gxr[4][RPT];  // [gate][row]
    auto load_gx = [&](int s) {
#pragma unroll
      for (int i = 0; i < RPT; ++i) {
        if (s < rlen[i]) {
          int t = dir ? (rlen[i] - 1 - s) : s;
          const float* p = gx + ((size_t)roff[i] + t) * GS + (size_t)dir * 4 * HID + unit0;
#pragma unroll
          for (int g = 0; g < 4; ++g) gxr[g][i] = *reinterpret_cast<const float2*>(p + g * HID);
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g) gxr[g][i] = make_float2(0.f, 0.f);
        }
      }
    };
    if (worker) load_gx(0);

    for (int s = 0; s < maxlen; ++s) {
      const int cur = s & 1, nxt = cur ^ 1;
      if (tid == 0 && s + 1 < maxlen) lbar_expect_tx(&hfull[nxt], (uint32_t)(HID * MT * sizeof(float)));  // arm for h_{s+1}
      if (s > 0) { lbar_wait_cluster(&hfull[cur], hph[cur]); hph[cur] ^= 1u; }                          // h_s landed
      if (worker) {
        // accumulators as packed pairs (unit j0, unit j0+1): one FFMA2 (fma.rn.f32x2) per gate and row
        float2 acc2[4][RPT];
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
          for (int i = 0; i < RPT; ++i) acc2[g][i] = gxr[g][i];
        if (s + 1 < maxlen) load_gx(s + 1);   // in flight during the k loop
        const float* hb = hT + (size_t)cur * HID * MT + RPT * rg;
        const float* wb = Wt + j0;
#pragma unroll 4
        for (int k = 0; k < HID; ++k) {
          float hv[RPT];
#pragma unroll
          for (int q = 0; q < RPT / 4; ++q) {
            const float4 t4 = *reinterpret_cast<const float4*>(hb + (size_t)k * MT + 4 * q);
            hv[4 * q] = t4.x; hv[4 * q + 1] = t4.y; hv[4 * q + 2] = t4.z; hv[4 * q + 3] = t4.w;
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float2 w = *reinterpret_cast<const float2*>(wb + (size_t)k * COLS + g * UPC);
#pragma unroll
            for (int i = 0; i < RPT; ++i) acc2[g][i] = __ffma2_rn(w, make_float2(hv[i], hv[i]), acc2[g][i]);
          }
        }
        float acc[4][2][RPT];
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
          for (int i = 0; i < RPT; ++i) { acc[g][0][i] = acc2[g][i].x; acc[g][1][i] = acc2[g][i].y; }
        // gates, state update, stash
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          if (s < rlen[i]) {
            int t = dir ? (rlen[i] - 1 - s) : s;
            size_t p = (size_t)roff[i] + t;
            float ig[2], fg[2], gg[2], og[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              ig[u] = fast_sigmoid(acc[0][u][i]);
              fg[u] = fast_sigmoid(acc[1][u][i]);
              gg[u] = fast_tanh(acc[2][u][i]);
              og[u] = fast_sigmoid(acc[3][u][i]);
              cst[u][i] = fg[u] * cst[u][i] + ig[u] * gg[u];
              hst[u][i] = og[u] * fast_tanh(cst[u][i]);
            }
            float* gp = gx + p * GS + (size_t)dir * 4 * HID + unit0;
            *reinterpret_cast<float2*>(gp) = make_float2(ig[0], ig[1]);
            *reinterpret_cast<float2*>(gp + HID) = make_float2(fg[0], fg[1]);
            *reinterpret_cast<float2*>(gp + 2 * HID) = make_float2(gg[0], gg[1]);
            *reinterpret_cast<float2*>(gp + 3 * HID) = make_float2(og[0], og[1]);
            *reinterpret_cast<float2*>(c_stash + (p * 2 + dir) * HID + unit0) = make_float2(cst[0][i], cst[1][i]);
            *reinterpret_cast<float2*>(h_out + p * 2 * HID + (size_t)dir * HID + unit0) = make_float2(hst[0][i], hst[1][i]);
            if (s == rlen[i] - 1)
              *reinterpret_cast<float2*>(c_n + (size_t)rrow[i] * 2 * HID + (size_t)dir * HID + unit0) =
                  make_float2(cst[0][i], cst[1][i]);
          }
        }
        // send the new h slice into every CTA's next buffer (frozen rows re-send their state); the bytes are
        // counted on the receiver's transaction barrier.  Double buffering + the data dependency of the
        // recurrence make the write-after-read safe without a second barrier.
        if (s + 1 < maxlen) {
          const uint32_t o = (uint32_t)(((size_t)nxt * HID * MT + (size_t)unit0 * MT + RPT * rg) * sizeof(float));
#pragma unroll
          for (int q = 0; q < RPT / 4; ++q) {
            const float4 h0 = make_float4(hst[0][4 * q], hst[0][4 * q + 1], hst[0][4 * q + 2], hst[0][4 * q + 3]);
            const float4 h1 = make_float4(hst[1][4 * q], hst[1][4 * q + 1], hst[1][4 * q + 2], hst[1][4 * q + 3]);
#pragma unroll
            for (int d = 0; d < CL; ++d) {
              st_async_f4(remote_hT[d] + o + 16 * q, h0, remote_bar[d] + nxt * 8);
              st_async_f4(remote_hT[d] + o + 16 * q + MT * sizeof(float), h1, remote_bar[d] + nxt * 8);
            }
          }
        }
      }
    }
  }
  // no CTA may exit while a peer can still write into its shared memory
  cluster_arrive();
  cluster_wait();
}

// ------------------------------------------------------------------------------------------------
// backward through time
// ------------------------------------------------------------------------------------------------
template <class C>
__global__ void __launch_bounds__(C::NT, 1)
lstm_bwd_kernel(float* __restrict__ gates, const float* __restrict__ c_stash, const float* __restrict__ w_hh,
                const int32_t* __restrict__ len, const int32_t* __restrict__ off, const int32_t* __restrict__ order,
                int N, int ntiles, const float* __restrict__ dh, const float* __restrict__ dcn, int* __restrict__ tile_counter) {
  constexpr int HID = C::HID, CL = C::CL, MT = C::MT, UPC = C::UPC, COLS = C::COLS, UP = C::UG;
  static_assert(C::UPT == 2 && MT == 32 && C::NT == 256, "backward kernel: 2 units per lane, 32-row tiles, 8 warps");
  constexpr int KG = HID / 4;                  // phase 2: groups of 4 k's (two warps of KG/2 lanes per 8-row group)
  static_assert(KG % 2 == 0 && KG / 2 <= 32, "phase-2 mapping");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Wc = reinterpret_cast<float*>(smem_raw);                 // [COLS][HID]  (c-major)
  float* dzT = Wc + (size_t)COLS * HID;                           // [COLS][MT]
  float* recv = dzT + (size_t)COLS * MT;                          // [CL][UPC][MT] partial dh from each peer
  int* s_row = reinterpret_cast<int*>(recv + (size_t)CL * UPC * MT);
  int* s_len = s_row + MT;
  int* s_off = s_len + MT;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cluster_id = blockIdx.x / CL;
  const int dir = cluster_id & 1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // phase 1: lane = unit pair, warp = group of 4 rows
  const bool worker = lane < UP;
  const int rg = warp;
  const int j0 = 2 * min(lane, UP - 1);
  const int unit0 = rank * UPC + j0;
  // phase 2: warps (2q, 2q+1) own rows 8q..8q+7; lanes own 4 consecutive k's
  const bool worker2 = lane < KG / 2;
  const int rg2 = warp >> 1;
  const int kg = (warp & 1) * (KG / 2) + min(lane, KG / 2 - 1);

  {
    const float* W = w_hh + (size_t)dir * 4 * HID * HID;
    for (int idx = tid; idx < COLS * HID; idx += C::NT) {
      int c = idx / HID, k = idx - c * HID;
      int g = c / UPC, jj = c - g * UPC;
      Wc[idx] = W[(size_t)(g * HID + rank * UPC + jj) * HID + k];
    }
  }
  // rfull: the CL partial slices of dh for the next iteration have landed in my recv (transaction barrier)
  // rfree: every CTA of the cluster has finished reading ITS recv, so mine may send (CL arrivals)
  __shared__ __align__(8) uint64_t rbar[2];
  uint64_t* rfull = &rbar[0];
  uint64_t* rfree = &rbar[1];
  uint32_t remote_recv[CL], remote_rfull[CL], remote_rfree[CL];
#pragma unroll
  for (int d = 0; d < CL; ++d) {
    remote_recv[d] = mapa_u32(smem_addr_u32(recv), d);
    remote_rfull[d] = mapa_u32(smem_addr_u32(rfull), d);
    remote_rfree[d] = mapa_u32(smem_addr_u32(rfree), d);
  }
  if (tid == 0) {
    lbar_init(rfull, 1);
    lbar_init(rfree, CL);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  cluster_arrive();      // every CTA of the cluster runs before a peer writes into its shared memory
  cluster_wait();
  uint32_t ph_full = 0u, ph_free = 0u;

  const size_t GS = (size_t)2 * 4 * HID;
  __shared__ int s_tile;
  int* remote_tile[CL];
#pragma unroll
  for (int d = 0; d < CL; ++d) remote_tile[d] = cluster.map_shared_rank(&s_tile, d);
  for (;;) {
    if (rank == 0 && tid == 0) {
      int t = atomicAdd(&tile_counter[dir], 1);
#pragma unroll
      for (int d = 0; d < CL; ++d) *remote_tile[d] = t;
    }
    cluster_arrive();
    cluster_wait();
    const int tile = s_tile;
    if (tile >= ntiles) break;
    __syncthreads();
    if (tid < MT) {
      int i = tile * MT + tid;
      int r = (i < N) ? order[i] : -1;
      s_row[tid] = r;
      s_len[tid] = (r >= 0) ? len[r] : 0;
      s_off[tid] = (r >= 0) ? off[r] : 0;
    }
    __syncthreads();
    int maxlen = 0;
    for (int i = 0; i < MT; ++i) maxlen = max(maxlen, s_len[i]);
    int rlen[4], roff[4], rrow[4];
    float dcc[2][4];   // dL/dc carried to the previous step
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      rlen[i] = worker ? s_len[4 * rg + i] : 0;
      roff[i] = worker ? s_off[4 * rg + i] : 0;
      rrow[i] = worker ? s_row[4 * rg + i] : -1;
      dcc[0][i] = dcc[1][i] = 0.f;
    }
    // stash of one iteration (gates, c_t, c_{t-1}, dh); (prefetching it a whole iteration ahead was measured
    // slower: the extra 56 live registers cost more than the hidden latency)
    float2 p_ig[4], p_fg[4], p_gg[4], p_og[4], p_ct[4], p_cp[4], p_dh[4];
    auto load_stash = [&](int s) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (s >= 0 && s < rlen[i]) {
          int t = dir ? (rlen[i] - 1 - s) : s;
          size_t p = (size_t)roff[i] + t;
          const float* gp = gates + p * GS + (size_t)dir * 4 * HID + unit0;
          p_ig[i] = *reinterpret_cast<const float2*>(gp);
          p_fg[i] = *reinterpret_cast<const float2*>(gp + HID);
          p_gg[i] = *reinterpret_cast<const float2*>(gp + 2 * HID);
          p_og[i] = *reinterpret_cast<const float2*>(gp + 3 * HID);
          p_ct[i] = *reinterpret_cast<const float2*>(c_stash + (p * 2 + dir) * HID + unit0);
          p_cp[i] = make_float2(0.f, 0.f);
          if (s > 0) {
            size_t pp = dir ? p + 1 : p - 1;
            p_cp[i] = *reinterpret_cast<const float2*>(c_stash + (pp * 2 + dir) * HID + unit0);
          }
          p_dh[i] = *reinterpret_cast<const float2*>(dh + p * 2 * HID + (size_t)dir * HID + unit0);
        }
      }
    };
    for (int s = maxlen - 1; s >= 0; --s) {
      if (worker) load_stash(s);          // issued before the wait so the loads overlap the DSMEM latency
      if (s < maxlen - 1) { lbar_wait_cluster(rfull, ph_full); ph_full ^= 1u; }   // partials of iteration s+1 landed
      if (worker) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float dz[4][2];
          if (s < rlen[i]) {
            int t = dir ? (rlen[i] - 1 - s) : s;
            size_t p = (size_t)roff[i] + t;
            float* gp = gates + p * GS + (size_t)dir * 4 * HID + unit0;
            const float2 ig = p_ig[i], fg = p_fg[i], gg = p_gg[i], og = p_og[i], ct = p_ct[i], cp = p_cp[i], dhu = p_dh[i];
            float dht[2] = {dhu.x, dhu.y};
            if (s == rlen[i] - 1) {   // the row's last step: start of its backward recursion
              float2 d0 = *reinterpret_cast<const float2*>(dcn + (size_t)rrow[i] * 2 * HID + (size_t)dir * HID + unit0);
              dcc[0][i] = d0.x; dcc[1][i] = d0.y;
            } else {
              // recurrent part: sum of the CL partials in fixed order
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                float r = 0.f;
#pragma unroll
                for (int src = 0; src < CL; ++src) r += recv[((size_t)src * UPC + j0 + u) * MT + 4 * rg + i];
                dht[u] += r;
              }
            }
            float iv[2] = {ig.x, ig.y}, fv[2] = {fg.x, fg.y}, gv[2] = {gg.x, gg.y}, ov[2] = {og.x, og.y};
            float cv[2] = {ct.x, ct.y}, cpv[2] = {cp.x, cp.y};
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              float tc = fast_tanh(cv[u]);
              float dc = dcc[u][i] + dht[u] * ov[u] * (1.f - tc * tc);
              dz[3][u] = dht[u] * tc * ov[u] * (1.f - ov[u]);
              dz[0][u] = dc * gv[u] * iv[u] * (1.f - iv[u]);
              dz[2][u] = dc * iv[u] * (1.f - gv[u] * gv[u]);
              dz[1][u] = dc * cpv[u] * fv[u] * (1.f - fv[u]);
              dcc[u][i] = dc * fv[u];
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) *reinterpret_cast<float2*>(gp + g * HID) = make_float2(dz[g][0], dz[g][1]);
          } else {
#pragma unroll
            for (int g = 0; g < 4; ++g) dz[g][0] = dz[g][1] = 0.f;
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            dzT[(size_t)(g * UPC + j0) * MT + 4 * rg + i] = dz[g][0];
            dzT[(size_t)(g * UPC + j0 + 1) * MT + 4 * rg + i] = dz[g][1];
          }
        }
      }
      __syncthreads();    // dzT complete; every thread of this CTA has consumed its recv values
      if (tid == 0 && s > 0) {
        lbar_expect_tx(rfull, (uint32_t)(CL * UPC * MT * sizeof(float)));           // arm for the partials of iteration s
#pragma unroll
        for (int d = 0; d < CL; ++d) rbar_arrive_release(remote_rfree[d]);           // "my recv may be overwritten"
      }
      // phase 2: partial dh_{t-1}[8 rows][4 k's] = sum_c dz[c][rows] * W[c][k]; packed pairs over rows (FFMA2)
      float2 a2[4][4];
      if (worker2 && s > 0) {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int i = 0; i < 4; ++i) a2[a][i] = make_float2(0.f, 0.f);
        const float* wb = Wc + 4 * kg;
        const float* zb = dzT + 8 * rg2;
#pragma unroll 4
        for (int c = 0; c < COLS; ++c) {
          const float4 z0 = *reinterpret_cast<const float4*>(zb + (size_t)c * MT);
          const float4 z1 = *reinterpret_cast<const float4*>(zb + (size_t)c * MT + 4);
          const float4 w = *reinterpret_cast<const float4*>(wb + (size_t)c * HID);
          const float2 z01 = make_float2(z0.x, z0.y), z23 = make_float2(z0.z, z0.w);
          const float2 z45 = make_float2(z1.x, z1.y), z67 = make_float2(z1.z, z1.w);
          const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const float2 ww = make_float2(wv[a], wv[a]);
            a2[a][0] = __ffma2_rn(ww, z01, a2[a][0]);
            a2[a][1] = __ffma2_rn(ww, z23, a2[a][1]);
            a2[a][2] = __ffma2_rn(ww, z45, a2[a][2]);
            a2[a][3] = __ffma2_rn(ww, z67, a2[a][3]);
          }
        }
      }
      if (s > 0) {
        lbar_wait_cluster(rfree, ph_free);   // every CTA has finished reading its recv -> safe to overwrite
        ph_free ^= 1u;
        if (worker2) {
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            int k = 4 * kg + a;
            int owner = k / UPC, kl = k - owner * UPC;
            const uint32_t o = (uint32_t)((((size_t)rank * UPC + kl) * MT + 8 * rg2) * sizeof(float));
            st_async_f4(remote_recv[owner] + o, make_float4(a2[a][0].x, a2[a][0].y, a2[a][1].x, a2[a][1].y), remote_rfull[owner]);
            st_async_f4(remote_recv[owner] + o + 16, make_float4(a2[a][2].x, a2[a][2].y, a2[a][3].x, a2[a][3].y), remote_rfull[owner]);
          }
        }
      }
      __syncthreads();    // dzT is rewritten by the next iteration's phase 1
    }
  }
  cluster_arrive();
  cluster_wait();
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef LCfg<200, 4, 32, 2, 4> FwdCfg200;  // 8 warps of 4 rows x 25 unit pairs, double-buffered h (8 rows per thread measured slower)
typedef LCfg<200, 4, 32, 2> BwdCfg200;     // 8 warps: phase 1 (25 unit pairs x 4 rows per warp), phase 2 (8 rows x 4 k's per lane)

template <class C, class K>
static int launch_cluster(K kernel, size_t smem, int ntiles, cudaStream_t st, void** args, const char* name) {
  static int max_clusters_cache = 0;
  static bool attr_set = false;
  if (!attr_set) {
    NNR_CUDA(cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C::CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cfg.blockDim = dim3(C::NT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  if (max_clusters_cache == 0) {
    cfg.gridDim = dim3(C::CL * 2);
    int nc = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&nc, (const void*)kernel, &cfg);
    if (e != cudaSuccess || nc < 2) { (void)cudaGetLastError(); nc = 32; }
    max_clusters_cache = nc & ~1;
  }
  int want = 2 * ntiles;                      // (tile, direction) pairs
  int nclusters = want < max_clusters_cache ? want : max_clusters_cache;
  if (nclusters < 2) nclusters = 2;
  cfg.gridDim = dim3(nclusters * C::CL);
  cudaError_t e = cudaLaunchKernelExC(&cfg, (const void*)kernel, args);
  nnr_count_launch(1);
  if (e != cudaSuccess) { nnr_set_error("%s: launch failed: %s", name, cudaGetErrorString(e)); return (int)e; }
  return 0;
}

// tensor-core variant (lstm_mma.cu); NNR_LSTM_ALGO=ffma selects the exact-fp32 FFMA kernels of this file
int nnr_lstm_fwd_mma(float* gx, const float* w_hh, const int32_t* len, const int32_t* off, const int32_t* order, int N, int H,
                     float* h_out, float* c_stash, float* c_n, int32_t* tile_counters, cudaStream_t st, void* h_planes,
                     size_t plane_stride, int two_planes, int cap);
int nnr_lstm_fwd_planes_ok(void);
int nnr_lstm_bwd_tm_ok(void);
int nnr_lstm_bwd_mma(float* gates, const float* c_stash, const float* w_hh, const int32_t* len, const int32_t* off,
                     const int32_t* order, int N, int H, const float* dh, const float* dcn, int32_t* tile_counters, cudaStream_t st,
                     void* dz_planes, size_t plane_stride, int two_planes, float* db_partial, float* db, int cap);
static bool lstm_use_mma() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("NNR_LSTM_ALGO");
    v = (e && !strcmp(e, "ffma")) ? 0 : 1;
  }
  return v == 1;
}

// The hidden sizes a recurrence entry point accepts, checked before any CUDA call.  The tensor-core kernels with the W slice in
// tensor memory (the default) take 0 < H <= 200, H % 4 == 0 (clusters of 2..5 CTAs of 40 units, 16 B chunks of 4 units); the
// exact-fp32 FFMA kernels and the shared-memory W variants are instantiated for hidden_dim 200 only.
static int lstm_check_hidden(const char* fn, int H, bool tm) {
  NNR_REQUIRE(H > 0 && H <= 200 && H % 4 == 0, NNR_ERR_UNSUPPORTED,
              "%s: hidden_dim %d: the tensor-core recurrence takes H %% 4 == 0 and H <= 200", fn, H);
  NNR_REQUIRE(H == 200 || lstm_use_mma(), NNR_ERR_UNSUPPORTED,
              "%s: hidden_dim %d: the exact-fp32 FFMA recurrence (NNR_LSTM_ALGO=ffma) takes hidden_dim 200 only", fn, H);
  NNR_REQUIRE(H == 200 || tm, NNR_ERR_UNSUPPORTED, "%s: hidden_dim %d: the shared-memory W variant (%s=0) takes hidden_dim 200 only", fn, H,
              !strcmp(fn, "nnr_lstm_fwd") ? "NNR_LSTM_FWD_TM" : "NNR_LSTM_BWD_TM");
  return 0;
}

extern "C" int nnr_lstm_fwd(float* gx, const float* w_hh, const int32_t* len, const int32_t* off, const int32_t* order,
                            int N, int L, int H, float* h_out, float* c_stash, float* c_n, int32_t* tile_counters,
                            void* stream) {
  NNR_REQUIRE(gx && w_hh && len && off && order && h_out && c_stash && c_n && tile_counters && N > 0 && L > 0, NNR_ERR_ARG,
              "nnr_lstm_fwd: bad arguments");
  if (int rc = lstm_check_hidden("nnr_lstm_fwd", H, nnr_lstm_fwd_planes_ok())) return rc;
  NNR_REQUIRE(nnr_aligned16(gx) && nnr_aligned16(h_out) && nnr_aligned16(c_stash) && nnr_aligned16(c_n), NNR_ERR_ALIGN,
              "nnr_lstm_fwd: buffers must be 16B aligned");
  if (lstm_use_mma()) return nnr_lstm_fwd_mma(gx, w_hh, len, off, order, N, H, h_out, c_stash, c_n, tile_counters, (cudaStream_t)stream, NULL, 0, 0, 0);
  typedef FwdCfg200 C;
  int ntiles = (N + C::MT - 1) / C::MT;
  NNR_CUDA(cudaMemsetAsync(tile_counters, 0, 2 * sizeof(int32_t), (cudaStream_t)stream));
  void* args[] = {&gx, &w_hh, &len, &off, &order, &N, &ntiles, &h_out, &c_stash, &c_n, &tile_counters};
  return launch_cluster<C>(lstm_fwd_kernel<C>, C::FWD_SMEM, ntiles, (cudaStream_t)stream, args, "lstm_fwd_kernel");
}

extern "C" int nnr_lstm_bwd(float* gates, const float* c_stash, const float* w_hh, const int32_t* len, const int32_t* off,
                            const int32_t* order, int N, int L, int H, const float* dh, const float* dcn,
                            int32_t* tile_counters, void* stream) {
  NNR_REQUIRE(gates && c_stash && w_hh && len && off && order && dh && dcn && tile_counters && N > 0 && L > 0, NNR_ERR_ARG,
              "nnr_lstm_bwd: bad arguments");
  if (int rc = lstm_check_hidden("nnr_lstm_bwd", H, nnr_lstm_bwd_tm_ok())) return rc;
  NNR_REQUIRE(nnr_aligned16(gates) && nnr_aligned16(c_stash) && nnr_aligned16(dh) && nnr_aligned16(dcn), NNR_ERR_ALIGN,
              "nnr_lstm_bwd: buffers must be 16B aligned");
  if (lstm_use_mma())
    return nnr_lstm_bwd_mma(gates, c_stash, w_hh, len, off, order, N, H, dh, dcn, tile_counters, (cudaStream_t)stream, NULL, 0, 0, NULL, NULL, 0);
  typedef BwdCfg200 C;
  int ntiles = (N + C::MT - 1) / C::MT;
  NNR_CUDA(cudaMemsetAsync(tile_counters, 0, 2 * sizeof(int32_t), (cudaStream_t)stream));
  void* args[] = {&gates, &c_stash, &w_hh, &len, &off, &order, &N, &ntiles, &dh, &dcn, &tile_counters};
  return launch_cluster<C>(lstm_bwd_kernel<C>, C::BWD_SMEM, ntiles, (cudaStream_t)stream, args, "lstm_bwd_kernel");
}

// forward recurrence whose h ALSO leaves as GEMM operand planes (h feeds the selective-gate GEMM and, in the backward pass, two
// weight-gradient GEMMs: newsEncoders.py:128-131): the split pass over h is skipped.  planes = [hi|lo][cap][2H] bf16 as
// nnr_tc_split(h, cap, 2H, ntok) would write them, rows [ntok, round_up(ntok, 64)) zeroed.
extern "C" int nnr_lstm_fwd_planes_supported(int H, int algo) {
  if (algo == NNR_GEMM_AUTO) algo = nnr_gemm_default_algo();
  return H == 200 && lstm_use_mma() && nnr_lstm_fwd_planes_ok() && (algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3);
}
extern "C" int nnr_lstm_fwd_planes(float* gx, const float* w_hh, const int32_t* len, const int32_t* off, const int32_t* order,
                                   int N, int L, int H, float* h_out, float* c_stash, float* c_n, int32_t* tile_counters, int cap,
                                   int algo, void* planes, size_t planes_bytes, void* stream) {
  NNR_REQUIRE(gx && w_hh && len && off && order && h_out && c_stash && c_n && tile_counters && planes && N > 0 && L > 0 && cap > 0,
              NNR_ERR_ARG, "nnr_lstm_fwd_planes: bad arguments");
  if (algo == NNR_GEMM_AUTO) algo = nnr_gemm_default_algo();
  NNR_REQUIRE(nnr_lstm_fwd_planes_supported(H, algo), NNR_ERR_UNSUPPORTED,
              "nnr_lstm_fwd_planes: needs H = 200, the tensor-memory forward kernel and a bf16 GEMM algorithm");
  NNR_REQUIRE(nnr_aligned16(gx) && nnr_aligned16(h_out) && nnr_aligned16(c_stash) && nnr_aligned16(c_n) && nnr_aligned16(planes),
              NNR_ERR_ALIGN, "nnr_lstm_fwd_planes: buffers must be 16B aligned");
  const int two = algo == NNR_GEMM_TC_BF16X3;
  const size_t plane = (size_t)cap * 2 * H;
  NNR_REQUIRE(planes_bytes >= plane * 2 * (two ? 2 : 1), NNR_ERR_WORKSPACE, "nnr_lstm_fwd_planes: planes buffer too small");
  return nnr_lstm_fwd_mma(gx, w_hh, len, off, order, N, H, h_out, c_stash, c_n, tile_counters, (cudaStream_t)stream, planes, plane, two, cap);
}

// BPTT with dL/dgx emitted as GEMM operand planes + its column sums (the bias gradient): dL/dgx is only ever read by the
// dW_ih / dW_hh / dx GEMMs and a column sum, so the fp32 tensor and the split pass over it are skipped.
extern "C" int nnr_lstm_bwd_planes_supported(int H, int algo) {
  if (algo == NNR_GEMM_AUTO) algo = nnr_gemm_default_algo();
  return H == 200 && lstm_use_mma() && (algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3);
}
extern "C" size_t nnr_lstm_bwd_planes_workspace_bytes(int N, int H) {
  if (N <= 0 || H <= 0) return 0;
  return (size_t)((N + 31) / 32) * 8 * (size_t)H * sizeof(float);
}
extern "C" int nnr_lstm_bwd_planes(const float* gates, const float* c_stash, const float* w_hh, const int32_t* len,
                                   const int32_t* off, const int32_t* order, int N, int L, int H, const float* dh,
                                   const float* dcn, int32_t* tile_counters, int cap, int algo, void* dz_planes,
                                   size_t planes_bytes, float* db, void* workspace, size_t workspace_bytes, void* stream) {
  NNR_REQUIRE(gates && c_stash && w_hh && len && off && order && dh && dcn && tile_counters && dz_planes && db && workspace &&
                  N > 0 && L > 0 && cap > 0, NNR_ERR_ARG, "nnr_lstm_bwd_planes: bad arguments");
  if (algo == NNR_GEMM_AUTO) algo = nnr_gemm_default_algo();
  NNR_REQUIRE(nnr_lstm_bwd_planes_supported(H, algo), NNR_ERR_UNSUPPORTED,
              "nnr_lstm_bwd_planes: needs hidden_dim 200, the tensor-core recurrence and a bf16 GEMM algorithm");
  NNR_REQUIRE(nnr_aligned16(gates) && nnr_aligned16(c_stash) && nnr_aligned16(dh) && nnr_aligned16(dcn) && nnr_aligned16(dz_planes),
              NNR_ERR_ALIGN, "nnr_lstm_bwd_planes: buffers must be 16B aligned");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(cap, 8 * H, algo), NNR_ERR_WORKSPACE, "nnr_lstm_bwd_planes: planes buffer too small");
  NNR_REQUIRE(workspace_bytes >= nnr_lstm_bwd_planes_workspace_bytes(N, H), NNR_ERR_WORKSPACE, "nnr_lstm_bwd_planes: workspace too small");
  return nnr_lstm_bwd_mma(const_cast<float*>(gates), c_stash, w_hh, len, off, order, N, H, dh, dcn, tile_counters, (cudaStream_t)stream,
                          dz_planes, (size_t)cap * 8 * H, algo == NNR_GEMM_TC_BF16X3 ? 1 : 0, (float*)workspace, db, cap);
}
