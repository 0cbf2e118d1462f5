// Tensor-core variant of the persistent bidirectional LSTM kernels (forward and BPTT) for 0 < H <= 200, H % 4 == 0 (clusters of
// CL = max(2, ceil(H / 40)) CTAs, see G).  The description below is for H = 200.
// Same interface, data layout and stash protocol as lstm.cu; replaces cuDNN's RNN behind nn.LSTM at
// newsEncoders.py:66-67,119-127.
//
// What changes against the FFMA kernels of lstm.cu:
//   * the recurrent product of a time step -- [32 rows x 200] x [200 x 4*units] -- runs on the tensor cores
//     (mma.sync m16n8k16, fp32 accumulate) with SPLIT operands: x = hi + lo in 16-bit, and
//     x*y ~= hi*hi + hi*lo + lo*hi (3 MMAs).  Forward splits h and W_hh in fp16 (|h| < 1: 22 mantissa bits
//     survive), BPTT splits d(pre-activations) and W_hh in bf16 (gradients need the fp32 exponent range;
//     16 mantissa bits, same grade as the bf16x3 GEMMs the gradients flow through next).
//   * a cluster is FIVE CTAs of 40 hidden units (160 gate columns): 40 units = 4 warps x 10 units = 4 x 5 n8 tiles,
//     so each of the four SM sub-partitions runs one warp with a 32 x 40 accumulator tile; the W slice lives in tensor
//     memory (see the W fill of each kernel), the h / dz tiles in shared memory with conflict-free ldmatrix pitches.
//   * the n8 tile column order is (gate, unit) = 2g + u for two units, so after a 4x4 shuffle transpose inside
//     each lane quad every lane owns ONE row and TEN consecutive units with all four gates: the point-wise LSTM
//     cell, the stash stores (32 B aligned runs) and the h broadcast (16 B chunks of the next step's A operand)
//     need no shared-memory staging.
//   * the K order of the h operand is a permutation of the units (the W slice is permuted identically when it
//     is loaded), chosen so that each lane's ten units land in one 16 B chunk + one 4 B chunk of the peers' tiles.
// The exchange protocol (st.async + mbarrier transaction counts, double-buffered h, rfull/rfree in BPTT), the
// longest-first dynamic tile scheduling and the packed-sequence semantics are those of lstm.cu.
#include "lstm_common.cuh"
#include "../../include/nnr_b200.h"
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

// optional in-kernel phase timing (clock64 of one lane of CTA 0), compiled in with -DNNR_LSTM_PROF
#ifdef NNR_LSTM_PROF
__device__ unsigned long long g_lstm_prof[16];
#define PROF_DECL unsigned long long pt0 = clock64(), pacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const bool prof_on = (blockIdx.x == 0 && threadIdx.x == 0);
#define PROF_MARK(i) { unsigned long long t_ = clock64(); pacc[i] += t_ - pt0; pt0 = t_; }
#define PROF_FLUSH(base) if (prof_on) { for (int i_ = 0; i_ < 8; ++i_) g_lstm_prof[base + i_] = pacc[i_]; }
#else
#define PROF_DECL
#define PROF_MARK(i)
#define PROF_FLUSH(base)
#endif

namespace {

// The cluster size CL sets the padded hidden size HP = 40 CL the kernels are laid out for (CL = max(2, ceil(H / 40))).  Units
// [H, HP) are ghost units: never read from or written to global memory, zero inside the kernel (zero W rows and K slots, h = c =
// dz = dc = 0).  Global strides use the runtime H; shared / tensor memory layouts use HP.  CL = 1 is not instantiated: the
// exchange and its transaction counts assume peers.
// Both kernels run 4 compute warps and 2 copy warps per CTA and keep the W slice in tensor memory, so two CTAs (of two
// different clusters) share an SM: one CTA's products keep the tensor pipe busy while the other is in its exchange wait /
// point-wise / store phases.
template <int CL_>
struct G {
  static constexpr int CL = CL_, HP = 40 * CL, MT = 32, UPC = 40, COLS = 160, CT = 128, NT = 192, UPW = 10, NTW = 5;   // CT compute + 64 copy threads
  // forward: A = h [32][K=FK (HP + zero pad to a multiple of 16)], B = W slice [160 cols][FK] in tensor memory.  HALF: HP % 16 == 8,
  // the last k-step is half padding (HP = 120, 200).
  static constexpr bool HALF = HP % 16 == 8;
  static constexpr int FK = (HP + 15) / 16 * 16, FKS = FK / 16;
  // h tile = [source CTA j][plane hi/lo][32 rows][40 slots = 80 B]: the slice a CTA produces is ONE contiguous 5120 B
  // block (a single cp.async.bulk per peer); row pitch 80 B keeps ldmatrix conflict free.  A 16 B zero chunk pads K.
  static constexpr int F_HROW = 80, F_HPLANE = MT * F_HROW, F_HBLK = 2 * F_HPLANE, F_HBUF = CL * F_HBLK;
  // staging tile for coalesced global traffic: [array][32 rows][40 units fp32 + 16 B pad]; the CTA's copy threads move
  // it to / from global memory in 16 B pieces (a row segment = 160 contiguous bytes), the owners access it per row
  static constexpr int SROW = 176, SARR = MT * SROW, SCHUNKS = MT * 10;   // 10 x 16 B chunks per row segment
  static constexpr int F_NARR = 6;                       // i, f, g, o (gx in, activated gates out), c, h
  static constexpr uint32_t F_TX = (CL - 1) * F_HBLK;    // bytes the peers copy into one CTA's next h tile per step
  static constexpr int F_ZERO = HALF ? 16 : 0;             // the K pad chunk the half k-step reads
  // forward tensor-memory columns: 20 per full k-step, 10 for the half one: 100 / 150 / 200 / 250 for CL = 2 .. 5
  static constexpr int F_TM_USED = 20 * (FKS - HALF) + 10 * HALF, F_TM_COLS = F_TM_USED <= 128 ? 128 : 256;
  static_assert(F_TM_USED <= 256, "forward W slice exceeds the tensor memory of one CTA");
  static constexpr size_t FWD_SMEM = 2 * (size_t)F_HBUF + F_ZERO + F_NARR * (size_t)SARR + 3 * MT * sizeof(int);
  // backward: A = dz [32][K'=160], B = W slice^T [HP units][160]; recv = partial dh from every CTA
  // ([source CTA][32 rows][40 units] fp32 = 5120 B blocks: one bulk copy each) and the staging tile of the same shape
  // the partials are copied from.
  static constexpr int BK = 160, BKS = 10, BPITCH = 336, BWPITCH = 320, RPITCH = UPC * 4;
  static constexpr int B_Z_PLANE = MT * BPITCH, B_RBLK = MT * RPITCH, B_RECV = CL * B_RBLK;
  static constexpr int B_NARR = 5;                       // i, f, g, o (stash in, dz out), dh
  static constexpr uint32_t B_TX = CL * B_RBLK;
  // backward phase 2: the 5 CL n8 tiles of output units over the 4 compute warps, the first EXTRA warps take one more
  // (CL = 5: 7, 6, 6, 6; CL = 4: 5 each; CL = 3: 4, 4, 4, 3; CL = 2: 3, 3, 2, 2)
  static constexpr int NTILE = 5 * CL, BASE = NTILE / 4, EXTRA = NTILE % 4, NTWB = BASE + (EXTRA > 0);
  // up to six of a warp's n8 tiles live in tensor memory as ready-made mma.sync B fragments, the remainder (CL = 5: warp 0's
  // seventh tile, 8 units) stays in shared memory
  static constexpr int B_NTM = NTWB < 6 ? NTWB : 6, B_NSM = NTWB - B_NTM;   // n8 tiles per warp in tensor / shared memory
  static_assert(B_NSM == 0 || (B_NSM == 1 && EXTRA == 1), "the shared-memory tile is warp 0's only");
  static constexpr int B_TM_USED = BKS * B_NTM * 4, B_TM_COLS = B_TM_USED <= 128 ? 128 : 256;   // 10 k-steps x B_NTM tiles x 4 registers
  // [8 units][160 k] bf16, XOR-swizzled (16 B chunk ^= (row >> 1) & 3) instead of padded
  static constexpr int B_W7_PLANE = B_NSM * 8 * BWPITCH;
  static constexpr size_t BWD_SMEM = 2 * (size_t)B_W7_PLANE + 2 * (size_t)B_Z_PLANE + 2 * (size_t)B_RECV + B_NARR * (size_t)SARR + 3 * MT * sizeof(int);
};

// tensor memory -> registers, N consecutive columns of the warp's lane quarter (x16 / x8 / x4 pieces)
template <int N>
__device__ __forceinline__ void tm_ld(uint32_t* r, uint32_t addr) {
  if constexpr (N >= 16) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr));
    tm_ld<N - 16>(r + 16, addr + 16);
  } else if constexpr (N >= 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(addr));
    tm_ld<N - 8>(r + 8, addr + 8);
  } else if constexpr (N >= 4) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
    tm_ld<N - 4>(r + 4, addr + 4);
  } else {
    static_assert(N == 0, "column count must be a multiple of 4");
  }
}

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
template <bool F16>
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if (F16)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// (a, b) -> packed 16-bit pairs hi, lo with a ~= hi.x + lo.x, b ~= hi.y + lo.y (a at the lower address)
template <bool F16>
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  if (F16) {
    __half2 h = __floats2half2_rn(a, b);
    float2 f = __half22float2(h);
    __half2 l = __floats2half2_rn(a - f.x, b - f.y);
    hi = *reinterpret_cast<uint32_t*>(&h);
    lo = *reinterpret_cast<uint32_t*>(&l);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    float2 f = __bfloat1622float2(h);
    __nv_bfloat162 l = __floats2bfloat162_rn(a - f.x, b - f.y);
    hi = *reinterpret_cast<uint32_t*>(&h);
    lo = *reinterpret_cast<uint32_t*>(&l);
  }
}
template <bool F16>
__device__ __forceinline__ void split1(float a, uint16_t& hi, uint16_t& lo) {
  uint32_t h, l;
  split2<F16>(a, 0.f, h, l);
  hi = (uint16_t)(h & 0xffffu);
  lo = (uint16_t)(l & 0xffffu);
}

// local shared memory -> a peer CTA's shared memory through the bulk-copy engine; the bytes are counted on the
// destination's transaction barrier.  (Thousands of 4-16 B st.async packets per step were measured to cost ~10 us:
// DSMEM wants few, large, contiguous transfers.)
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes, uint32_t remote_bar) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_cluster_addr),
               "r"(src_cta_addr), "r"(bytes), "r"(remote_bar)
               : "memory");
}
// named barriers: 1 = the four compute warps; 2 = "staging tile written" (compute arrives, copy waits);
// 3 = "staging tile loaded" (copy arrives, compute waits)
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 4x4 transpose of float2 blocks inside a lane quad: on return lane q holds in X[s] what lane s held in X[q]
__device__ __forceinline__ void quad_transpose(float2 (&X)[4], int q) {
  {
    const bool odd = q & 1;
    float2 s0 = odd ? X[0] : X[1], s1 = odd ? X[2] : X[3];
    float2 r0, r1;
    r0.x = __shfl_xor_sync(0xffffffffu, s0.x, 1); r0.y = __shfl_xor_sync(0xffffffffu, s0.y, 1);
    r1.x = __shfl_xor_sync(0xffffffffu, s1.x, 1); r1.y = __shfl_xor_sync(0xffffffffu, s1.y, 1);
    if (odd) { X[0] = r0; X[2] = r1; } else { X[1] = r0; X[3] = r1; }
  }
  {
    const bool up = q & 2;
    float2 s0 = up ? X[0] : X[2], s1 = up ? X[1] : X[3];
    float2 r0, r1;
    r0.x = __shfl_xor_sync(0xffffffffu, s0.x, 2); r0.y = __shfl_xor_sync(0xffffffffu, s0.y, 2);
    r1.x = __shfl_xor_sync(0xffffffffu, s1.x, 2); r1.y = __shfl_xor_sync(0xffffffffu, s1.y, 2);
    if (up) { X[0] = r0; X[1] = r1; } else { X[2] = r0; X[3] = r1; }
  }
}

// forward K order: slot -> hidden unit.  CTA j owns slots 40j .. 40j+39: warp w's first 8 units at 40j + 8w .. +7 (one
// 16 B chunk), its last 2 at 40j + 32 + 2w, +1
__device__ __forceinline__ int fwd_slot_unit(int kk) {
  const int j = kk / 40, rem = kk - 40 * j;
  if (rem < 32) return 40 * j + 10 * (rem >> 3) + (rem & 7);
  const int t = rem - 32;
  return 40 * j + 10 * (t >> 1) + 8 + (t & 1);
}

// ------------------------------------------------------------------------------------------------
// forward, W slice in tensor memory, two CTAs per SM (see the comment at the W fill)
// ------------------------------------------------------------------------------------------------
// HC: the hidden size as a compile-time constant (200: no ghost units, the arithmetic and addressing of a fixed-size kernel), or 0
// (taken from H_arg at run time)
template <bool SINGLE, int CL, int HC>   // SINGLE: one 16-bit product (hi x hi) instead of the three split products -- the bf16 variant
__global__ void __launch_bounds__(G<CL>::NT, 2)
lstm_fwd_tm_kernel(float* __restrict__ gx, const float* __restrict__ w_hh, const int32_t* __restrict__ len,
                    const int32_t* __restrict__ off, const int32_t* __restrict__ order, int N, int H_arg, int ntiles,
                    float* __restrict__ h_out, float* __restrict__ c_stash, float* __restrict__ c_n, int* __restrict__ tile_counter,
                    __nv_bfloat16* __restrict__ hp, size_t hp_stride, int hp_lo) {
  // hp != NULL: h also leaves as the bf16 operand planes of the tensor-core GEMMs that consume it ([hi|lo][cap][2H], plane
  // stride hp_stride elements, lo plane only if hp_lo) -- the split pass over h is skipped (same rounding as tc_split_store4)
  using G = ::G<CL>;
  constexpr int MT = G::MT, UPC = G::UPC, NTW = G::NTW, UPW = G::UPW;
  const int H = HC ? HC : H_arg;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* Hsm = smem_raw;                                   // [2 buffers][CL blocks][2 planes][MT][80 B]
  unsigned char* Zero16 = Hsm + 2 * G::F_HBUF;                     // the K pad chunk (HALF only)
  unsigned char* Stg = Zero16 + G::F_ZERO;                        // [F_NARR][MT][SROW] staging tile
  int* s_row = reinterpret_cast<int*>(Stg + G::F_NARR * G::SARR);
  int* s_len = s_row + MT;
  int* s_off = s_len + MT;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cluster_id = blockIdx.x / CL;
  const int dir = cluster_id & 1;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int q = lane & 3, r8 = lane >> 2;
  const int R = r8 + 8 * q;                     // the tile row this lane owns in the point-wise phase
  const int unit0 = rank * UPC + w * UPW;       // first of the lane's ten hidden units

  // ---- W slice -> TENSOR MEMORY, already in mma.sync B-fragment form.  Lane l of compute warp w (TMEM lanes 32 w + l; a warp
  // can only reach the lane quarter of its own index) keeps, for every k-step ks and n8 tile nt of the warp's 40 gate
  // columns, the registers b0 = W[n][16 ks + 2 (l % 4) + {0, 1}], b1 = the same 8 further along k, n = 40 w + 8 nt + l / 4
  // (rows in (warp, n-tile, gate, unit) order, k permuted by fwd_slot_unit like the h operand), as fp16 hi and lo:
  // columns ks * 20 + {0..9: hi (nt, b0/b1), 10..19: lo}; with HALF the last k-step (upper 8 k = zero pad) only stores b0:
  // columns 20 ks + {0..4: hi, 5..9: lo}.  250 of the 256 allocated columns at CL = 5.  As shared-memory planes the slice
  // would take 2 x 69 KB and leave room for one CTA per SM instead of two (see G).
  __shared__ uint32_t tmem_slot;
  if (w == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr_u32(&tmem_slot)), "n"(G::F_TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tm_w = tmem_slot + ((uint32_t)((w & 3) * 32) << 16);       // this warp's lane quarter
  if (w < 4) {
    const float* W = w_hh + (size_t)dir * 4 * H * H;
    const int c = lane >> 2, g = c >> 1, u = c & 1;
#pragma unroll 1
    for (int ks = 0; ks < G::FKS; ++ks) {
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        const int unit = rank * UPC + w * UPW + 2 * nt + u;       // gate row; ghost rows are zero
        const float* wrow = W + (size_t)(g * H + unit) * H;
        uint32_t hi[2], lo[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int kk = 16 * ks + 8 * j + 2 * (lane & 3);
          const int k0 = fwd_slot_unit(kk), k1 = fwd_slot_unit(kk + 1);   // K slots of ghost units (and of the pad) are zero
          const float v0 = (unit < H && k0 < H) ? wrow[k0] : 0.f;
          const float v1 = (unit < H && k1 < H) ? wrow[k1] : 0.f;
          split2<true>(v0, v1, hi[j], lo[j]);
        }
        if (!G::HALF || ks < G::FKS - 1) {
          asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(tm_w + (uint32_t)(ks * 20 + nt * 2)), "r"(hi[0]), "r"(hi[1]) : "memory");
          asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(tm_w + (uint32_t)(ks * 20 + 10 + nt * 2)), "r"(lo[0]), "r"(lo[1]) : "memory");
        } else {
          asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(tm_w + (uint32_t)(ks * 20 + nt)), "r"(hi[0]) : "memory");
          asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(tm_w + (uint32_t)(ks * 20 + 5 + nt)), "r"(lo[0]) : "memory");
        }
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  // h buffers, the pad chunk and the staging tile start zero (the staging bytes of ghost units are never loaded)
  for (int idx = tid; idx < (2 * G::F_HBUF + G::F_ZERO + G::F_NARR * G::SARR) / 16; idx += G::NT)
    reinterpret_cast<uint4*>(Hsm)[idx] = make_uint4(0u, 0u, 0u, 0u);
  __shared__ __align__(8) uint64_t hfull[2];        // "all of h for the next step has landed in buffer b"
  __shared__ int s_tile;
  const uint32_t h_local = smem_addr_u32(Hsm), bar_local = smem_addr_u32(&hfull[0]);
  if (tid == 0) {
    lbar_init(&hfull[0], 1);
    lbar_init(&hfull[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // every CTA of the cluster must have started before its shared memory is written from a peer (the tile index below, then
  // the h exchange): compute-sanitizer racecheck flags the first remote store otherwise ("block that might not have entered yet")
  cluster_arrive();
  cluster_wait();
  uint32_t hph[2] = {0u, 0u};
  const size_t GS = (size_t)2 * 4 * H;
  PROF_DECL

  // per-lane fragment offsets (bytes)
  const uint32_t a_row = (uint32_t)((lane & 15) * G::F_HROW);   // A: lanes 0-15 address k chunk 2ks, lanes 16-31 chunk 2ks+1
  const bool a_hi = (lane >> 4) != 0;
  const uint32_t zero_local = smem_addr_u32(Zero16), stg_local = smem_addr_u32(Stg);
  const bool copy_role = w >= 4;                                 // warps 4-5 move the staging tile to / from global memory
  const int c_ch = tid & 15, c_rs = (tid - G::CT) >> 4;          // cooperative copy: chunk and row slot of a copy thread
  const bool ch_ok = c_ch < 10 && rank * UPC + c_ch * 4 < H;     // the chunk's 4 units are all real or all ghost (H % 4 == 0)
  const uint32_t c_so = (uint32_t)(c_rs * G::SROW + c_ch * 16);  // its offset inside an array of the staging tile
  // where this lane's h values go inside this CTA's block of an h tile (plane 0; plane 1 is F_HPLANE further)
  const uint32_t stage_v4 = (uint32_t)(rank * G::F_HBLK + R * G::F_HROW + w * 16);
  const uint32_t stage_b32 = (uint32_t)(rank * G::F_HBLK + R * G::F_HROW + 64 + w * 4);

  for (;;) {
    if (rank == 0 && tid == 0) {
      int t = atomicAdd(&tile_counter[dir], 1);
#pragma unroll
      for (int d = 0; d < CL; ++d) *cluster.map_shared_rank(&s_tile, d) = t;
    }
    cluster_arrive();
    cluster_wait();
    const int tile = s_tile;
    if (tile >= ntiles) break;
    __syncthreads();
    if (tid < MT) {
      int i = tile * MT + tid;
      int rr = (i < N) ? order[i] : -1;
      s_row[tid] = rr;
      s_len[tid] = (rr >= 0) ? len[rr] : 0;
      s_off[tid] = (rr >= 0) ? off[rr] : 0;
    }
    for (int idx = tid; idx < G::F_HBUF / 16; idx += G::NT) reinterpret_cast<uint4*>(Hsm)[idx] = make_uint4(0u, 0u, 0u, 0u);  // h_0 = 0
    __syncthreads();
    int maxlen = 0;
    for (int i = 0; i < MT; ++i) maxlen = max(maxlen, s_len[i]);
    const int rlen = s_len[R], roff = s_off[R], rrow = s_row[R];

    if (copy_role) {
      // ---- copy warps: coalesced traffic between the staging tile and global memory, off the compute warps' critical
      // path.  Thread t moves the 16 B chunk ch = t & 15 (10 of 16 lanes active) of the 160 B row segments of rows
      // (t >> 4) + 4 rr, rr = 0..7, of every array (64 copy threads).
      int c_len[8], c_off[8];
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) { c_len[rr] = s_len[c_rs + 4 * rr]; c_off[rr] = s_off[c_rs + 4 * rr]; }
      if (ch_ok) {                        // gx of step 0
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          if (0 < c_len[rr]) {
            const int t = dir ? (c_len[rr] - 1) : 0;
            const float* g1 = gx + ((size_t)c_off[rr] + t) * GS + (size_t)dir * 4 * H + rank * UPC + c_ch * 4;
#pragma unroll
            for (int a = 0; a < 4; ++a) cp_async16(stg_local + c_so + rr * 4 * G::SROW + a * G::SARR, g1 + a * H);
          }
        }
      }
      cp_async_commit();
      cp_async_wait_all();
      bar_arrive(3, G::NT);
      for (int s = 0; s < maxlen; ++s) {
        bar_sync(2, G::NT);              // the staging tile holds the stash of step s
        if (ch_ok) {
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            const int rl = c_len[rr];
            if (s < rl) {
              const int t = dir ? (rl - 1 - s) : s;
              const size_t p = (size_t)c_off[rr] + t;
              const unsigned char* sp = Stg + c_so + rr * 4 * G::SROW;
              float* g0 = gx + p * GS + (size_t)dir * 4 * H + rank * UPC + c_ch * 4;
#pragma unroll
              for (int a = 0; a < 4; ++a) *reinterpret_cast<float4*>(g0 + a * H) = *reinterpret_cast<const float4*>(sp + a * G::SARR);
              const float4 cv = *reinterpret_cast<const float4*>(sp + 4 * G::SARR);
              *reinterpret_cast<float4*>(c_stash + (p * 2 + dir) * H + rank * UPC + c_ch * 4) = cv;
              const float4 hv = *reinterpret_cast<const float4*>(sp + 5 * G::SARR);
              const size_t ho = p * 2 * H + (size_t)dir * H + rank * UPC + c_ch * 4;
              *reinterpret_cast<float4*>(h_out + ho) = hv;
              if (hp) {
                const __nv_bfloat162 h01 = __floats2bfloat162_rn(hv.x, hv.y), h23 = __floats2bfloat162_rn(hv.z, hv.w);
                uint2 hw;
                hw.x = *reinterpret_cast<const uint32_t*>(&h01); hw.y = *reinterpret_cast<const uint32_t*>(&h23);
                *reinterpret_cast<uint2*>(hp + ho) = hw;
                if (hp_lo) {
                  const __nv_bfloat162 l01 = __floats2bfloat162_rn(hv.x - __low2float(h01), hv.y - __high2float(h01));
                  const __nv_bfloat162 l23 = __floats2bfloat162_rn(hv.z - __low2float(h23), hv.w - __high2float(h23));
                  uint2 lw;
                  lw.x = *reinterpret_cast<const uint32_t*>(&l01); lw.y = *reinterpret_cast<const uint32_t*>(&l23);
                  *reinterpret_cast<uint2*>(hp + hp_stride + ho) = lw;
                }
              }
              if (s == rl - 1)
                *reinterpret_cast<float4*>(c_n + (size_t)s_row[c_rs + 4 * rr] * 2 * H + (size_t)dir * H + rank * UPC + c_ch * 4) = cv;
              if (s + 1 < rl) {            // the row's next token is the adjacent one
                const float* g1 = dir ? g0 - GS : g0 + GS;
#pragma unroll
                for (int a = 0; a < 4; ++a) cp_async16(stg_local + c_so + rr * 4 * G::SROW + a * G::SARR, g1 + a * H);
              }
            }
          }
        }
        if (s + 1 < maxlen) {
          cp_async_commit();
          cp_async_wait_all();
          bar_arrive(3, G::NT);          // gx of step s+1 is in the staging tile
        }
      }
      continue;
    }

    // ---- compute warps ---------------------------------------------------------------------------------------------
    float cst[UPW], hst[UPW];
#pragma unroll
    for (int i = 0; i < UPW; ++i) cst[i] = hst[i] = 0.f;

    for (int s = 0; s < maxlen; ++s) {
      const int cur = s & 1, nxt = cur ^ 1;
      PROF_MARK(5)
      if (tid == 0 && s + 1 < maxlen) lbar_expect_tx(&hfull[nxt], G::F_TX);
      if (s > 0) { lbar_wait_cluster(&hfull[cur], hph[cur]); hph[cur] ^= 1u; }
      PROF_MARK(0)

      // ---- recurrent product on the tensor cores: acc[mt][nt] (16 x 8) += h_tile x W_slice^T --------------
      float acc[2][NTW][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
      const uint32_t hA = h_local + (uint32_t)(cur * G::F_HBUF) + a_row;
      // fragments of k-step ks+1 are loaded before the MMAs of k-step ks are issued (register double buffer);
      // consecutive MMAs on one accumulator are ten instructions apart
      struct Frag { uint32_t ah[2][4], al[2][4], bh[NTW][2], bl[NTW][2]; };
      auto load_frags = [&](Frag& f, int ks) {
        // k chunks 2ks and 2ks+1 of the global slot order: chunk c lives in block c / 5 at 16 B offset c % 5
        const int c0 = 2 * ks, c1 = 2 * ks + 1;
        const uint32_t o0 = (uint32_t)((c0 / 5) * G::F_HBLK + (c0 % 5) * 16), o1 = (uint32_t)((c1 / 5) * G::F_HBLK + (c1 % 5) * 16);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          uint32_t ad_h, ad_l;
          if (c1 < 5 * CL) {
            ad_h = hA + mt * 16 * G::F_HROW + (a_hi ? o1 : o0);
            ad_l = ad_h + G::F_HPLANE;
          } else {                      // K pad: the upper chunk reads zeros
            ad_h = a_hi ? zero_local : hA + mt * 16 * G::F_HROW + o0;
            ad_l = a_hi ? zero_local : ad_h + G::F_HPLANE;
          }
          ldsm_x4(ad_h, f.ah[mt][0], f.ah[mt][1], f.ah[mt][2], f.ah[mt][3]);
          if (!SINGLE) ldsm_x4(ad_l, f.al[mt][0], f.al[mt][1], f.al[mt][2], f.al[mt][3]);
        }
        // B fragments of this k-step from tensor memory (asynchronous: tm_wait() before their first use)
        if (!G::HALF || ks < G::FKS - 1) {
          uint32_t r[20];
          if (!SINGLE) {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                           "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                         : "r"(tm_w + (uint32_t)(ks * 20)));
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]) : "r"(tm_w + (uint32_t)(ks * 20 + 16)));
          } else {
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                         : "r"(tm_w + (uint32_t)(ks * 20)));
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[8]), "=r"(r[9]) : "r"(tm_w + (uint32_t)(ks * 20 + 8)));
          }
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt) {
            f.bh[nt][0] = r[2 * nt]; f.bh[nt][1] = r[2 * nt + 1];
            if (!SINGLE) { f.bl[nt][0] = r[10 + 2 * nt]; f.bl[nt][1] = r[10 + 2 * nt + 1]; }
          }
        } else {                         // half k-step: the upper 8 k are padding, b1 = 0
          uint32_t r[10];
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                       : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                       : "r"(tm_w + (uint32_t)(ks * 20)));
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[8]), "=r"(r[9]) : "r"(tm_w + (uint32_t)(ks * 20 + 8)));
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt) {
            f.bh[nt][0] = r[nt]; f.bh[nt][1] = 0u;
            if (!SINGLE) { f.bl[nt][0] = r[5 + nt]; f.bl[nt][1] = 0u; }
          }
        }
      };
      auto tm_wait = [&]() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); };
      auto mma_all = [&](const Frag& f) {
        if (!SINGLE) {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) mma16816<true>(acc[mt][nt], f.al[mt], f.bh[nt][0], f.bh[nt][1]);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) mma16816<true>(acc[mt][nt], f.ah[mt], f.bl[nt][0], f.bl[nt][1]);
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt) mma16816<true>(acc[mt][nt], f.ah[mt], f.bh[nt][0], f.bh[nt][1]);
      };
      {
        Frag f0, f1;
        load_frags(f0, 0);
        tm_wait();
#pragma unroll
        for (int ks = 0; ks < G::FKS; ks += 2) {
          if (ks + 1 < G::FKS) load_frags(f1, ks + 1);       // in flight during the MMAs of k-step ks
          mma_all(f0);
          if (ks + 1 < G::FKS) {
            tm_wait();
            if (ks + 2 < G::FKS) load_frags(f0, ks + 2);
            mma_all(f1);
            if (ks + 2 < G::FKS) tm_wait();
          }
        }
      }

      PROF_MARK(1)
      // ---- quad transpose: lane (r8, q) ends with row R = r8 + 8q, gates x 10 units -------------------------
      float2 pre[NTW][4];
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) {
        float2 X[4] = {make_float2(acc[0][nt][0], acc[0][nt][1]), make_float2(acc[0][nt][2], acc[0][nt][3]),
                       make_float2(acc[1][nt][0], acc[1][nt][1]), make_float2(acc[1][nt][2], acc[1][nt][3])};
        quad_transpose(X, q);
#pragma unroll
        for (int g = 0; g < 4; ++g) pre[nt][g] = X[g];
      }

      // ---- LSTM cell on the lane's row: gx comes from the staging tile, the stash goes back into it --------------
      bar_sync(3, G::NT);            // the copy warps have stored step s-1 and fetched gx of step s
      if (s < rlen) {
        unsigned char* sp = Stg + R * G::SROW + w * (UPW * 4);
#pragma unroll
        for (int nt = 0; nt < NTW; ++nt) {
          const bool live = unit0 + 2 * nt < H;   // units 2 nt, 2 nt + 1 are both real or both ghost (H even)
          float2* gi = reinterpret_cast<float2*>(sp + 0 * G::SARR + nt * 8);
          float2* gf = reinterpret_cast<float2*>(sp + 1 * G::SARR + nt * 8);
          float2* gg_ = reinterpret_cast<float2*>(sp + 2 * G::SARR + nt * 8);
          float2* go = reinterpret_cast<float2*>(sp + 3 * G::SARR + nt * 8);
          const float2 xi = *gi, xf = *gf, xg = *gg_, xo = *go;
          float ig[2], fg[2], gg[2], og[2];
          const float zi[2] = {pre[nt][0].x + xi.x, pre[nt][0].y + xi.y};
          const float zf[2] = {pre[nt][1].x + xf.x, pre[nt][1].y + xf.y};
          const float zg[2] = {pre[nt][2].x + xg.x, pre[nt][2].y + xg.y};
          const float zo[2] = {pre[nt][3].x + xo.x, pre[nt][3].y + xo.y};
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            ig[u] = fast_sigmoid(zi[u]);
            fg[u] = fast_sigmoid(zf[u]);
            gg[u] = fast_tanh(zg[u]);
            og[u] = fast_sigmoid(zo[u]);
            const float cnew = fg[u] * cst[2 * nt + u] + ig[u] * gg[u];
            const float hnew = og[u] * fast_tanh(cnew);
            cst[2 * nt + u] = live ? cnew : 0.f;   // ghost units stay exactly zero
            hst[2 * nt + u] = live ? hnew : 0.f;
          }
          *gi = make_float2(ig[0], ig[1]);
          *gf = make_float2(fg[0], fg[1]);
          *gg_ = make_float2(gg[0], gg[1]);
          *go = make_float2(og[0], og[1]);
          *reinterpret_cast<float2*>(sp + 4 * G::SARR + nt * 8) = make_float2(cst[2 * nt], cst[2 * nt + 1]);
          *reinterpret_cast<float2*>(sp + 5 * G::SARR + nt * 8) = make_float2(hst[2 * nt], hst[2 * nt + 1]);
        }
      }
      PROF_MARK(2)
      // ---- the lane's ten h values (fp16 hi / lo) go into this CTA's block of the next tile; one bulk copy per peer
      if (s + 1 < maxlen) {
        uint32_t hi[NTW], lo[NTW];
#pragma unroll
        for (int nt = 0; nt < NTW; ++nt) split2<true>(hst[2 * nt], hst[2 * nt + 1], hi[nt], lo[nt]);
        unsigned char* blk = Hsm + (size_t)nxt * G::F_HBUF;
        *reinterpret_cast<uint4*>(blk + stage_v4) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint32_t*>(blk + stage_b32) = hi[4];
        *reinterpret_cast<uint4*>(blk + G::F_HPLANE + stage_v4) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint32_t*>(blk + G::F_HPLANE + stage_b32) = lo[4];
      }
      bar_sync(1, G::CT);              // the CTA's h block is complete
      if (s + 1 < maxlen && tid == 0) {
        fence_proxy_async_smem();
        const uint32_t src = h_local + (uint32_t)(nxt * G::F_HBUF + rank * G::F_HBLK);
        const uint32_t bar = bar_local + nxt * 8;
#pragma unroll
        for (int d = 1; d < CL; ++d) {
          const int peer = (rank + d) % CL;
          bulk_copy_to_peer(mapa_u32(src, peer), src, G::F_HBLK, mapa_u32(bar, peer));
        }
      }
      bar_arrive(2, G::NT);            // hand the staging tile (stash of step s) to the copy warps
      PROF_MARK(3)
    }
  }
  PROF_FLUSH(0)
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (w == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_slot), "n"(G::F_TM_COLS) : "memory");
  cluster_arrive();
  cluster_wait();
}


// ------------------------------------------------------------------------------------------------
// backward through time
// ------------------------------------------------------------------------------------------------
// The W slice lives in tensor memory (see G): the CTA needs 104 KB of shared memory, and two CTAs share an SM.
template <bool SINGLE, int CL, int HC>   // SINGLE: one 16-bit product (hi x hi) instead of the three split products -- the bf16 variant
__global__ void __launch_bounds__(G<CL>::NT, 2)
lstm_bwd_mma_kernel(float* __restrict__ gates, const float* __restrict__ c_stash, const float* __restrict__ w_hh,
                    const int32_t* __restrict__ len, const int32_t* __restrict__ off, const int32_t* __restrict__ order,
                    int N, int H_arg, int ntiles, const float* __restrict__ dh, const float* __restrict__ dcn, int* __restrict__ tile_counter,
                    __nv_bfloat16* __restrict__ dzp, size_t dzp_stride, int dzp_lo, float* __restrict__ db_partial) {
  // dzp != NULL: dL/dgx leaves as the bf16 operand planes of the tensor-core GEMMs ([hi|lo][cap][8H], plane stride
  // dzp_stride elements, lo plane only if dzp_lo) instead of fp32 into `gates`, and the column sums of every tile (the
  // bias gradient) go to db_partial[tile][8H] -- fixed summation order, so the result does not depend on which cluster
  // ran the tile.
  using G = ::G<CL>;
  constexpr int MT = G::MT, UPC = G::UPC, UPW = G::UPW, NTW = G::NTW;
  const int H = HC ? HC : H_arg;                                   // HC: see lstm_fwd_tm_kernel
  constexpr int PITCH = G::BPITCH, WP = G::BWPITCH, RP = G::RPITCH;
  constexpr int NTH = G::NT;                                       // threads of the CTA
  constexpr int NCOPY = NTH - G::CT;                               // copy threads: 16 chunk lanes x RSLOT row slots
  constexpr int RSLOT = NCOPY / 16, RPT = MT / RSLOT;              // row slots, rows per copy thread (4 x 8)
  constexpr int NTWB = G::NTWB;                                    // n8 tiles of the warp with the most
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* Wsm = smem_raw;                                   // [2 planes][B_NSM x 8 units][WP] swizzled  (B operand of the shared-memory tile)
  unsigned char* Zsm = Wsm + 2 * G::B_W7_PLANE;                    // [2 planes][MT][PITCH]          (A operand: dz)
  unsigned char* Rsm = Zsm + 2 * G::B_Z_PLANE;                     // [CL sources][MT][40] fp32 partial dh from each CTA
  unsigned char* Ssm = Rsm + G::B_RECV;                            // [CL owners][MT][40]  fp32 partials staged for the bulk copies
  unsigned char* Stg = Ssm + G::B_RECV;                            // [B_NARR][MT][SROW] staging tile
  int* s_row = reinterpret_cast<int*>(Stg + G::B_NARR * G::SARR);
  int* s_len = s_row + MT;
  int* s_off = s_len + MT;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cluster_id = blockIdx.x / CL;
  const int dir = cluster_id & 1;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int q = lane & 3, r8 = lane >> 2;
  const int R = r8 + 8 * q;
  const int unit0 = rank * UPC + w * UPW;

  // phase 2 tiling: 5 CL n8 tiles of output units over 4 warps (G::NTILE); tile nt of warp w exists iff active(nt)
  const int nt0 = w * G::BASE + min(w, G::EXTRA);
  auto active = [&](int nt) { return nt < G::BASE || w < G::EXTRA; };
  // W slice (bf16 hi / lo): row n = hidden unit k of the OUTPUT dh, column kk = own gate column in
  // (warp, gate, unit) order -- the order phase 1 writes dz in.  Ghost gate columns and ghost output units are zero.
  const float* W = w_hh + (size_t)dir * 4 * H * H;
  auto wval = [&](int kk, int n) -> float {
    const int ww = kk / 40, rem = kk - ww * 40, g = rem / UPW, i = rem - g * UPW;
    const int unit = rank * UPC + ww * UPW + i;
    return (unit < H && n < H) ? W[(size_t)(g * H + unit) * H + n] : 0.f;
  };
  // -> TENSOR MEMORY, already in mma.sync B-fragment form.  Lane l of compute warp w (TMEM lanes 32 w + l) keeps, for every
  // k-step ks and each of the warp's first B_NTM n8 tiles nt, the registers b0 = W^T[16 ks + 2 (l % 4) + {0, 1}][n], b1 = the
  // same 8 further along k, n = 8 (nt0 + nt) + l / 4, as bf16 hi and lo: columns (ks * B_NTM + nt) * 4 + {0: hi b0, 1: hi b1,
  // 2: lo b0, 3: lo b1}.  With CL = 5 warp 0's seventh tile (units 48..55) stays in shared memory.
  __shared__ uint32_t tmem_slot;
  if (w == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr_u32(&tmem_slot)), "n"(G::B_TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tm_w = tmem_slot + ((uint32_t)((w & 3) * 32) << 16);   // this warp's lane quarter
  if (w < 4) {
#pragma unroll 1
    for (int ks = 0; ks < G::BKS; ++ks) {
#pragma unroll 1
      for (int nt = 0; nt < G::B_NTM; ++nt) {
        const int n = 8 * (nt0 + nt) + (lane >> 2);
        const int k0 = 16 * ks + 2 * (lane & 3);
        uint32_t h0, l0, h1, l1;
        split2<false>(wval(k0, n), wval(k0 + 1, n), h0, l0);
        split2<false>(wval(k0 + 8, n), wval(k0 + 9, n), h1, l1);
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(tm_w + (uint32_t)((ks * G::B_NTM + nt) * 4)), "r"(h0),
                     "r"(h1), "r"(l0), "r"(l1)
                     : "memory");
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  for (int idx = tid; idx < G::B_NSM * G::BK * 8; idx += NTH) {   // units 8 B_NTM .. 8 B_NTM + 7 (warp 0's seventh n-tile)
    const int kk = idx >> 3, r = idx & 7;
    uint16_t hi, lo;
    split1<false>(wval(kk, 8 * G::B_NTM + r), hi, lo);
    const size_t o = (size_t)r * WP + (((kk >> 3) ^ ((r >> 1) & 3)) << 4) + (kk & 7) * 2;
    *reinterpret_cast<uint16_t*>(Wsm + o) = hi;
    *reinterpret_cast<uint16_t*>(Wsm + G::B_W7_PLANE + o) = lo;
  }
  __shared__ __align__(8) uint64_t rbar[2];
  __shared__ int s_tile;
  uint64_t* rfull = &rbar[0];      // the CL partial slices for the next iteration have landed in my recv
  uint64_t* rfree = &rbar[1];      // every CTA of the cluster has consumed ITS recv (CL arrivals)
  const uint32_t w_local = smem_addr_u32(Wsm), z_local = smem_addr_u32(Zsm), r_local = smem_addr_u32(Rsm), s_local = smem_addr_u32(Ssm);
  const uint32_t stg_local = smem_addr_u32(Stg);
  const uint32_t rfull_local = smem_addr_u32(rfull), rfree_local = smem_addr_u32(rfree);
  if (tid == 0) {
    lbar_init(rfull, 1);
    lbar_init(rfree, CL);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  cluster_arrive();      // all CTAs of the cluster are running before the first remote shared-memory store (see the forward kernel)
  cluster_wait();
  uint32_t ph_full = 0u, ph_free = 0u;
  const size_t GS = (size_t)2 * 4 * H;
  PROF_DECL

  const uint32_t a_off = (uint32_t)((lane & 15) * PITCH + (lane >> 4) * 16);
  // B of the shared-memory tile: row = lane & 7, logical chunk 2ks + kh, physical chunk = logical ^ ((row >> 1) & 3)
  const uint32_t b_row6 = (uint32_t)((lane & 7) * WP);
  const uint32_t b_kh = (uint32_t)((lane >> 3) & 1), b_x = (uint32_t)((lane & 7) >> 1);
  const bool copy_role = w >= 4;                                 // warps 4-5 move the staging tile to / from global memory
  const int c_ch = tid & 15, c_rs = (tid - G::CT) >> 4;
  const uint32_t c_so = (uint32_t)(c_rs * G::SROW + c_ch * 16);
  const bool ch_ok = c_ch < 10 && rank * UPC + c_ch * 4 < H;     // the chunk's 4 units are all real or all ghost (H % 4 == 0)
  const bool leader = (tid == 96);                               // barrier / copy-engine duties (a warp with the fewest n-tiles)

  for (;;) {
    if (rank == 0 && tid == 0) {
      int t = atomicAdd(&tile_counter[dir], 1);
#pragma unroll
      for (int d = 0; d < CL; ++d) *cluster.map_shared_rank(&s_tile, d) = t;
    }
    cluster_arrive();
    cluster_wait();
    const int tile = s_tile;
    if (tile >= ntiles) break;
    __syncthreads();
    if (tid < MT) {
      int i = tile * MT + tid;
      int rr = (i < N) ? order[i] : -1;
      s_row[tid] = rr;
      s_len[tid] = (rr >= 0) ? len[rr] : 0;
      s_off[tid] = (rr >= 0) ? off[rr] : 0;
    }
    __syncthreads();
    int maxlen = 0;
    for (int i = 0; i < MT; ++i) maxlen = max(maxlen, s_len[i]);
    const int rlen = s_len[R], roff = s_off[R], rrow = s_row[R];
    if (copy_role) {
      // ---- copy warps: the activated gates and dh of iteration s-1 come into the staging tile, dL/dgx of iteration s
      // goes out, with the same chunk mapping as the forward kernel
      int c_len[RPT], c_off[RPT];         // rows c_rs + RSLOT * rr of the tile
#pragma unroll
      for (int rr = 0; rr < RPT; ++rr) { c_len[rr] = s_len[c_rs + RSLOT * rr]; c_off[rr] = s_off[c_rs + RSLOT * rr]; }
      auto prefetch_stash = [&](int s1) {
        if (ch_ok) {
#pragma unroll
          for (int rr = 0; rr < RPT; ++rr) {
            if (s1 < c_len[rr]) {
              const int t = dir ? (c_len[rr] - 1 - s1) : s1;
              const size_t p = (size_t)c_off[rr] + t;
              const float* g1 = gates + p * GS + (size_t)dir * 4 * H + rank * UPC + c_ch * 4;
#pragma unroll
              for (int a = 0; a < 4; ++a) cp_async16(stg_local + c_so + rr * RSLOT * G::SROW + a * G::SARR, g1 + a * H);
              cp_async16(stg_local + c_so + rr * RSLOT * G::SROW + 4 * G::SARR, dh + p * 2 * H + (size_t)dir * H + rank * UPC + c_ch * 4);
            }
          }
        }
        cp_async_commit();
        cp_async_wait_all();
        bar_arrive(3, NTH);
      };
      prefetch_stash(maxlen - 1);
      float csum[4][4];                  // column sums of this thread's 4 gates x 4 units over its rows and all steps
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) csum[a][j] = 0.f;
      for (int s = maxlen - 1; s >= 0; --s) {
        bar_sync(2, NTH);              // the staging tile holds dL/dgx of iteration s
        if (ch_ok) {
#pragma unroll
          for (int rr = 0; rr < RPT; ++rr) {
            if (s < c_len[rr]) {
              const int t = dir ? (c_len[rr] - 1 - s) : s;
              const size_t p = (size_t)c_off[rr] + t;
              const unsigned char* spc = Stg + c_so + rr * RSLOT * G::SROW;
              const size_t go = p * GS + (size_t)dir * 4 * H + rank * UPC + c_ch * 4;
              if (dzp) {
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                  const float4 v = *reinterpret_cast<const float4*>(spc + a * G::SARR);
                  csum[a][0] += v.x; csum[a][1] += v.y; csum[a][2] += v.z; csum[a][3] += v.w;
                  // same rounding as tc_split_store4 (gemm_tc.cu): hi = rn(x), lo = rn(x - hi)
                  const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y), h23 = __floats2bfloat162_rn(v.z, v.w);
                  __nv_bfloat16* o = dzp + go + a * H;
                  uint2 hv;
                  hv.x = *reinterpret_cast<const uint32_t*>(&h01); hv.y = *reinterpret_cast<const uint32_t*>(&h23);
                  *reinterpret_cast<uint2*>(o) = hv;
                  if (dzp_lo) {
                    const __nv_bfloat162 l01 = __floats2bfloat162_rn(v.x - __low2float(h01), v.y - __high2float(h01));
                    const __nv_bfloat162 l23 = __floats2bfloat162_rn(v.z - __low2float(h23), v.w - __high2float(h23));
                    uint2 lv;
                    lv.x = *reinterpret_cast<const uint32_t*>(&l01); lv.y = *reinterpret_cast<const uint32_t*>(&l23);
                    *reinterpret_cast<uint2*>(o + dzp_stride) = lv;
                  }
                }
              } else {
                float* g0 = gates + go;
#pragma unroll
                for (int a = 0; a < 4; ++a) *reinterpret_cast<float4*>(g0 + a * H) = *reinterpret_cast<const float4*>(spc + a * G::SARR);
              }
            }
          }
        }
        if (s > 0) prefetch_stash(s - 1);
      }
      if (dzp) {
        // per-tile column sums: the RSLOT row-slot threads of a column group are combined through the (now idle) staging
        // tile in slot order
        float* scr = reinterpret_cast<float*>(Stg);
        bar_sync(4, NCOPY);      // every copy warp is done reading the staging tile
        if (c_ch < 10) {
#pragma unroll
          for (int a = 0; a < 4; ++a)
            *reinterpret_cast<float4*>(scr + c_rs * G::COLS + a * UPC + c_ch * 4) = make_float4(csum[a][0], csum[a][1], csum[a][2], csum[a][3]);
        }
        bar_sync(4, NCOPY);
        for (int col = tid - G::CT; col < G::COLS; col += NCOPY) {
          float sum = 0.f;
#pragma unroll
          for (int rs = 0; rs < RSLOT; ++rs) sum += scr[rs * G::COLS + col];
          const int a = col / UPC, u = col - a * UPC;
          if (rank * UPC + u < H) db_partial[(size_t)tile * GS + (size_t)dir * 4 * H + a * H + rank * UPC + u] = sum;
        }
      }
      continue;
    }

    // ---- compute warps ---------------------------------------------------------------------------------------------
    float dcc[UPW];       // dL/dc carried to the previous step
    float2 ccur[NTW];     // c_t of the current iteration (= the c_{t-1} read one iteration earlier)
#pragma unroll
    for (int i = 0; i < UPW; ++i) dcc[i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < NTW; ++nt) ccur[nt] = make_float2(0.f, 0.f);

    for (int s = maxlen - 1; s >= 0; --s) {
      PROF_MARK(5)
      // c_{t-1} of this lane's row and units, straight from global memory (in flight during the wait below)
      float2 p_cp[NTW];
#pragma unroll
      for (int nt = 0; nt < NTW; ++nt) p_cp[nt] = make_float2(0.f, 0.f);
      if (s < rlen) {
        const int t = dir ? (rlen - 1 - s) : s;
        const size_t p = (size_t)roff + t;
        if (s > 0) {
          const float* cpp = c_stash + ((dir ? p + 1 : p - 1) * 2 + dir) * H + unit0;
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt)
            if (unit0 + 2 * nt < H) p_cp[nt] = *reinterpret_cast<const float2*>(cpp + 2 * nt);
        }
        if (s == rlen - 1) {          // first iteration of the row: its c_t has not been seen as a c_{t-1} yet
          const float* cp = c_stash + (p * 2 + dir) * H + unit0;
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt)
            if (unit0 + 2 * nt < H) ccur[nt] = *reinterpret_cast<const float2*>(cp + 2 * nt);
        }
      }
      PROF_MARK(0)
      if (s < maxlen - 1) { lbar_wait_cluster(rfull, ph_full); ph_full ^= 1u; }   // partials of iteration s+1 landed
      bar_sync(3, NTH);            // the copy warps have fetched the stash of iteration s
      PROF_MARK(1)
      // ---- phase 1: d(pre-activations) of this lane's row and ten units ---------------------------------------
      {
        float dz[4][UPW];
        unsigned char* sp = Stg + R * G::SROW + w * (UPW * 4);
        if (s < rlen) {
          float dht[UPW];
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt) {
            const float2 v = *reinterpret_cast<const float2*>(sp + 4 * G::SARR + nt * 8);
            dht[2 * nt] = v.x; dht[2 * nt + 1] = v.y;
          }
          if (s == rlen - 1) {       // the row's last step: start of its backward recursion
            const float* d0 = dcn + (size_t)rrow * 2 * H + (size_t)dir * H + unit0;
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) {
              const float2 v = unit0 + 2 * nt < H ? *reinterpret_cast<const float2*>(d0 + 2 * nt) : make_float2(0.f, 0.f);
              dcc[2 * nt] = v.x; dcc[2 * nt + 1] = v.y;
            }
          } else {                   // recurrent part: the CL partials summed in fixed order
            // unit u of row r sits at column (u + 10 (r >> 2)) % 40 of its block: without the rotation the 32 row owners
            // of a warp hit 4 bank groups (8-way conflicts), with it 16
            const float* rv = reinterpret_cast<const float*>(Rsm + (size_t)R * RP);
            const int rot = w * UPW + 10 * (R >> 2);
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) {
              float2 acc2 = make_float2(0.f, 0.f);
              const int col = (rot + 2 * nt) % UPC;
#pragma unroll
              for (int src = 0; src < CL; ++src) {
                const float2 v = *reinterpret_cast<const float2*>(rv + (size_t)src * MT * (RP / 4) + col);
                acc2.x += v.x; acc2.y += v.y;
              }
              dht[2 * nt] += acc2.x; dht[2 * nt + 1] += acc2.y;
            }
          }
#pragma unroll
          for (int nt = 0; nt < NTW; ++nt) {
            const float2 ig = *reinterpret_cast<const float2*>(sp + 0 * G::SARR + nt * 8);
            const float2 fg = *reinterpret_cast<const float2*>(sp + 1 * G::SARR + nt * 8);
            const float2 gg = *reinterpret_cast<const float2*>(sp + 2 * G::SARR + nt * 8);
            const float2 og = *reinterpret_cast<const float2*>(sp + 3 * G::SARR + nt * 8);
            const float iv[2] = {ig.x, ig.y}, fv[2] = {fg.x, fg.y}, gv[2] = {gg.x, gg.y}, ov[2] = {og.x, og.y};
            const float cv[2] = {ccur[nt].x, ccur[nt].y}, cpv[2] = {p_cp[nt].x, p_cp[nt].y};
            const bool live = unit0 + 2 * nt < H;   // ghost units: dz = dc = 0 exactly
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int i = 2 * nt + u;
              const float tc = fast_tanh(cv[u]);
              const float dc = dcc[i] + dht[i] * ov[u] * (1.f - tc * tc);
              dz[3][i] = live ? dht[i] * tc * ov[u] * (1.f - ov[u]) : 0.f;
              dz[0][i] = live ? dc * gv[u] * iv[u] * (1.f - iv[u]) : 0.f;
              dz[2][i] = live ? dc * iv[u] * (1.f - gv[u] * gv[u]) : 0.f;
              dz[1][i] = live ? dc * cpv[u] * fv[u] * (1.f - fv[u]) : 0.f;
              dcc[i] = live ? dc * fv[u] : 0.f;
            }
            ccur[nt] = p_cp[nt];
          }
          // dL/dgx of this step goes back into the staging tile (stored to global memory cooperatively below)
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) *reinterpret_cast<float2*>(sp + g * G::SARR + nt * 8) = make_float2(dz[g][2 * nt], dz[g][2 * nt + 1]);
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int i = 0; i < UPW; ++i) dz[g][i] = 0.f;
        }
        // dz -> A operand (bf16 hi / lo), 40 consecutive k' = (gate, unit) of this warp: 5 x 16 B per plane
        if (s > 0) {
          uint32_t hi[20], lo[20];
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt) split2<false>(dz[g][2 * nt], dz[g][2 * nt + 1], hi[g * 5 + nt], lo[g * 5 + nt]);
          uint4* zh = reinterpret_cast<uint4*>(Zsm + (size_t)R * PITCH + w * 80);
          uint4* zl = reinterpret_cast<uint4*>(Zsm + G::B_Z_PLANE + (size_t)R * PITCH + w * 80);
#pragma unroll
          for (int c = 0; c < 5; ++c) {
            zh[c] = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            zl[c] = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
          }
        }
      }
      PROF_MARK(2)
      bar_sync(1, G::CT);   // dz tile complete; every compute thread has consumed its recv values
      if (leader && s > 0) {
        lbar_expect_tx(rfull, G::B_TX);                                             // arm for the partials of iteration s
#pragma unroll
        for (int d = 0; d < CL; ++d) rbar_arrive_relaxed(mapa_u32(rfree_local, d));  // "my recv may be overwritten"
      }
      bar_arrive(2, NTH);  // hand the staging tile (dL/dgx of iteration s) to the copy warps
      if (s == 0) break;
      PROF_MARK(3)
      // ---- phase 2: partial dh_{t-1}[32 x units of this warp's n-tiles] = dz[32 x 160] x W_slice --------------
      float acc[2][NTWB][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < NTWB; ++nt)
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
      {   // the fragments live only in this block: with their lifetime left open, CL = 4 compiles to a different register schedule
        // A fragments (dz, shared memory) double-buffered in registers; B fragments of one k-step from tensor memory
        // (4 B_NTM registers: B_NTM tiles x {hi b0, hi b1, lo b0, lo b1}), the seventh tile of warp 0 (CL = 5) from shared memory
        struct FragA { uint32_t ah[2][4], al[2][4]; };
        auto load_a = [&](FragA& f, int ks) {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            ldsm_x4(z_local + a_off + mt * 16 * PITCH + ks * 32, f.ah[mt][0], f.ah[mt][1], f.ah[mt][2], f.ah[mt][3]);
            if (!SINGLE)
              ldsm_x4(z_local + G::B_Z_PLANE + a_off + mt * 16 * PITCH + ks * 32, f.al[mt][0], f.al[mt][1], f.al[mt][2], f.al[mt][3]);
          }
        };
        auto step = [&](const FragA& fa, int ks) {
          constexpr int NTM = G::B_NTM;
          uint32_t r[4 * NTM], b6h[2] = {0u, 0u}, b6l[2] = {0u, 0u};
          tm_ld<4 * NTM>(r, tm_w + (uint32_t)(ks * 4 * NTM));
          if (G::B_NSM > 0 && active(NTM)) {
            const uint32_t bc = (((uint32_t)(2 * ks) + b_kh) ^ b_x) << 4;
            ldsm_x2(w_local + b_row6 + bc, b6h[0], b6h[1]);
            if (!SINGLE) ldsm_x2(w_local + G::B_W7_PLANE + b_row6 + bc, b6l[0], b6l[1]);
          }
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (!SINGLE) {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
              for (int nt = 0; nt < NTM; ++nt)
                if (active(nt)) mma16816<false>(acc[mt][nt], fa.al[mt], r[4 * nt], r[4 * nt + 1]);
              if (G::B_NSM > 0 && active(NTM)) mma16816<false>(acc[mt][NTWB - 1], fa.al[mt], b6h[0], b6h[1]);
            }
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
              for (int nt = 0; nt < NTM; ++nt)
                if (active(nt)) mma16816<false>(acc[mt][nt], fa.ah[mt], r[4 * nt + 2], r[4 * nt + 3]);
              if (G::B_NSM > 0 && active(NTM)) mma16816<false>(acc[mt][NTWB - 1], fa.ah[mt], b6l[0], b6l[1]);
            }
          }
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
            for (int nt = 0; nt < NTM; ++nt)
              if (active(nt)) mma16816<false>(acc[mt][nt], fa.ah[mt], r[4 * nt], r[4 * nt + 1]);
            if (G::B_NSM > 0 && active(NTM)) mma16816<false>(acc[mt][NTWB - 1], fa.ah[mt], b6h[0], b6h[1]);
          }
        };
        FragA a0, a1;
        load_a(a0, 0);
#pragma unroll
        for (int ks = 0; ks < G::BKS; ks += 2) {
          load_a(a1, ks + 1);
          step(a0, ks);
          if (ks + 2 < G::BKS) load_a(a0, ks + 2);
          step(a1, ks + 1);
        }
      }
      PROF_MARK(4)
      // rfree: every CTA has finished reading its recv -> it may be overwritten; it also tells that every peer has
      // received the partials of the previous iteration, i.e. the copy engine is done with the staging tile
      lbar_wait_cluster(rfree, ph_free);
      ph_free ^= 1u;
      PROF_MARK(6)
#pragma unroll
      for (int nt = 0; nt < NTWB; ++nt) {
        if (active(nt)) {
          const int k = 8 * (nt0 + nt) + 2 * q;          // output hidden unit of acc[..][nt][0]
          const int owner = k / UPC, kl = k - owner * UPC;
          unsigned char* dst = Ssm + (size_t)owner * G::B_RBLK;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            const int ra = 16 * mt + r8, rb = ra + 8;      // rotated columns, see the reader in phase 1
            *reinterpret_cast<float2*>(dst + ra * RP + ((kl + 10 * (ra >> 2)) % UPC) * 4) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
            *reinterpret_cast<float2*>(dst + rb * RP + ((kl + 10 * (rb >> 2)) % UPC) * 4) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
          }
        }
      }
      bar_sync(1, G::CT);   // partials staged (also: every warp is done with the dz tile before the next phase 1 rewrites it)
      PROF_MARK(7)
      if (leader) {
        fence_proxy_async_smem();
#pragma unroll
        for (int d = 0; d < CL; ++d) {
          const int owner = (rank + d) % CL;
          bulk_copy_to_peer(mapa_u32(r_local + (uint32_t)(rank * G::B_RBLK), owner), s_local + (uint32_t)(owner * G::B_RBLK), G::B_RBLK,
                            mapa_u32(rfull_local, owner));
        }
      }
    }
  }
  PROF_FLUSH(8)
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (w == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_slot), "n"(G::B_TM_COLS) : "memory");
  cluster_arrive();
  cluster_wait();
}

template <int CL, class K>
int launch_cluster(K kernel, size_t smem, int ntiles, cudaStream_t st, void** args, const char* name, int (*cache_tab)[16],
                   bool (*attr_tab)[16], int variant) {
  int dev = 0;
  NNR_CUDA(cudaGetDevice(&dev));
  dev &= 15;                                  // the attribute and the occupancy are per device (and per instantiation)
  int* cache = &cache_tab[variant][dev];
  bool* attr_set = &attr_tab[variant][dev];
  if (!*attr_set) {
    NNR_CUDA(cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // all of the L1 / shared-memory array as shared memory: without it the driver sizes the carve-out for ONE CTA (85 KB
    // forward) and the second CTA per SM never becomes resident (measured: 26 clusters either way)
    NNR_CUDA(cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    *attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cfg.blockDim = dim3(G<CL>::NT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  if (*cache == 0) {
    cfg.gridDim = dim3(CL * 2);
    int nc = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&nc, (const void*)kernel, &cfg);
    if (e != cudaSuccess || nc < 2) { (void)cudaGetLastError(); nc = 24; }
    // Two CTAs per SM: the occupancy query does not see that the 85 KB CTAs fit twice (it answers 1 CTA / SM = 26 clusters
    // on B200, with or without the shared-memory carve-out hint), the hardware does co-schedule them.  Measured on B200,
    // N = 3520, L = 128 forward: 26 clusters 4.67 ms, 40: 4.09, 52: 3.50, 56: 3.43, 58: 3.32, 64: 3.45, 72: 3.40 -> 2 nc + 6.
    // Clusters beyond what fits start late, find the tile counter exhausted and exit.  The rule was measured at CL = 5
    // (hidden_dim 200); the smaller clusters of other hidden sizes and the BPTT kernel use it unchanged.
    *cache = (2 * nc + 6) & ~1;
    if (getenv("NNR_LSTM_DEBUG")) {
      int bps = -1;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, (const void*)kernel, G<CL>::NT, smem);
      fprintf(stderr, "[nnr lstm] %s: threads %d smem %zu -> occupancy %d CTAs/SM, max active clusters %d (query rc %d), using %d\n", name,
              G<CL>::NT, smem, bps, nc, (int)e, *cache);
    }
  }
  int want = 2 * ntiles;                      // (tile, direction) pairs
  int nclusters = want < *cache ? want : *cache;
  if (nclusters < 2) nclusters = 2;
  cfg.gridDim = dim3(nclusters * CL);
  cudaError_t e = cudaLaunchKernelExC(&cfg, (const void*)kernel, args);
  nnr_count_launch(1);
  if (e != cudaSuccess) { nnr_set_error("%s: launch failed: %s", name, cudaGetErrorString(e)); return (int)e; }
  return 0;
}

}  // namespace

#ifdef NNR_LSTM_PROF
extern "C" int nnr_debug_lstm_prof(unsigned long long* out16) {
  cudaDeviceSynchronize();
  return (int)cudaMemcpyFromSymbol(out16, g_lstm_prof, 16 * sizeof(unsigned long long));
}
#endif
int nnr_lstm_mma_max_clusters = 0;   // co-resident clusters of the last forward launch (cudaOccupancyMaxActiveClusters)
extern "C" int nnr_debug_lstm_clusters(void) { return nnr_lstm_mma_max_clusters; }
extern "C" int nnr_gemm_default_algo(void);
// the reduced-precision ("bf16") variant of BASELINE config 4: NNR_GEMM_ALGO=bf16 selects single-product tensor-core GEMMs and,
// here, ONE 16-bit product per recurrent step instead of the three split products
static int nnr_lstm_single_product() {
  static int v = -1;
  if (v < 0) v = (nnr_gemm_default_algo() == NNR_GEMM_TC_BF16) ? 1 : 0;
  return v;
}

// zero rows [ntok, round_up(ntok, 64)) of operand planes written by a producer kernel: the k tail MN-major GEMM tiles read
__global__ void planes_zero_tail_kernel(__nv_bfloat16* __restrict__ pl, size_t stride, int nplanes, int cols, int cap,
                                        const int32_t* __restrict__ ntok_dev) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
  const int ntok = min(*ntok_dev, cap);
  const int r1 = min(cap, (ntok + 63) / 64 * 64);
  const int c8 = cols / 8;                                     // 16-byte groups per row
  const long long total = (long long)(r1 - ntok) * c8 * nplanes;
  for (long long i = gt; i < total; i += nthreads) {
    const int p = (int)(i / ((long long)(r1 - ntok) * c8));
    const long long rem = i - (long long)p * (r1 - ntok) * c8;
    const int r = ntok + (int)(rem / c8), c = (int)(rem % c8) * 8;
    *reinterpret_cast<uint4*>(pl + (size_t)p * stride + (size_t)r * cols + c) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// CTAs per cluster for hidden size H (0 < H <= 200): 40 units per CTA, at least two CTAs
static int lstm_cluster_size(int H) { return H <= 80 ? 2 : (H + 39) / 40; }

// per-instantiation slots of the occupancy / attribute caches: [CL - 2] for a run-time H, [4] for hidden_dim 200
static int lstm_kernel_slot(int H) { return H == 200 ? 4 : lstm_cluster_size(H) - 2; }

template <int CL, int HC>
static int lstm_fwd_tm_launch(void** args, int ntiles, cudaStream_t st, int single, int (*cache)[16], bool (*attr_set)[16]) {
  return single ? launch_cluster<CL>(lstm_fwd_tm_kernel<true, CL, HC>, G<CL>::FWD_SMEM, ntiles, st, args, "lstm_fwd_tm_kernel<single>", cache, attr_set, 1)
                : launch_cluster<CL>(lstm_fwd_tm_kernel<false, CL, HC>, G<CL>::FWD_SMEM, ntiles, st, args, "lstm_fwd_tm_kernel", cache, attr_set, 0);
}

// 0 < H <= 200 and H % 4 == 0; h_planes needs H = 200 (lstm.cu checks)
int nnr_lstm_fwd_mma(float* gx, const float* w_hh, const int32_t* len, const int32_t* off, const int32_t* order, int N, int H,
                     float* h_out, float* c_stash, float* c_n, int32_t* tile_counters, cudaStream_t st, void* h_planes,
                     size_t plane_stride, int two_planes, int cap) {
  static int cache[5][2][16] = {};     // [lstm_kernel_slot][single][device]
  static bool attr_set[5][2][16] = {};
  const int CL = lstm_cluster_size(H), slot = lstm_kernel_slot(H);
  int ntiles = (N + G<5>::MT - 1) / G<5>::MT;
  NNR_CUDA(cudaMemsetAsync(tile_counters, 0, 2 * sizeof(int32_t), st));
  const int single = nnr_lstm_single_product();
  __nv_bfloat16* hp = (__nv_bfloat16*)h_planes;
  void* args[] = {&gx, &w_hh, &len, &off, &order, &N, &H, &ntiles, &h_out, &c_stash, &c_n, &tile_counters, &hp, &plane_stride, &two_planes};
  int rc;
  switch (CL) {
    case 2: rc = lstm_fwd_tm_launch<2, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    case 3: rc = lstm_fwd_tm_launch<3, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    case 4: rc = lstm_fwd_tm_launch<4, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    default:
      rc = H == 200 ? lstm_fwd_tm_launch<5, 200>(args, ntiles, st, single, cache[slot], attr_set[slot])
                    : lstm_fwd_tm_launch<5, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]);
      break;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  nnr_lstm_mma_max_clusters = cache[slot][single][dev & 15];
  if (rc || !hp) return rc;
  planes_zero_tail_kernel<<<32, 256, 0, st>>>(hp, plane_stride, two_planes ? 2 : 1, 2 * H, cap, off + N);
  nnr_count_launch(1);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { nnr_set_error("planes_zero_tail_kernel: launch failed: %s", cudaGetErrorString(e)); return (int)e; }
  return 0;
}

// column sums of dL/dgx = the per-tile partials added in tile order; the same launch zeroes the plane rows
// [ntok, round_up(ntok, 64)) that the MN-major tiles of the weight-gradient GEMMs read
__global__ void lstm_dz_finish_kernel(const float* __restrict__ db_partial, int ntiles, int cols, float* __restrict__ db,
                                      __nv_bfloat16* __restrict__ dzp, size_t dzp_stride, int nplanes, int cap,
                                      const int32_t* __restrict__ ntok_dev) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
  if (gt < cols) {
    float s = 0.f;
    for (int t = 0; t < ntiles; ++t) s += db_partial[(size_t)t * cols + gt];
    db[gt] = s;
  }
  const int ntok = min(*ntok_dev, cap);
  const int r1 = min(cap, (ntok + 63) / 64 * 64);
  const int c8 = cols / 8;                                     // 16-byte groups per row
  const long long total = (long long)(r1 - ntok) * c8 * nplanes;
  for (long long i = gt; i < total; i += nthreads) {
    const int pl = (int)(i / ((long long)(r1 - ntok) * c8));
    const long long rem = i - (long long)pl * (r1 - ntok) * c8;
    const int r = ntok + (int)(rem / c8), c = (int)(rem % c8) * 8;
    *reinterpret_cast<uint4*>(dzp + (size_t)pl * dzp_stride + (size_t)r * cols + c) = make_uint4(0u, 0u, 0u, 0u);
  }
}

template <int CL, int HC>
static int lstm_bwd_tm_launch(void** args, int ntiles, cudaStream_t st, int single, int (*cache)[16], bool (*attr_set)[16]) {
  return single ? launch_cluster<CL>(lstm_bwd_mma_kernel<true, CL, HC>, G<CL>::BWD_SMEM, ntiles, st, args, "lstm_bwd_tm_kernel<single>", cache, attr_set, 1)
                : launch_cluster<CL>(lstm_bwd_mma_kernel<false, CL, HC>, G<CL>::BWD_SMEM, ntiles, st, args, "lstm_bwd_tm_kernel", cache, attr_set, 0);
}

// 0 < H <= 200 and H % 4 == 0; dz_planes needs H = 200 (lstm.cu checks)
int nnr_lstm_bwd_mma(float* gates, const float* c_stash, const float* w_hh, const int32_t* len, const int32_t* off,
                     const int32_t* order, int N, int H, const float* dh, const float* dcn, int32_t* tile_counters, cudaStream_t st,
                     void* dz_planes, size_t plane_stride, int two_planes, float* db_partial, float* db, int cap) {
  static int cache[5][2][16] = {};     // [lstm_kernel_slot][single][device]
  static bool attr_set[5][2][16] = {};
  const int CL = lstm_cluster_size(H), slot = lstm_kernel_slot(H);
  int ntiles = (N + G<5>::MT - 1) / G<5>::MT;
  NNR_CUDA(cudaMemsetAsync(tile_counters, 0, 2 * sizeof(int32_t), st));
  __nv_bfloat16* dzp = (__nv_bfloat16*)dz_planes;
  void* args[] = {&gates, &c_stash, &w_hh, &len, &off, &order, &N, &H, &ntiles, &dh, &dcn, &tile_counters,
                  &dzp, &plane_stride, &two_planes, &db_partial};
  const int single = nnr_lstm_single_product();
  int rc;
  switch (CL) {
    case 2: rc = lstm_bwd_tm_launch<2, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    case 3: rc = lstm_bwd_tm_launch<3, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    case 4: rc = lstm_bwd_tm_launch<4, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]); break;
    default:
      rc = H == 200 ? lstm_bwd_tm_launch<5, 200>(args, ntiles, st, single, cache[slot], attr_set[slot])
                    : lstm_bwd_tm_launch<5, 0>(args, ntiles, st, single, cache[slot], attr_set[slot]);
      break;
  }
  if (rc || !dz_planes) return rc;
  const int cols = 8 * H;
  lstm_dz_finish_kernel<<<(cols + 255) / 256 * 4, 256, 0, st>>>(db_partial, ntiles, cols, db, dzp, plane_stride, two_planes ? 2 : 1, cap, off + N);
  nnr_count_launch(1);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { nnr_set_error("lstm_dz_finish_kernel: launch failed: %s", cudaGetErrorString(e)); return (int)e; }
  return 0;
}
