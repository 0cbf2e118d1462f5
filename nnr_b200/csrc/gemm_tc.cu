// tcgen05 / TMEM / TMA GEMM backend of nnr_gemm (sm_100a).
//
//   C[M,N] = epi( op(A)[M,K] * op(B)[K,N] )      fp32 in, fp32 out, fp32-grade accuracy
//
// Arithmetic: split operands.  Every fp32 operand x is split into hi and lo = round(x - hi) planes and
// D += A_hi*B_hi + A_hi*B_lo + A_lo*B_hi runs on the 5th-generation tensor cores with fp32 accumulation in TMEM:
//   NNR_GEMM_TC_BF16X3 (default)  bf16 hi / lo planes, tcgen05.mma kind::f16  -- measured 6e-6 of max|C|
//   NNR_GEMM_TC_TF32X3            tf32 hi / lo planes, tcgen05.mma kind::tf32 -- 4e-6 (K=400) ... 1.1e-5 (K=1600)
//   NNR_GEMM_TC_BF16              one bf16 plane (the reduced-precision variant)
// What remains of the error comes from the tensor core truncating when it adds into the TMEM accumulator, so long
// contractions (wgrad: K = tokens) are cut into chains of <= 2048 k whose partial sums are combined in a fixed order
// in exact fp32.
//
// Structure
//   pre-pass   tc_split_kernel: row-major operand -> planes [hi|lo][rows][cols] in the workspace (elementwise,
//              16-byte accesses); zero-fills the column pad and, for device-bounded row counts, the row tail.
//              No transposes: an operand whose contraction index runs along its ROWS (dgrad weights, both
//              wgrad operands) is consumed MN-major straight from the same row-major planes.
//   main       persistent kernel, one CTA per SM, static round-robin over (m-tile, n-tile, k-split) with the
//              valid tile count computed on the device from m_dev / k_dev (no host synchronisation):
//     warp 0     TMA producer: cp.async.bulk.tensor.3d (SWIZZLE_128B) of A_hi, A_lo, B_hi, B_lo for one 128-byte
//                (64 bf16 / 32 tf32) k-block into a ring of shared-memory stages; mbarrier expect_tx completion.
//     warp 1     TMEM allocator (512 columns = two accumulators) and single-thread tcgen05.mma issuer:
//                12 MMAs per stage (4 k-steps x 3 split products), tcgen05.commit frees the stage / publishes
//                the accumulator.
//     warps 2-9  epilogue (two warps per TMEM lane quarter, half the columns each): tcgen05.ld one accumulator row per
//                thread, 32x16 transpose through a per-warp shared-memory tile, then fused bias / tanh / relu+residual
//                (+dropout) / sigmoid-gate / add with coalesced 16-byte global accesses; overlaps the next tile's main
//                loop (double-buffered TMEM).
//   CTA pairs  row counts >= 2*128*148 run 256-row tiles on 2-CTA clusters (tcgen05.mma.cta_group::2): each CTA loads its
//              128 rows of A and half of the B tile, the leader issues the MMAs for both (see the PAIR template flag).
//   split-K    partials + a deterministic fixed-order reduce.
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include <cuda.h>
#include <cuda_bf16.h>

extern "C" int nnr_gemm_default_algo(void);

#define TC_BM 128
#define TC_THREADS 320        // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quarter)
#define TC_TMEM_COLS 512
#define TC_ACC_COLS 256
#define TC_EPI_PITCH 80       // bytes per row of an epilogue warp's 32 x 16 fp32 transpose tile (conflict-free 16 B accesses)
#define TC_EPI_SCRATCH (8 * 32 * TC_EPI_PITCH)
#define TC_SMEM_BUDGET (205 * 1024)   // pipeline stages; + TC_EPI_SCRATCH + alignment slack + barriers <= 227 KB
#define TC_CHAIN_K 2048      // max contraction length accumulated in TMEM before an fp32 combine (split-K GEMMs); 1024 and 2048 give the same gradient error tables (profiles/r2_parity_config2.md), 2048 halves the partial traffic

// ------------------------------------------------------------------------------------------------
// device helpers (raw PTX)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint64_t* bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
template <bool BF16>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if (BF16) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
        "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
        "r"(accumulate)
        : "memory");
  }
}
// ---- CTA-pair (cta_group::2) variants: one 256 x BLOCK_N tile per pair of SMs; each CTA loads its own 128 rows of A
// and HALF of the B tile, the leader CTA issues the MMAs for both, so every SM ingests A + B/2 per k-block ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the bytes land in THIS CTA's shared memory but are counted on the LEADER's full barrier
__device__ __forceinline__ void tma_load_3d_pair(const CUtensorMap* map, uint32_t leader_bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// arrives on the barrier at the same shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
template <bool BF16>
__device__ __forceinline__ void tc_mma_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if (BF16) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
        "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
        "r"(accumulate)
        : "memory");
  }
}

// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives row (lane base + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// sm_100 shared-memory matrix descriptor, SWIZZLE_128B (layout type 2), version 1.
//   K-major : rows of 128 B, 8-row groups SBO = 1024 B apart, LBO unused.
//   MN-major: atoms of 8 k-rows x 128 B (one TMA box row each); k-groups SBO = 1024 B apart, successive
//             groups of 128 B along M/N are LBO bytes apart (= one TMA box).
//   MN-major TF32 is special: the only legal layout is SWIZZLE_128B_BASE32B (layout type 1: 32-byte chunks
//             swizzled within 128 B, TMA mode SWIZZLE_128B_ATOM_32B), whose atom holds 4 k-rows -> SBO = 512 B.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}

// optional in-kernel phase stamps (clock64 of CTA 0), compiled in with -DNNR_TC_PROF; read back with nnr_debug_tc_prof
#ifdef NNR_TC_PROF
__device__ unsigned long long g_tc_prof[16];
#define TC_STAMP(i) { if (blockIdx.x == 0) g_tc_prof[i] = clock64(); }
#else
#define TC_STAMP(i) {}
#endif

struct TcParams {
  int M, N, K;                 // capacities
  const int32_t* m_dev;
  const int32_t* k_dev;
  int block_n, stages, nplanes;
  int a_mn, b_mn;              // operand is MN-major (contraction index along its rows)
  int split_k;                 // 0: one pass over all of K;  1: chains of chain_kb k-blocks, partials
  int chain_kb;
  uint32_t idesc;
  float* partial;
  int epi_fast;                // N % 4 == 0 and every epilogue pointer / leading dimension 16-byte aligned: straight-line float4 path
  __nv_bfloat16* c_planes;     // optional: the result also as bf16 operand planes [hi|lo][c_prows][c_pitch] (fast epilogue only)
  long long c_pitch, c_pstride;   // row pitch and plane stride in elements
  int c_lo, c_rows;            // write the lo plane (split algos); rows of the planes
  EpiP epi;
};

__device__ __forceinline__ bool al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }

// ---- epilogue over 4 consecutive columns of one row (the coalesced layout: a quad of lanes covers 64 contiguous
// bytes of a row, a warp instruction 8 rows x 64 B), cnt = valid columns (N tail) --------------------------------
__device__ __forceinline__ void ld4(const float* p, int cnt, float* o) {
  if (cnt == 4 && al16(p)) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = (i < cnt) ? __ldg(p + i) : 0.f;
  }
}
__device__ __forceinline__ void st4(float* p, int cnt, const float* o) {
  if (cnt == 4 && al16(p)) {
    *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) if (i < cnt) p[i] = o[i];
  }
}
// The epilogue of one 4-column item is split in a load part and a finish part so that the loads of the four items a
// lane handles per chunk are all in flight before the first store (a store would otherwise fence the next item's loads).
struct Epi4In { float rb[4], ax[4], cc[4]; };
__device__ __forceinline__ void epi_load4(const EpiP& e, int m, int n, int cnt, Epi4In& in, int rmap) {
  if (e.epilogue == NNR_EPI_GATE) {
    ld4(e.rowbias + (size_t)rmap * e.ldrowbias + n, cnt, in.rb);     // rmap = rowmap[m], loaded once per tile by the caller
    ld4(e.aux + (size_t)m * e.ldaux + n, cnt, in.ax);
  } else if (e.epilogue == NNR_EPI_ADD_AUX || (e.epilogue == NNR_EPI_BIAS_RELU_RES && e.aux)) {
    ld4(e.aux + (size_t)m * e.ldaux + n, cnt, in.ax);
  }
  if (e.accumulate) ld4(e.C + (size_t)m * e.ldc + n, cnt, in.cc);
}
__device__ __forceinline__ void epi_finish4(const EpiP& e, int m, int n, float* v, int cnt, const float* bias4, const Epi4In& in) {
  if (e.epilogue == NNR_EPI_BIAS || e.epilogue == NNR_EPI_BIAS_TANH || e.epilogue == NNR_EPI_BIAS_RELU_RES) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += bias4[i];
  }
  if (e.epilogue == NNR_EPI_BIAS_TANH) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = tanh_fast(v[i]);
  } else if (e.epilogue == NNR_EPI_BIAS_RELU_RES) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = fmaxf(v[i], 0.f);
    if (e.aux_out) st4(e.aux_out + (size_t)m * e.ldaux_out + n, cnt, v);
    if (e.aux) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] += in.ax[i];
    }
    if (e.p_drop > 0.f) {
      const uint64_t seed = nnr_resolve_seed(e.seed);
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] *= dropout_scale(seed, (uint64_t)m * (uint64_t)e.N + n + i, e.p_drop, e.inv_keep);
    }
  } else if (e.epilogue == NNR_EPI_GATE) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = sigmoid_fast(v[i] + in.rb[i]);
    if (e.aux_out) st4(e.aux_out + (size_t)m * e.ldaux_out + n, cnt, v);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] *= in.ax[i];
  } else if (e.epilogue == NNR_EPI_ADD_AUX) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += in.ax[i];
  }
  if (e.accumulate) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += in.cc[i];
  }
  st4(e.C + (size_t)m * e.ldc + n, cnt, v);
}

// ---- fast epilogue of one output tile (one warp: 32 rows x its half of the tile's columns) -----------------------------
// The epilogue kind is a template parameter and every per-tile quantity is hoisted, so a 16-column chunk is a short
// straight-line sequence: the in-kernel stamps (scripts/gemm_phase_prof.py) of the run-time-switched version showed 1.1-1.4 us
// per chunk (5.5 us per 128 x 128 tile, 13 us with the relu/residual/dropout epilogue) -- more than the main loop of every
// K <= 400 token-level GEMM.  Three more things hide latency: the tcgen05.ld of chunk c+1 is issued as soon as chunk c has
// left the registers, the streamed operands (aux / C / row bias) of chunk c+1 are loaded before chunk c is finished, and the
// transpose tile is addressed in the shared state space (the generic form compiled to LD.E / ST.E).
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
// the registers pass through the wait so that no use of them is scheduled above it
__device__ __forceinline__ void tmem_ld16_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                 "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

struct EpiTile {                 // per-lane constants of one tile: the lane finishes rows row0 + 8 i, i = 0..3, in every chunk
  uint32_t o_c[4], o_aux[4], o_ao[4], o_rb[4];   // element offsets of those rows (32-bit: host-checked)
  uint32_t rvalid;               // bit i: row row0 + 8 i < M
  int row0;
};
// the streamed operands of one chunk: aux (or the old C when accumulating without aux), the gate's row bias, the bias
template <int EP>
__device__ __forceinline__ void epi_load_in(const TcParams& p, const EpiTile& t, int n, bool has_bias, bool need_ax, bool acc_early,
                                            float4 (&ax)[4], float4 (&rb)[4], float4& bb) {
  bb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) { ax[i] = make_float4(0.f, 0.f, 0.f, 0.f); rb[i] = make_float4(0.f, 0.f, 0.f, 0.f); }
  if (n < p.N) {
    if (has_bias) bb = __ldg(reinterpret_cast<const float4*>(p.epi.bias + n));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (t.rvalid & (1u << i)) {
        if (need_ax) ax[i] = __ldg(reinterpret_cast<const float4*>(p.epi.aux + t.o_aux[i] + n));
        else if (acc_early) ax[i] = *reinterpret_cast<const float4*>(p.epi.C + t.o_c[i] + n);
        if (EP == NNR_EPI_GATE) rb[i] = __ldg(reinterpret_cast<const float4*>(p.epi.rowbias + t.o_rb[i] + n));
      }
    }
  }
}

#define TC_EPK_PARTIAL 6      // kernel-template value: the tile is one split-K partial (plain store into the partial slices)
template <int EP>
__device__ __forceinline__ void epi_tile_fast(const TcParams& p, const EpiTile& t, uint32_t lane_addr, bool has_k, int c_begin, int c_end,
                                              int n0, uint32_t tile_s, int lane, int M, uint64_t drop_seed, float* __restrict__ Cout) {
  const int tr = lane >> 2, tc4 = (lane & 3) * 4;
  constexpr bool PARTIAL = EP == TC_EPK_PARTIAL;
  constexpr bool BIASED = EP == NNR_EPI_BIAS || EP == NNR_EPI_BIAS_TANH || EP == NNR_EPI_BIAS_RELU_RES;
  const bool has_bias = BIASED && p.epi.bias != nullptr;
  const bool need_ax = EP == NNR_EPI_GATE || EP == NNR_EPI_ADD_AUX || (EP == NNR_EPI_BIAS_RELU_RES && p.epi.aux != nullptr);
  const bool accumulate = !PARTIAL && p.epi.accumulate != 0;
  const bool acc_early = accumulate && !need_ax;      // one streamed operand per row lives in registers: aux, else the old C
  const bool planes = !PARTIAL && p.c_planes != nullptr;
  const bool drop = EP == NNR_EPI_BIAS_RELU_RES && p.epi.p_drop > 0.f;
  const uint32_t my_row = tile_s + (uint32_t)lane * TC_EPI_PITCH;
  const uint32_t rd_row = tile_s + (uint32_t)tr * TC_EPI_PITCH + (uint32_t)tc4 * 4;

  // the gate epilogue streams two operands per row (aux and the row bias: 32 registers per chunk): its inputs are loaded at
  // the top of their own chunk (under the tcgen05.ld wait and the transpose) instead of one chunk ahead -- the second set
  // would not fit the 168 registers a 320-thread CTA leaves per thread
  constexpr bool AHEAD = EP != NNR_EPI_GATE;
  uint32_t r[16];
  float4 ax[4], rb[4], bb, axn[4], rbn[4], bbn;
  if (has_k) tmem_ld16_issue(lane_addr + (uint32_t)c_begin, r);
  if (AHEAD) epi_load_in<EP>(p, t, n0 + c_begin + tc4, has_bias, need_ax, acc_early, ax, rb, bb);
  for (int c0 = c_begin; c0 < c_end; c0 += 16) {
    const bool more = c0 + 16 < c_end;
    if (AHEAD) { if (more) epi_load_in<EP>(p, t, n0 + c0 + 16 + tc4, has_bias, need_ax, acc_early, axn, rbn, bbn); }
    else epi_load_in<EP>(p, t, n0 + c0 + tc4, has_bias, need_ax, acc_early, ax, rb, bb);
    if (has_k) tmem_ld16_wait(r);
    else {
#pragma unroll
      for (int i = 0; i < 16; ++i) r[i] = 0u;
    }
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) sts128(my_row + qd * 16, r[4 * qd], r[4 * qd + 1], r[4 * qd + 2], r[4 * qd + 3]);
    if (has_k && more) tmem_ld16_issue(lane_addr + (uint32_t)(c0 + 16), r);
    __syncwarp();
    float4 o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = lds128(rd_row + (uint32_t)(8 * i) * TC_EPI_PITCH);
    const int n = n0 + c0 + tc4;
    if (n < p.N) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (!(t.rvalid & (1u << i))) continue;
        float4 v = make_float4(o[i].x + bb.x, o[i].y + bb.y, o[i].z + bb.z, o[i].w + bb.w);
        if (EP == NNR_EPI_BIAS_TANH) {
          v.x = tanh_fast(v.x); v.y = tanh_fast(v.y); v.z = tanh_fast(v.z); v.w = tanh_fast(v.w);
        } else if (EP == NNR_EPI_BIAS_RELU_RES) {
          v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
          if (p.epi.aux_out) *reinterpret_cast<float4*>(p.epi.aux_out + t.o_ao[i] + n) = v;
          if (need_ax) { v.x += ax[i].x; v.y += ax[i].y; v.z += ax[i].z; v.w += ax[i].w; }
          if (drop) {
            // N % 4 == 0 and n % 4 == 0 on this path: the four elements are one quad of the mask, one hash
            const uint64_t e0 = (uint64_t)(t.row0 + 8 * i) * (uint64_t)p.epi.N + n;
            float ks[4];
            dropout_scale4(drop_seed, e0 >> 2, p.epi.p_drop, p.epi.inv_keep, ks);
            v.x *= ks[0]; v.y *= ks[1]; v.z *= ks[2]; v.w *= ks[3];
          }
        } else if (EP == NNR_EPI_GATE) {
          v.x = sigmoid_fast(v.x + rb[i].x); v.y = sigmoid_fast(v.y + rb[i].y);
          v.z = sigmoid_fast(v.z + rb[i].z); v.w = sigmoid_fast(v.w + rb[i].w);
          if (p.epi.aux_out) *reinterpret_cast<float4*>(p.epi.aux_out + t.o_ao[i] + n) = v;
          v.x *= ax[i].x; v.y *= ax[i].y; v.z *= ax[i].z; v.w *= ax[i].w;
        } else if (EP == NNR_EPI_ADD_AUX) {
          v.x += ax[i].x; v.y += ax[i].y; v.z += ax[i].z; v.w += ax[i].w;
        }
        if (acc_early) { v.x += ax[i].x; v.y += ax[i].y; v.z += ax[i].z; v.w += ax[i].w; }
        else if (accumulate) {
          const float4 cc = *reinterpret_cast<const float4*>(Cout + t.o_c[i] + n);
          v.x += cc.x; v.y += cc.y; v.z += cc.z; v.w += cc.w;
        }
        *reinterpret_cast<float4*>(Cout + t.o_c[i] + n) = v;
        if (planes) {               // same rounding as tc_split_store4: hi = rn(x), lo = rn(x - hi)
          const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y), h23 = __floats2bfloat162_rn(v.z, v.w);
          __nv_bfloat16* op = p.c_planes + (long long)(t.row0 + 8 * i) * p.c_pitch + n;
          uint2 hv;
          hv.x = *reinterpret_cast<const uint32_t*>(&h01); hv.y = *reinterpret_cast<const uint32_t*>(&h23);
          *reinterpret_cast<uint2*>(op) = hv;
          if (p.c_lo) {
            const __nv_bfloat162 l01 = __floats2bfloat162_rn(v.x - __low2float(h01), v.y - __high2float(h01));
            const __nv_bfloat162 l23 = __floats2bfloat162_rn(v.z - __low2float(h23), v.w - __high2float(h23));
            uint2 lv;
            lv.x = *reinterpret_cast<const uint32_t*>(&l01); lv.y = *reinterpret_cast<const uint32_t*>(&l23);
            *reinterpret_cast<uint2*>(op + p.c_pstride) = lv;
          }
        }
      }
      if (planes) {                 // rows [M, round_up(M, 64)) of the planes are the zero tail an MN-major consumer reads
        const int mz = min(p.c_rows, (M + 63) & ~63);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int mm = t.row0 + 8 * i;
          if (mm >= M && mm < mz) {
            __nv_bfloat16* op = p.c_planes + (long long)mm * p.c_pitch + n;
            *reinterpret_cast<uint2*>(op) = make_uint2(0u, 0u);
            if (p.c_lo) *reinterpret_cast<uint2*>(op + p.c_pstride) = make_uint2(0u, 0u);
          }
        }
      }
    }
    __syncwarp();
    if (AHEAD && more) {
      bb = bbn;
#pragma unroll
      for (int i = 0; i < 4; ++i) { ax[i] = axn[i]; rb[i] = rbn[i]; }
    }
  }
}

// EPK >= 0: the epilogue kind, fixed at compile time (fast path: the host guarantees p.epi_fast, no split-K partials);
// EPK = -1: the run-time-switched epilogue that takes any alignment, N tail and the split-K partials
template <bool BF16, bool PAIR, int EPK>
__global__ void __launch_bounds__(TC_THREADS, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                const __grid_constant__ CUtensorMap map_b, TcParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int KELEM = BF16 ? 64 : 32;                 // elements per 128 bytes = k-block depth = MN group width
  constexpr int TILE_M = PAIR ? 2 * TC_BM : TC_BM;      // output rows per scheduled tile (a CTA always owns 128 of them)
  int M = p.M, K = p.K;
  if (p.m_dev) M = min(M, *p.m_dev);
  if (p.k_dev) K = min(K, *p.k_dev);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) TC_STAMP(0)
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs of the pair)
  const int sched_id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int sched_n = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int b_rows = PAIR ? (p.block_n >> 1) : p.block_n;   // rows of the B tile this CTA holds

  // ---- tile space (device-side effective sizes) ----
  const int m_tiles = (M + TILE_M - 1) / TILE_M;
  const int n_tiles = (p.N + p.block_n - 1) / p.block_n;
  const int nkb = (K + KELEM - 1) / KELEM;
  const int kb_per = p.split_k ? p.chain_kb : max(nkb, 1);
  const int splits = p.split_k ? max(1, (nkb + kb_per - 1) / kb_per) : 1;
  const int total_tiles = m_tiles * n_tiles * splits;

  // ---- smem carve-up ----
  const uint32_t a_tile = TC_BM * 128, b_tile = (uint32_t)b_rows * 128;
  const uint32_t stage_bytes = (uint32_t)p.nplanes * (a_tile + b_tile);       // multiples of 1024
  unsigned char* tiles = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char* epi_scratch = tiles + (size_t)p.stages * stage_bytes;          // [8 epilogue warps][32][TC_EPI_PITCH]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_scratch + TC_EPI_SCRATCH);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tmem_full = empty_bar + p.stages;      // [2]
  uint64_t* tmem_empty = tmem_full + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], PAIR ? 16 : 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (PAIR) cluster_sync_all();         // the peer's barriers exist before anything is signalled across the pair
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TC_STAMP(1)

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int it = 0;
      for (int tile = sched_id; tile < total_tiles; tile += sched_n) {
        const int n_idx = tile % n_tiles, rest = tile / n_tiles;
        const int m0 = (rest % m_tiles) * TILE_M + (int)rank * TC_BM, n0 = n_idx * p.block_n + (int)rank * b_rows, z = rest / m_tiles;
        const int kb0 = z * kb_per, kb1 = min(nkb, kb0 + kb_per);
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          const uint32_t base = smem_u32(tiles + (size_t)s * stage_bytes);
          if (!PAIR) mbar_expect_tx(&full_bar[s], stage_bytes);
          else if (rank == 0) mbar_expect_tx(&full_bar[s], 2 * stage_bytes);      // both CTAs' loads complete on the leader's barrier
          const uint32_t lbar = PAIR ? mapa_rank(smem_u32(&full_bar[s]), 0) : 0u;
          auto load_a = [&](uint32_t dst, int c0, int c1, int c2) {
            if (PAIR) tma_load_3d_pair(&map_a, lbar, dst, c0, c1, c2); else tma_load_3d(&map_a, &full_bar[s], dst, c0, c1, c2);
          };
          auto load_b = [&](uint32_t dst, int c0, int c1, int c2) {
            if (PAIR) tma_load_3d_pair(&map_b, lbar, dst, c0, c1, c2); else tma_load_3d(&map_b, &full_bar[s], dst, c0, c1, c2);
          };
          for (int pl = 0; pl < p.nplanes; ++pl) {
            const uint32_t sa = base + pl * a_tile;
            const uint32_t sb = base + p.nplanes * a_tile + pl * b_tile;
            if (!p.a_mn) load_a(sa, kb * KELEM, m0, pl);
            else for (int g = 0; g < TC_BM / KELEM; ++g) load_a(sa + g * (KELEM * 128), m0 + g * KELEM, kb * KELEM, pl);
            if (!p.b_mn) load_b(sb, kb * KELEM, n0, pl);
            else for (int g = 0; g < b_rows / KELEM; ++g) load_b(sb + g * (KELEM * 128), n0 + g * KELEM, kb * KELEM, pl);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (in a CTA pair: the leader only, for both CTAs) =====
    if (lane == 0 && rank == 0) {
      int it = 0, tl = 0;
      const uint32_t lbo = KELEM * 128;                               // bytes of one MN-group box
      const uint64_t a_step = p.a_mn ? (uint64_t)((BF16 ? 2048 : 1024) >> 4) : 2;   // descriptor advance per MMA
      const uint64_t b_step = p.b_mn ? (uint64_t)((BF16 ? 2048 : 1024) >> 4) : 2;
      for (int tile = sched_id; tile < total_tiles; tile += sched_n, ++tl) {
        const int rest = tile / n_tiles;
        const int z = rest / m_tiles;
        const int kb0 = z * kb_per, kb1 = min(nkb, kb0 + kb_per);
        const int buf = tl & 1;
        mbar_wait(&tmem_empty[buf], ((tl >> 1) & 1) ^ 1);              // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * TC_ACC_COLS;
        uint32_t first = 1;
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % p.stages;
          mbar_wait(&full_bar[s], (it / p.stages) & 1);
          tc_fence_after();
          if (it == 0) TC_STAMP(2)
          const uint32_t base = smem_u32(tiles + (size_t)s * stage_bytes);
          // MN-major fp32 operands use the BASE32B layout (type 1, 4-row atoms); everything else plain SW128
          const uint32_t a_lt = (p.a_mn && !BF16) ? 1u : 2u, a_sbo = (p.a_mn && !BF16) ? 512u : 1024u;
          const uint32_t b_lt = (p.b_mn && !BF16) ? 1u : 2u, b_sbo = (p.b_mn && !BF16) ? 512u : 1024u;
          const uint64_t a_hi = make_sw128_desc(base, p.a_mn ? lbo : 0, a_sbo, a_lt);
          const uint64_t a_lo = make_sw128_desc(base + a_tile, p.a_mn ? lbo : 0, a_sbo, a_lt);
          const uint64_t b_hi = make_sw128_desc(base + p.nplanes * a_tile, p.b_mn ? lbo : 0, b_sbo, b_lt);
          const uint64_t b_lo = make_sw128_desc(base + p.nplanes * a_tile + b_tile, p.b_mn ? lbo : 0, b_sbo, b_lt);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t ao = a_step * k, bo = b_step * k;
            if (PAIR) tc_mma_pair<BF16>(d_tmem, a_hi + ao, b_hi + bo, p.idesc, first ? 0u : 1u);
            else tc_mma<BF16>(d_tmem, a_hi + ao, b_hi + bo, p.idesc, first ? 0u : 1u);
            first = 0;
            if (p.nplanes == 2) {           // split operands: the two cross products (lo*lo is below fp32 resolution)
              if (PAIR) {
                tc_mma_pair<BF16>(d_tmem, a_hi + ao, b_lo + bo, p.idesc, 1u);
                tc_mma_pair<BF16>(d_tmem, a_lo + ao, b_hi + bo, p.idesc, 1u);
              } else {
                tc_mma<BF16>(d_tmem, a_hi + ao, b_lo + bo, p.idesc, 1u);
                tc_mma<BF16>(d_tmem, a_lo + ao, b_hi + bo, p.idesc, 1u);
              }
            }
          }
          if (PAIR) tc_commit_pair(&empty_bar[s]); else tc_commit(&empty_bar[s]);     // frees the stage in both CTAs
        }
        if (tl < 2) TC_STAMP(3 + tl)
        if (PAIR) tc_commit_pair(&tmem_full[buf]); else tc_commit(&tmem_full[buf]);
      }
    }
  } else {
    // ===== epilogue: warps 2..9; warp % 4 selects the TMEM lane quarter, (warp-2)/4 the column half =====
    const int q = warp & 3;
    const int chalf = (warp - 2) >> 2;
    const uint64_t drop_seed = (p.epi.p_drop > 0.f) ? nnr_resolve_seed(p.epi.seed) : 0ull;
    const int nchunks = p.block_n >> 4;
    const int c_begin = chalf ? ((nchunks + 1) >> 1) << 4 : 0;
    const int c_end = chalf ? p.block_n : ((nchunks + 1) >> 1) << 4;
    int tl = 0;
    for (int tile = sched_id; tile < total_tiles; tile += sched_n, ++tl) {
      const int n_idx = tile % n_tiles, rest = tile / n_tiles;
      const int m0 = (rest % m_tiles) * TILE_M + (int)rank * TC_BM, n0 = n_idx * p.block_n, z = rest / m_tiles;
      const int kb0 = z * kb_per, kb1 = min(nkb, kb0 + kb_per);
      const int buf = tl & 1;
      const uint32_t lane_addr = tmem_base + buf * TC_ACC_COLS + ((uint32_t)(q * 32) << 16);
      // Each thread reads one accumulator row (tcgen05.ld 32x32b), the warp transposes 32 x 16 chunks through its
      // shared-memory tile, and all global traffic of the epilogue (C, aux, row bias, accumulate) then runs in the
      // coalesced layout: lane -> (row = lane / 4 + 8 i, 4 columns = 4 (lane % 4)), 64 contiguous bytes per row.
      unsigned char* my_tile = epi_scratch + (size_t)(warp - 2) * 32 * TC_EPI_PITCH;
      const int tr = lane >> 2, tc4 = (lane & 3) * 4;
      // a lane finishes the same four rows in every chunk of the tile: their row-map entries (gate epilogue) are fetched
      // once, before the accumulator is waited for, so the row-bias loads of the chunks are not behind a dependent load
      int rmap[4] = {0, 0, 0, 0};
      if ((EPK < 0 || EPK == NNR_EPI_GATE) && p.epi.epilogue == NNR_EPI_GATE && !p.partial) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int mm = m0 + q * 32 + tr + 8 * i;
          if (mm < M) rmap[i] = __ldg(p.epi.rowmap + mm);
        }
      }
      // fast path: the four rows a lane finishes are the same in every chunk of the tile -> their element offsets once per
      // tile (32-bit: the host enables the path only when every operand has fewer than 2^32 elements)
      const bool fast = EPK >= 0;
      uint32_t o_c[4], o_aux[4], o_ao[4], o_rb[4];
      uint32_t rvalid = 0;
      if (fast) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int mm = m0 + q * 32 + tr + 8 * i;
          if (mm < M) rvalid |= 1u << i;
          const uint32_t mr = (mm < M) ? (uint32_t)mm : 0u;
          o_c[i] = (EPK == TC_EPK_PARTIAL) ? ((uint32_t)z * (uint32_t)M + mr) * (uint32_t)p.N : mr * (uint32_t)p.epi.ldc;
          o_aux[i] = mr * (uint32_t)p.epi.ldaux;
          o_ao[i] = mr * (uint32_t)p.epi.ldaux_out;
          o_rb[i] = (uint32_t)rmap[i] * (uint32_t)p.epi.ldrowbias;
        }
      }
      mbar_wait(&tmem_full[buf], (tl >> 1) & 1);
      tc_fence_after();
      if (warp == 2 && lane == 0 && tl < 2) TC_STAMP(5 + 2 * tl)
      if (EPK >= 0) {
        EpiTile et;
#pragma unroll
        for (int i = 0; i < 4; ++i) { et.o_c[i] = o_c[i]; et.o_aux[i] = o_aux[i]; et.o_ao[i] = o_ao[i]; et.o_rb[i] = o_rb[i]; }
        et.rvalid = rvalid; et.row0 = m0 + q * 32 + tr;
        epi_tile_fast<(EPK >= 0 ? EPK : 0)>(p, et, lane_addr, kb1 > kb0, c_begin, c_end, n0, smem_u32(my_tile), lane, M, drop_seed,
                                            EPK == TC_EPK_PARTIAL ? p.partial : p.epi.C);
      } else
      for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        float v[16];
        if (kb1 > kb0) tmem_ld16(lane_addr + (uint32_t)c0, v);
        else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0.f;
        }
#pragma unroll
        for (int qd = 0; qd < 4; ++qd)
          *reinterpret_cast<float4*>(my_tile + lane * TC_EPI_PITCH + qd * 16) = make_float4(v[4 * qd], v[4 * qd + 1], v[4 * qd + 2], v[4 * qd + 3]);
        __syncwarp();
        const int n = n0 + c0 + tc4;
        const int cnt = min(4, p.N - n);
        float o[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 x = *reinterpret_cast<const float4*>(my_tile + (tr + 8 * i) * TC_EPI_PITCH + tc4 * 4);
          o[i][0] = x.x; o[i][1] = x.y; o[i][2] = x.z; o[i][3] = x.w;
        }
        if (cnt > 0) {
          if (p.partial) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int mm = m0 + q * 32 + tr + 8 * i;
              if (mm < M) st4(p.partial + ((size_t)z * M + mm) * p.N + n, cnt, o[i]);
            }
          } else {
            Epi4In in[4];
            float bias4[4] = {0.f, 0.f, 0.f, 0.f};
            if (p.epi.bias && (p.epi.epilogue == NNR_EPI_BIAS || p.epi.epilogue == NNR_EPI_BIAS_TANH || p.epi.epilogue == NNR_EPI_BIAS_RELU_RES))
              ld4(p.epi.bias + n, cnt, bias4);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int mm = m0 + q * 32 + tr + 8 * i;
              if (mm < M) epi_load4(p.epi, mm, n, cnt, in[i], rmap[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int mm = m0 + q * 32 + tr + 8 * i;
              if (mm < M) epi_finish4(p.epi, mm, n, o[i], cnt, bias4, in[i]);
            }
          }
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (warp == 2 && lane == 0 && tl < 2) TC_STAMP(6 + 2 * tl)
      if (lane == 0) {
        if (PAIR && rank != 0) mbar_arrive_cluster(mapa_rank(smem_u32(&tmem_empty[buf]), 0));   // the leader's MMA warp waits for both CTAs
        else mbar_arrive(&tmem_empty[buf]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) TC_STAMP(9)
  if (PAIR) cluster_sync_all();         // no CTA leaves while its peer may still read its operands / signal its barriers
  if (warp == 1) {
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
  }
}

// deterministic combine of the split-K partials (number of active splits is recomputed from k_dev)
__global__ void tc_splitk_reduce_kernel(const float* __restrict__ partial, int K, const int32_t* __restrict__ k_dev, int kelem,
                                        int chain_kb, int M, int N, const int32_t* __restrict__ m_dev, EpiP epi) {
  if (m_dev) M = min(M, *m_dev);
  if (k_dev) K = min(K, *k_dev);
  const int nkb = (K + kelem - 1) / kelem;
  const int splits = max(1, (nkb + chain_kb - 1) / chain_kb);
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * N) return;
  int m = (int)(i / N), n = (int)(i - (size_t)m * N);
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += partial[((size_t)s * M + m) * N + n];
  epi_store(epi, m, n, acc);
}
// N % 4 == 0: a thread combines four adjacent outputs with 16-byte loads, four splits in flight; the splits are added in
// the same ascending order as above (same bits), the epilogue is the 4-wide one of the main kernel
__global__ void __launch_bounds__(256) tc_splitk_reduce4_kernel(const float* __restrict__ partial, int K, const int32_t* __restrict__ k_dev,
                                                                int kelem, int chain_kb, int M, int N, const int32_t* __restrict__ m_dev,
                                                                EpiP epi) {
  if (m_dev) M = min(M, *m_dev);
  if (k_dev) K = min(K, *k_dev);
  const int nkb = (K + kelem - 1) / kelem;
  const int splits = max(1, (nkb + chain_kb - 1) / chain_kb);
  const int N4 = N >> 2;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * N4) return;
  const int m = (int)(i / N4), n = (int)(i - (size_t)m * N4) * 4;
  const size_t plane = (size_t)M * N;
  const float* src = partial + (size_t)m * N + n;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int s = 0;
  for (; s + 4 <= splits; s += 4) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const float4*>(src + (size_t)(s + u) * plane));
#pragma unroll
    for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
  for (; s < splits; ++s) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + (size_t)s * plane));
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  float o[4] = {acc.x, acc.y, acc.z, acc.w};
  float bias4[4] = {0.f, 0.f, 0.f, 0.f};
  if (epi.bias && (epi.epilogue == NNR_EPI_BIAS || epi.epilogue == NNR_EPI_BIAS_TANH || epi.epilogue == NNR_EPI_BIAS_RELU_RES))
    ld4(epi.bias + n, 4, bias4);
  Epi4In in;
  epi_load4(epi, m, n, 4, in, epi.epilogue == NNR_EPI_GATE ? __ldg(epi.rowmap + m) : 0);
  epi_finish4(epi, m, n, o, 4, bias4, in);
}

// ------------------------------------------------------------------------------------------------
// pre-pass: row-major X[R, C] (ld) -> planes.  TF32: fp32 [2][R][Cp] (hi, lo).  BF16: bf16 [1][R][Cp].
// Columns [C, Cp) are written as zeros; with r_dev, rows [R_eff, round_up(R_eff, 64)) are zeros too (they
// are the k tail of an MN-major operand) and rows beyond are left untouched.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
template <int MODE>   // 0: fp32 planes (rna_tf32 hi, lo)   1: one bf16 plane   2: bf16 hi, lo planes
__global__ void __launch_bounds__(256) tc_split_kernel(const float* __restrict__ src, int64_t ld, int R, int C, int Cp,
                                                       const int32_t* __restrict__ r_dev, bool vec, void* __restrict__ out,
                                                       size_t plane_stride) {
  int Rv = R;
  if (r_dev) Rv = min(R, *r_dev);
  const int Rw = r_dev ? min(R, (Rv + 63) / 64 * 64) : R;
  const int cq_per_row = Cp >> 2;                                   // float4 groups per row
  const long long total = (long long)Rw * cq_per_row;
  const long long stride = (long long)gridDim.x * blockDim.x;
  // grid-stride over (row, 4-column group); four independent 16-byte loads in flight per thread
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += 4 * stride) {
    float4 x[4];
    int rr[4], cc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = i0 + u * stride;
      x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      rr[u] = -1;
      if (i < total) {
        const int r = (int)(i / cq_per_row), cq = (int)(i - (long long)r * cq_per_row) * 4;
        rr[u] = r; cc[u] = cq;
        if (r < Rv) {
          const float* sp = src + (size_t)r * ld + cq;
          if (vec && cq + 3 < C) x[u] = __ldg(reinterpret_cast<const float4*>(sp));
          else {
            if (cq < C) x[u].x = __ldg(sp);
            if (cq + 1 < C) x[u].y = __ldg(sp + 1);
            if (cq + 2 < C) x[u].z = __ldg(sp + 2);
            if (cq + 3 < C) x[u].w = __ldg(sp + 3);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (rr[u] < 0) continue;
      if (MODE >= 1) {
        __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(out) + (size_t)rr[u] * Cp + cc[u];
        __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(ob);
        const __nv_bfloat162 h01 = __floats2bfloat162_rn(x[u].x, x[u].y), h23 = __floats2bfloat162_rn(x[u].z, x[u].w);
        o[0] = h01;                                                  // Cp % 8 == 0 -> 8-byte aligned
        o[1] = h23;
        if (MODE == 2) {
          __nv_bfloat162* l = reinterpret_cast<__nv_bfloat162*>(ob + plane_stride);
          l[0] = __floats2bfloat162_rn(x[u].x - __low2float(h01), x[u].y - __high2float(h01));
          l[1] = __floats2bfloat162_rn(x[u].z - __low2float(h23), x[u].w - __high2float(h23));
        }
      } else {
        float* hi = reinterpret_cast<float*>(out) + (size_t)rr[u] * Cp + cc[u];
        float4 h, l;
        h.x = rna_tf32(x[u].x); h.y = rna_tf32(x[u].y); h.z = rna_tf32(x[u].z); h.w = rna_tf32(x[u].w);
        l.x = rna_tf32(x[u].x - h.x); l.y = rna_tf32(x[u].y - h.y); l.z = rna_tf32(x[u].z - h.z); l.w = rna_tf32(x[u].w - h.w);
        *reinterpret_cast<float4*>(hi) = h;
        *reinterpret_cast<float4*>(hi + plane_stride) = l;
      }
    }
  }
}

template <int MODE>
__device__ __forceinline__ void tc_split_store4(void* out, size_t plane_stride, int Cp, int r, int c, float4 x) {
  if (MODE >= 1) {
    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(out) + (size_t)r * Cp + c;
    __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(ob);
    const __nv_bfloat162 h01 = __floats2bfloat162_rn(x.x, x.y), h23 = __floats2bfloat162_rn(x.z, x.w);
    o[0] = h01;
    o[1] = h23;
    if (MODE == 2) {
      __nv_bfloat162* l = reinterpret_cast<__nv_bfloat162*>(ob + plane_stride);
      l[0] = __floats2bfloat162_rn(x.x - __low2float(h01), x.y - __high2float(h01));
      l[1] = __floats2bfloat162_rn(x.z - __low2float(h23), x.w - __high2float(h23));
    }
  } else {
    float* hi = reinterpret_cast<float*>(out) + (size_t)r * Cp + c;
    float4 h, l;
    h.x = rna_tf32(x.x); h.y = rna_tf32(x.y); h.z = rna_tf32(x.z); h.w = rna_tf32(x.w);
    l.x = rna_tf32(x.x - h.x); l.y = rna_tf32(x.y - h.y); l.z = rna_tf32(x.z - h.z); l.w = rna_tf32(x.w - h.w);
    *reinterpret_cast<float4*>(hi) = h;
    *reinterpret_cast<float4*>(hi + plane_stride) = l;
  }
}

// Split + column sums in one pass over the matrix (a bias gradient is the column sum of the same dL/dy whose planes
// feed the dgrad / wgrad GEMMs): one CTA per tcs_rows(R) rows (64, or 16 when the matrix is small so that the grid still covers the SMs); thread (rs, g) owns 4-column groups g, g + G, ... and rows
// r0 + rs, r0 + rs + RS, ...; per-CTA partial sums (row slots combined in fixed order) go to `partial`, a second
// kernel adds the partials of the valid row blocks in block order -> deterministic.
static __host__ __device__ __forceinline__ int tcs_rows(int R) { return R >= 16384 ? 64 : 16; }
#define TCS_MAXG 2            // 4-column groups per thread: C <= 2048
// PRE: the matrix is dL/d(relu output) and is first multiplied by the dropout mask of nnr_dropout (counter = r * C + c;
// the masked values are also stored to `dropped`, the residual branch needs them) and then by (relu_out > 0): the
// backward of "dropout -> relu -> Linear" without materialising either product (layers.py:286-289, userEncoders.py:91).
struct SplitPre { const float* relu_out; float* dropped; float p, inv_keep; uint64_t seed; };
template <int MODE, bool PRE>
__global__ void __launch_bounds__(256) tc_split_colsum_kernel(const float* __restrict__ src, int64_t ld, int R, int C, int Cp,
                                                              const int32_t* __restrict__ r_dev, void* __restrict__ out,
                                                              size_t plane_stride, float* __restrict__ partial, SplitPre pre) {
  __shared__ float4 s_acc[256];
  if (PRE && pre.p > 0.f) pre.seed = nnr_resolve_seed(pre.seed);
  int Rv = R;
  if (r_dev) Rv = min(R, *r_dev);
  const int Rw = r_dev ? min(R, (Rv + 63) / 64 * 64) : R;        // rows whose planes must be defined (zero tail)
  const int rpc = tcs_rows(R);
  const int r0 = blockIdx.x * rpc;
  if (r0 >= Rw) return;
  const int ncq = Cp >> 2;
  const int G = min(ncq, 256), RS = 256 / G;
  const int tid = threadIdx.x, g = tid % G, rs = tid / G;
  const bool active = rs < RS;
  float4 acc[TCS_MAXG];
#pragma unroll
  for (int j = 0; j < TCS_MAXG; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int r1 = min(r0 + rpc, Rw);
  if (active) {
    for (int rb = r0 + rs; rb < r1; rb += 4 * RS) {
      float4 x[4][TCS_MAXG];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int r = rb + u * RS;
#pragma unroll
        for (int j = 0; j < TCS_MAXG; ++j) {
          const int cq = (g + j * G) * 4;
          x[u][j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (r < r1 && r < Rv && cq < Cp) {
            const float* sp = src + (size_t)r * ld + cq;
            if (cq + 3 < C) x[u][j] = __ldg(reinterpret_cast<const float4*>(sp));
            else {
              if (cq < C) x[u][j].x = __ldg(sp);
              if (cq + 1 < C) x[u][j].y = __ldg(sp + 1);
              if (cq + 2 < C) x[u][j].z = __ldg(sp + 2);
            }
            if (PRE) {
              float* xv = reinterpret_cast<float*>(&x[u][j]);
              const size_t o = (size_t)r * ld + cq;
              float ks[4] = {1.f, 1.f, 1.f, 1.f};
              if (pre.p > 0.f) {
                const uint64_t e0 = (uint64_t)r * (uint64_t)C + cq;
                if ((e0 & 3) == 0) dropout_scale4(pre.seed, e0 >> 2, pre.p, pre.inv_keep, ks);      // one hash for the quad
                else {
#pragma unroll
                  for (int e = 0; e < 4; ++e) ks[e] = dropout_scale(pre.seed, e0 + e, pre.p, pre.inv_keep);
                }
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (cq + e < C) {
                  if (pre.p > 0.f) xv[e] *= ks[e];
                  if (pre.dropped) pre.dropped[o + e] = xv[e];
                  xv[e] *= (__ldg(pre.relu_out + o + e) > 0.f) ? 1.f : 0.f;
                }
              }
            }
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int r = rb + u * RS;
        if (r >= r1) continue;
#pragma unroll
        for (int j = 0; j < TCS_MAXG; ++j) {
          const int cq = (g + j * G) * 4;
          if (cq >= Cp) continue;
          tc_split_store4<MODE>(out, plane_stride, Cp, r, cq, x[u][j]);
          acc[j].x += x[u][j].x; acc[j].y += x[u][j].y; acc[j].z += x[u][j].z; acc[j].w += x[u][j].w;
        }
      }
    }
  }
  // combine the row slots in fixed order, one group pass at a time
  for (int j = 0; j < TCS_MAXG; ++j) {
    __syncthreads();
    if (active) s_acc[rs * G + g] = acc[j];
    __syncthreads();
    const int cq = (g + j * G) * 4;
    if (rs == 0 && cq < Cp) {
      float4 t = s_acc[g];
      for (int q = 1; q < RS; ++q) { const float4 o = s_acc[q * G + g]; t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w; }
      float* dst = partial + (size_t)blockIdx.x * Cp + cq;
      *reinterpret_cast<float4*>(dst) = t;
    }
  }
}
// out[c] = sum over the valid row blocks; 16 slices per column (slice s takes blocks s, s+16, ...) combined in slice order
__global__ void __launch_bounds__(512) tc_split_colsum_reduce(const float* __restrict__ partial, int nblocks, int R, int C, int Cp,
                                                              const int32_t* __restrict__ r_dev, float* __restrict__ out, int accumulate) {
  __shared__ float s_sum[16][33];
  const int cl = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  int Rv = R;
  if (r_dev) Rv = min(R, *r_dev);
  const int nb = min(nblocks, (Rv + tcs_rows(R) - 1) / tcs_rows(R));
  float a0 = 0.f, a1 = 0.f;
  if (c < C) {
    int b = sl;
    for (; b + 16 < nb; b += 32) { a0 += partial[(size_t)b * Cp + c]; a1 += partial[(size_t)(b + 16) * Cp + c]; }
    if (b < nb) a0 += partial[(size_t)b * Cp + c];
  }
  s_sum[sl][cl] = a0 + a1;
  __syncthreads();
  if (sl == 0 && c < C) {
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) acc += s_sum[q][cl];
    out[c] = accumulate ? out[c] + acc : acc;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    else (void)cudaGetLastError();
  }
  return fn;
}

static size_t up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct TcPlan {
  bool bf16;
  int a_mn, b_mn;               // MN-major flags
  int a_rows, a_cols, b_rows, b_cols;   // stored (row-major) shapes of the operands
  int a_cp, b_cp;               // plane pitches
  int block_n, stages, split_k, chain_kb, max_splits, nplanes, kelem;
  int pair;                     // 1: CTA-pair kernel (256-row tiles, B tile split across the pair)
  size_t a_plane, b_plane, a_off, b_off, partial_off, total, smem;
};

static int pick_block_n(int N, int step, int nplanes) {
  int best = step;
  double best_cost = 1e30;
  for (int bn = 256; bn >= 32; bn -= step) {
    double padded = (double)((N + bn - 1) / bn) * bn;
    double cost = padded * (1.0 + 40.0 / bn);
    // a two-stage ring cannot hide the TMA latency behind one stage of MMAs: prefer tiles that leave room for three
    // (measured: a two-stage ring loses more than the larger tile gains)
    size_t stage = (size_t)nplanes * ((size_t)TC_BM * 128 + (size_t)bn * 128);
    if (TC_SMEM_BUDGET / stage < 3) cost *= 1.3;
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

// CTA-pair tiles: 256 x bn with bn <= 256, bn % 16 == 0 (K-major B) or % 128 == 0 (MN-major B: each CTA holds whole 64-wide
// groups), three pipeline stages required.  Returns 0 when no such tile keeps the padding reasonable.
static int pick_block_n_pair(int N, int step, int nplanes) {
  int best = 0;
  double best_cost = 1e30;
  for (int bn = 256; bn >= 64; bn -= step) {
    size_t stage = (size_t)nplanes * ((size_t)TC_BM * 128 + (size_t)(bn / 2) * 128);
    if (TC_SMEM_BUDGET / stage < 3) continue;
    double padded = (double)((N + bn - 1) / bn) * bn;
    if (padded > 1.15 * N) continue;
    double cost = padded * (1.0 + 40.0 / bn);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

// mode: 0 = 3xTF32 (fp32 hi/lo planes), 1 = BF16 (one plane), 2 = BF16x3 (bf16 hi/lo planes)
static int algo_mode(int algo) {
  if (algo == NNR_GEMM_AUTO) algo = nnr_gemm_default_algo();
  return algo == NNR_GEMM_TC_BF16 ? 1 : (algo == NNR_GEMM_TC_BF16X3 ? 2 : 0);
}
static TcPlan make_plan(const nnr_gemm_args* a, int mode) {
  TcPlan pl;
  const bool bf16 = mode != 0;
  pl.bf16 = bf16;
  pl.kelem = bf16 ? 64 : 32;
  pl.nplanes = mode == 1 ? 1 : 2;
  pl.a_mn = a->transA ? 1 : 0;                 // A stored [K, M]: contraction along rows
  pl.b_mn = a->transB ? 0 : 1;                 // B stored [K, N]: contraction along rows
  pl.a_rows = a->transA ? a->K : a->M; pl.a_cols = a->transA ? a->M : a->K;
  pl.b_rows = a->transB ? a->N : a->K; pl.b_cols = a->transB ? a->K : a->N;
  const size_t pad = bf16 ? 8 : 4;             // 16-byte row pitch
  pl.a_cp = (int)up((size_t)pl.a_cols, pad);
  pl.b_cp = (int)up((size_t)pl.b_cols, pad);
  pl.block_n = pick_block_n(a->N, pl.b_mn ? pl.kelem : 16, pl.nplanes);
  // large row counts (token-level GEMMs) are bound by L2->SM operand delivery: use 256-row tiles on CTA pairs
  pl.pair = 0;
  if (a->M >= 2 * TC_BM * 148 && !(a->transA) && a->k_dev == nullptr) {
    int bnp = pick_block_n_pair(a->N, pl.b_mn ? 2 * pl.kelem : 16, pl.nplanes);
    if (bnp) { pl.pair = 1; pl.block_n = bnp; }
  }
  long tiles = (long)((a->M + TC_BM - 1) / TC_BM) * ((a->N + pl.block_n - 1) / pl.block_n);
  // split-K: (a) fill the machine when the output grid is small, (b) bound the TMEM accumulation chain
  int nkb_cap = (a->K + pl.kelem - 1) / pl.kelem;
  pl.split_k = 0;
  pl.chain_kb = TC_CHAIN_K / pl.kelem;
  if (!pl.pair && tiles * 2 <= 148 && nkb_cap >= 8) {   // an output grid that already fills more than half the SMs is not split
    int target = (int)((148 + tiles - 1) / tiles);
    int chain = (nkb_cap + target - 1) / target;
    if (chain < 4) chain = 4;
    if (chain > TC_CHAIN_K / pl.kelem) chain = TC_CHAIN_K / pl.kelem;
    if (chain < nkb_cap) { pl.split_k = 1; pl.chain_kb = chain; }
  }
  pl.max_splits = pl.split_k ? (nkb_cap + pl.chain_kb - 1) / pl.chain_kb : 1;
  size_t stage = (size_t)pl.nplanes * ((size_t)TC_BM * 128 + (size_t)(pl.pair ? pl.block_n / 2 : pl.block_n) * 128);
  int stages = (int)(TC_SMEM_BUDGET / stage);
  if (stages < 2) stages = 2;
  if (stages > 6) stages = 6;
  pl.stages = stages;
  pl.smem = 1024 + (size_t)stages * stage + TC_EPI_SCRATCH + (2 * stages + 4) * 8 + 16;
  const size_t esz = bf16 ? 2 : 4;
  pl.a_plane = (size_t)pl.a_rows * pl.a_cp;
  pl.b_plane = (size_t)pl.b_rows * pl.b_cp;
  size_t o = 0;
  pl.a_off = o; if (!a->A_planes) o = up(o + pl.a_plane * esz * pl.nplanes, 1024);
  pl.b_off = o; if (!a->B_planes) o = up(o + pl.b_plane * esz * pl.nplanes, 1024);
  pl.partial_off = o;
  if (pl.split_k) o = up(o + (size_t)pl.max_splits * a->M * a->N * sizeof(float), 1024);
  pl.total = o;
  return pl;
}

int nnr_gemm_tc_supported(const nnr_gemm_args* a) {
  if (!get_encode()) return 0;
  // tiny problems are launch-bound either way; the FFMA kernel handles them exactly
  // (an operand that exists only as planes cannot go there, so it stays on this path whatever the size)
  if ((double)a->M * a->N * a->K < 2.0e6 && a->A && a->B) return 0;
  if (a->K < 8) return 0;
  // device-side bounds: m_dev needs row-major A (rows = M); k_dev needs both operands stored [K, .]
  if (a->m_dev && a->transA) return 0;
  if (a->k_dev && !(a->transA && !a->transB)) return 0;
  return 1;
}

size_t nnr_gemm_tc_workspace_bytes(const nnr_gemm_args* a) { return make_plan(a, algo_mode(a->algo)).total; }

static int encode_map(CUtensorMap* map, const void* base, bool bf16, int cols, int64_t pitch, int rows, int64_t plane_rows,
                      int nplanes, int box_c, int box_r, bool mn) {
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)nplanes};
  const size_t esz = bf16 ? 2 : 4;
  cuuint64_t gstr[2] = {(cuuint64_t)pitch * esz, (cuuint64_t)pitch * esz * (cuuint64_t)plane_rows};
  cuuint32_t box[3] = {(cuuint32_t)box_c, (cuuint32_t)box_r, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = get_encode()(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), gdim, gstr,
                            box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            (mn && !bf16) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { nnr_set_error("nnr_gemm(tc): cuTensorMapEncodeTiled failed (%d)", (int)r); return NNR_ERR_ARG; }
  return 0;
}

template <int MODE>
static int split_operand(const float* X, int64_t ld, int R, int C, int Cp, const int32_t* r_dev, void* out, size_t plane_stride,
                         cudaStream_t st) {
  bool vec = nnr_aligned16(X) && (ld % 4 == 0);
  long long total = (long long)R * (Cp / 4);
  long long want = (total + 256 * 4 - 1) / (256 * 4);
  int grid = (int)(want < 148 * 16 ? want : 148 * 16);
  if (grid < 1) grid = 1;
  void* ph = nnr_prof_begin(1, 0.0, st);
  tc_split_kernel<MODE><<<grid, 256, 0, st>>>(X, ld, R, C, Cp, r_dev, vec, out, plane_stride);
  nnr_prof_end(ph, st);
  NNR_LAUNCH_CHECK("tc_split_kernel");
  return 0;
}

template <bool BF16, bool PAIR>
static const void* tc_kernel_ptr2(int epk) {
  if (!BF16) return (const void*)gemm_tc_kernel<BF16, PAIR, -1>;
  switch (epk) {
    case NNR_EPI_NONE: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_NONE : -1>;
    case NNR_EPI_BIAS: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_BIAS : -1>;
    case NNR_EPI_BIAS_TANH: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_BIAS_TANH : -1>;
    case NNR_EPI_BIAS_RELU_RES: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_BIAS_RELU_RES : -1>;
    case NNR_EPI_GATE: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_GATE : -1>;
    case NNR_EPI_ADD_AUX: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? NNR_EPI_ADD_AUX : -1>;
    case TC_EPK_PARTIAL: return (const void*)gemm_tc_kernel<BF16, PAIR, BF16 ? TC_EPK_PARTIAL : -1>;
    default: return (const void*)gemm_tc_kernel<BF16, PAIR, -1>;
  }
}
template <bool BF16>
static const void* tc_kernel_ptr(bool pair, int epk) {
  return pair ? tc_kernel_ptr2<BF16, true>(epk) : tc_kernel_ptr2<BF16, false>(epk);
}

template <int MODE>
static int run_tc(const nnr_gemm_args* a, cudaStream_t st) {
  constexpr bool BF16 = MODE != 0;
  TcPlan pl = make_plan(a, MODE);
  NNR_REQUIRE(pl.total == 0 || (a->workspace && a->workspace_bytes >= pl.total), NNR_ERR_WORKSPACE,
              "nnr_gemm(tc): workspace %zu < %zu", a->workspace_bytes, pl.total);
  NNR_REQUIRE(nnr_aligned16(a->workspace), NNR_ERR_ALIGN, "nnr_gemm(tc): workspace must be 16B aligned");
  NNR_REQUIRE(nnr_aligned16(a->A_planes) && nnr_aligned16(a->B_planes) && a->a_planes_pitch % (BF16 ? 8 : 4) == 0 &&
                  a->b_planes_pitch % (BF16 ? 8 : 4) == 0,
              NNR_ERR_ALIGN, "nnr_gemm(tc): operand planes must be 16B aligned with a 16B pitch");
  NNR_REQUIRE(pl.smem <= 227 * 1024, NNR_ERR_UNSUPPORTED, "nnr_gemm(tc): smem plan too large");
  char* ws = (char*)a->workspace;
  const void* pa = a->A_planes;
  const void* pb = a->B_planes;
  int64_t a_pitch = a->a_planes_pitch, a_prow = a->a_planes_rows, b_pitch = a->b_planes_pitch, b_prow = a->b_planes_rows;
  int rc;
  // rows of A are M (m_dev) when row-major, K (k_dev) when MN-major; rows of B are K (k_dev) when MN-major
  if (!pa) {
    void* w = ws + pl.a_off;
    rc = split_operand<MODE>(a->A, a->lda, pl.a_rows, pl.a_cols, pl.a_cp, pl.a_mn ? a->k_dev : a->m_dev, w, pl.a_plane, st);
    if (rc) return rc;
    pa = w; a_pitch = pl.a_cp; a_prow = pl.a_rows;
  }
  if (!pb) {
    void* w = ws + pl.b_off;
    rc = split_operand<MODE>(a->B, a->ldb, pl.b_rows, pl.b_cols, pl.b_cp, pl.b_mn ? a->k_dev : nullptr, w, pl.b_plane, st);
    if (rc) return rc;
    pb = w; b_pitch = pl.b_cp; b_prow = pl.b_rows;
  }
  CUtensorMap map_a, map_b;
  const int ke = pl.kelem;
  rc = encode_map(&map_a, pa, BF16, pl.a_cols, a_pitch, pl.a_rows, a_prow, pl.nplanes, ke, pl.a_mn ? ke : TC_BM, pl.a_mn != 0);
  if (rc) return rc;
  rc = encode_map(&map_b, pb, BF16, pl.b_cols, b_pitch, pl.b_rows, b_prow, pl.nplanes, ke,
                  pl.b_mn ? ke : (pl.pair ? pl.block_n / 2 : pl.block_n), pl.b_mn != 0);
  if (rc) return rc;
  TcParams p;
  p.M = a->M; p.N = a->N; p.K = a->K; p.m_dev = a->m_dev; p.k_dev = a->k_dev;
  p.block_n = pl.block_n; p.stages = pl.stages; p.nplanes = pl.nplanes;
  p.a_mn = pl.a_mn; p.b_mn = pl.b_mn; p.split_k = pl.split_k; p.chain_kb = pl.chain_kb;
  // instruction descriptor: D=f32 (bits 4-5 = 1), A/B format (tf32 = 2, bf16 = 1) at bits 7-9 / 10-12, A/B major at
  // bits 15 / 16 (1 = MN-major), N >> 3 at bits 17-22, M >> 4 at bits 24-28
  const uint32_t fmt = BF16 ? 1u : 2u;
  p.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)pl.a_mn << 15) | ((uint32_t)pl.b_mn << 16) |
            ((uint32_t)(pl.block_n >> 3) << 17) | ((uint32_t)((pl.pair ? 2 * TC_BM : TC_BM) >> 4) << 24);
  p.partial = pl.split_k ? (float*)(ws + pl.partial_off) : nullptr;
  p.epi = make_epi(a);
  {
    auto ok = [](const void* ptr, int64_t ld) { return !ptr || (nnr_aligned16(ptr) && ld % 4 == 0); };
    p.epi_fast = (a->N % 4 == 0) && ok(a->C, a->ldc) && ok(a->aux, a->ldaux) && ok(a->aux_out, a->ldaux_out) &&
                 ok(a->rowbias, a->ldrowbias) && ok(a->bias, 4);
    if (a->epilogue == NNR_EPI_GATE && !(a->rowbias && a->rowmap && a->aux)) p.epi_fast = 0;
    if (a->epilogue == NNR_EPI_ADD_AUX && !a->aux) p.epi_fast = 0;
    const double lim = 4294967296.0;            // 32-bit element offsets inside the kernel
    if ((double)a->M * (double)a->ldc >= lim || (double)a->M * (double)a->ldaux >= lim || (double)a->M * (double)a->ldaux_out >= lim ||
        (double)a->M * (double)a->ldrowbias >= lim)
      p.epi_fast = 0;
  }
  p.c_planes = nullptr; p.c_pitch = 0; p.c_pstride = 0; p.c_lo = 0; p.c_rows = 0;
  if (a->C_planes) {
    NNR_REQUIRE(BF16 && p.epi_fast && !pl.split_k && a->N % 8 == 0 && a->c_planes_pitch >= a->N && a->c_planes_pitch % 8 == 0 &&
                    a->c_planes_rows >= a->M && nnr_aligned16(a->C_planes),
                NNR_ERR_UNSUPPORTED, "nnr_gemm: C_planes needs a bf16 tensor-core algo, N %% 8 == 0, aligned epilogue operands, no split-K");
    p.c_planes = (__nv_bfloat16*)a->C_planes;
    p.c_pitch = a->c_planes_pitch;
    p.c_pstride = a->c_planes_rows * a->c_planes_pitch;
    p.c_lo = pl.nplanes == 2;
    p.c_rows = (int)a->c_planes_rows;
  }
  // per-device caches: the dynamic shared-memory attribute is a property of (function, device), and so is the SM count
  static bool attr_set[16][2][2][8] = {};
  static int num_sms_tab[16] = {};
  int dev = 0;
  NNR_CUDA(cudaGetDevice(&dev));
  dev &= 15;
  // the epilogue kind is a template parameter of the kernel on the fast path (bf16 operand planes only; the fp32-plane
  // kernels keep the run-time-switched epilogue)
  int epk = (BF16 && p.epi_fast && !pl.split_k) ? a->epilogue : -1;
  // split-K partials: plain 16-byte stores into the [split][M][N] slices (offsets in 32 bits)
  if (BF16 && pl.split_k && a->N % 4 == 0 && nnr_aligned16(p.partial) &&
      (double)pl.max_splits * (double)a->M * (double)a->N < 4294967296.0)
    epk = TC_EPK_PARTIAL;
  const void* kernel = tc_kernel_ptr<BF16>(pl.pair != 0, epk);
  if (!attr_set[dev][BF16 ? 1 : 0][pl.pair][epk + 1]) {
    NNR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set[dev][BF16 ? 1 : 0][pl.pair][epk + 1] = true;
  }
  if (num_sms_tab[dev] == 0) NNR_CUDA(cudaDeviceGetAttribute(&num_sms_tab[dev], cudaDevAttrMultiProcessorCount, dev));
  const int num_sms = num_sms_tab[dev];
  void* ph = nnr_prof_begin(0, -1.0, st);     // flops are filled in by the caller-side profiler (needs m_dev/k_dev)
  {
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    if (pl.pair) {
      long cap_tiles = (long)((a->M + 2 * TC_BM - 1) / (2 * TC_BM)) * ((a->N + pl.block_n - 1) / pl.block_n);
      long pairs = cap_tiles < num_sms / 2 ? cap_tiles : num_sms / 2;
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      cfg.gridDim = dim3((unsigned)(2 * pairs));
    } else {
      long cap_tiles = (long)((a->M + TC_BM - 1) / TC_BM) * ((a->N + pl.block_n - 1) / pl.block_n) * pl.max_splits;
      cfg.gridDim = dim3((unsigned)(cap_tiles < num_sms ? cap_tiles : num_sms));
    }
    cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
    void* kargs[] = {(void*)&map_a, (void*)&map_b, (void*)&p};
    cudaError_t e = cudaLaunchKernelExC(&cfg, kernel, kargs);
    nnr_count_launch(1);
    if (e != cudaSuccess) { nnr_set_error("gemm_tc_kernel(%s): launch failed: %s", pl.pair ? "pair" : "single", cudaGetErrorString(e)); return (int)e; }
    nnr_prof_end(ph, st);
  }
  if (pl.split_k) {
    size_t tot = (size_t)a->M * a->N;
    void* ph2 = nnr_prof_begin(2, 0.0, st);
    if (a->N % 4 == 0 && nnr_aligned16(p.partial))
      tc_splitk_reduce4_kernel<<<(unsigned)((tot / 4 + 255) / 256), 256, 0, st>>>(p.partial, a->K, a->k_dev, pl.kelem, pl.chain_kb, a->M,
                                                                                 a->N, a->m_dev, p.epi);
    else
      tc_splitk_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(p.partial, a->K, a->k_dev, pl.kelem, pl.chain_kb, a->M,
                                                                            a->N, a->m_dev, p.epi);
    nnr_prof_end(ph2, st);
    NNR_LAUNCH_CHECK("tc_splitk_reduce_kernel");
  }
  return 0;
}

int nnr_gemm_tc(const nnr_gemm_args* a, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int mode = algo_mode(a->algo);
  if (mode == 1) return run_tc<1>(a, st);
  if (mode == 2) return run_tc<2>(a, st);
  return run_tc<0>(a, st);
}

// ------------------------------------------------------------------------------------------------
// public pre-split entry points
// ------------------------------------------------------------------------------------------------
extern "C" int64_t nnr_tc_split_pitch(int C, int algo) { return (int64_t)up((size_t)C, algo_mode(algo) ? 8 : 4); }
extern "C" size_t nnr_tc_split_bytes(int R, int C, int algo) {
  if (R <= 0 || C <= 0) return 0;
  const int mode = algo_mode(algo);
  return (size_t)R * (size_t)nnr_tc_split_pitch(C, algo) * (mode == 0 ? 8 : (mode == 1 ? 2 : 4));
}
extern "C" int nnr_tc_split(const float* X, int64_t ld, int R, int C, const int32_t* r_dev, int algo, void* planes,
                            size_t planes_bytes, void* stream) {
  NNR_REQUIRE(X && planes && R > 0 && C > 0 && ld >= C, NNR_ERR_ARG, "nnr_tc_split: bad arguments");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(R, C, algo), NNR_ERR_WORKSPACE, "nnr_tc_split: planes buffer too small");
  NNR_REQUIRE(nnr_aligned16(planes), NNR_ERR_ALIGN, "nnr_tc_split: planes must be 16B aligned");
  const int mode = algo_mode(algo);
  int Cp = (int)nnr_tc_split_pitch(C, algo);
  if (mode == 1) return split_operand<1>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (cudaStream_t)stream);
  if (mode == 2) return split_operand<2>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (cudaStream_t)stream);
  return split_operand<0>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (cudaStream_t)stream);
}

// split + column sums of the same matrix in one pass (see tc_split_colsum_kernel); workspace = per-row-block partials
extern "C" size_t nnr_tc_split_colsum_workspace_bytes(int R, int C, int algo) {
  if (R <= 0 || C <= 0) return 0;
  return (size_t)((R + tcs_rows(R) - 1) / tcs_rows(R)) * (size_t)nnr_tc_split_pitch(C, algo) * sizeof(float);
}
extern "C" int nnr_tc_split_colsum(const float* X, int64_t ld, int R, int C, const int32_t* r_dev, int algo, void* planes,
                                   size_t planes_bytes, float* colsum, int accumulate, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  NNR_REQUIRE(X && planes && colsum && workspace && R > 0 && C > 0 && ld >= C, NNR_ERR_ARG, "nnr_tc_split_colsum: bad arguments");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(R, C, algo), NNR_ERR_WORKSPACE, "nnr_tc_split_colsum: planes buffer too small");
  NNR_REQUIRE(workspace_bytes >= nnr_tc_split_colsum_workspace_bytes(R, C, algo), NNR_ERR_WORKSPACE,
              "nnr_tc_split_colsum: workspace too small");
  NNR_REQUIRE(nnr_aligned16(planes) && nnr_aligned16(workspace) && nnr_aligned16(X) && ld % 4 == 0, NNR_ERR_ALIGN,
              "nnr_tc_split_colsum: X, planes, workspace must be 16B aligned and ld %% 4 == 0");
  const int mode = algo_mode(algo);
  const int Cp = (int)nnr_tc_split_pitch(C, algo);
  NNR_REQUIRE(Cp <= 4 * 256 * TCS_MAXG, NNR_ERR_UNSUPPORTED, "nnr_tc_split_colsum: more than %d columns", 4 * 256 * TCS_MAXG);
  cudaStream_t st = (cudaStream_t)stream;
  const int nblocks = (R + tcs_rows(R) - 1) / tcs_rows(R);
  void* ph = nnr_prof_begin(1, 0.0, st);
  if (mode == 1) tc_split_colsum_kernel<1, false><<<nblocks, 256, 0, st>>>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (float*)workspace, SplitPre{});
  else if (mode == 2) tc_split_colsum_kernel<2, false><<<nblocks, 256, 0, st>>>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (float*)workspace, SplitPre{});
  else tc_split_colsum_kernel<0, false><<<nblocks, 256, 0, st>>>(X, ld, R, C, Cp, r_dev, planes, (size_t)R * Cp, (float*)workspace, SplitPre{});
  nnr_prof_end(ph, st);
  NNR_LAUNCH_CHECK("tc_split_colsum_kernel");
  tc_split_colsum_reduce<<<(C + 31) / 32, 512, 0, st>>>((const float*)workspace, nblocks, R, C, Cp, r_dev, colsum, accumulate);
  NNR_LAUNCH_CHECK("tc_split_colsum_reduce");
  return 0;
}

// dL/d(pre-activation) of "dropout -> relu -> Linear" as operand planes + column sums (bias gradient), see SplitPre
extern "C" int nnr_relu_bwd_split_colsum(const float* dy, const float* relu_out, int64_t ld, int R, int C, float p_drop,
                                         uint64_t seed, float* dy_dropped, int algo, void* planes, size_t planes_bytes,
                                         float* colsum, int accumulate, void* workspace, size_t workspace_bytes, void* stream) {
  NNR_REQUIRE(dy && relu_out && planes && colsum && workspace && R > 0 && C > 0 && ld >= C, NNR_ERR_ARG,
              "nnr_relu_bwd_split_colsum: bad arguments");
  NNR_REQUIRE(p_drop >= 0.f && p_drop < 1.f, NNR_ERR_ARG, "nnr_relu_bwd_split_colsum: p_drop=%f", p_drop);
  NNR_REQUIRE(algo == NNR_GEMM_TC_TF32X3 || algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3, NNR_ERR_UNSUPPORTED,
              "nnr_relu_bwd_split_colsum: planes exist only for the tensor-core GEMM algorithms");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(R, C, algo), NNR_ERR_WORKSPACE, "nnr_relu_bwd_split_colsum: planes buffer too small");
  NNR_REQUIRE(workspace_bytes >= nnr_tc_split_colsum_workspace_bytes(R, C, algo), NNR_ERR_WORKSPACE,
              "nnr_relu_bwd_split_colsum: workspace too small");
  NNR_REQUIRE(nnr_aligned16(planes) && nnr_aligned16(workspace) && nnr_aligned16(dy) && ld % 4 == 0, NNR_ERR_ALIGN,
              "nnr_relu_bwd_split_colsum: dy, planes, workspace must be 16B aligned and ld %% 4 == 0");
  const int mode = algo_mode(algo);
  const int Cp = (int)nnr_tc_split_pitch(C, algo);
  NNR_REQUIRE(Cp <= 4 * 256 * TCS_MAXG, NNR_ERR_UNSUPPORTED, "nnr_relu_bwd_split_colsum: more than %d columns", 4 * 256 * TCS_MAXG);
  cudaStream_t st = (cudaStream_t)stream;
  const int nblocks = (R + tcs_rows(R) - 1) / tcs_rows(R);
  SplitPre pre;
  pre.relu_out = relu_out; pre.dropped = dy_dropped; pre.p = p_drop; pre.inv_keep = 1.0f / (1.0f - p_drop); pre.seed = seed;
  if (mode == 1) tc_split_colsum_kernel<1, true><<<nblocks, 256, 0, st>>>(dy, ld, R, C, Cp, nullptr, planes, (size_t)R * Cp, (float*)workspace, pre);
  else if (mode == 2) tc_split_colsum_kernel<2, true><<<nblocks, 256, 0, st>>>(dy, ld, R, C, Cp, nullptr, planes, (size_t)R * Cp, (float*)workspace, pre);
  else tc_split_colsum_kernel<0, true><<<nblocks, 256, 0, st>>>(dy, ld, R, C, Cp, nullptr, planes, (size_t)R * Cp, (float*)workspace, pre);
  NNR_LAUNCH_CHECK("tc_split_colsum_kernel");
  tc_split_colsum_reduce<<<(C + 31) / 32, 512, 0, st>>>((const float*)workspace, nblocks, R, C, Cp, nullptr, colsum, accumulate);
  NNR_LAUNCH_CHECK("tc_split_colsum_reduce");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Word-embedding gather + dropout written DIRECTLY as operand planes (newsEncoders.py:117-118): the embedded tokens
// are only ever consumed by GEMMs (gx = x W_ih^T forward, dW_ih = dz^T x backward), so the packed fp32 [tokens, E]
// tensor never has to exist: one warp per (row, t) token slot reads the table row, applies the keep mask of
// nnr_embed_gather_fwd (same counter = (slot * E + e), same scale) and stores hi/lo.  Extra warps zero the row tail
// [ntok, round_up(ntok, 64)) that the MN-major (wgrad) tiles read.
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) embed_gather_planes_kernel(const float* __restrict__ table, const int32_t* __restrict__ ids,
                                                                  const int32_t* __restrict__ len, const int32_t* __restrict__ off,
                                                                  int N, int L, int E, int V, int cap, int Cp, void* __restrict__ out,
                                                                  size_t plane_stride, float p, float inv_keep, uint64_t seed) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long slots = (long long)N * L;
  if (p > 0.0f) seed = nnr_resolve_seed(seed);
  const int ncq = Cp >> 2, E4 = E >> 2;
  if (w >= slots) {                                                   // zero tail rows
    const int ntok = off[N];
    const long long row = (long long)ntok + (w - slots);
    if (row >= min((long long)cap, ((long long)ntok + 63) / 64 * 64)) return;
    for (int q = lane; q < ncq; q += 32) tc_split_store4<MODE>(out, plane_stride, Cp, (int)row, q * 4, make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const int slot = (int)w;
  const int r = slot / L, t = slot - r * L;
  if (t >= len[r]) return;
  int id = ids[slot];
  id = min(max(id, 0), V - 1);
  const float4* src = reinterpret_cast<const float4*>(table + (size_t)id * E);
  const int row = off[r] + t;
  const uint64_t ebase4 = ((uint64_t)slot * (uint64_t)E) >> 2;        // E % 4 == 0
  for (int q = lane; q < ncq; q += 32) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);                       // column pad [E, Cp)
    if (q < E4) {
      v = __ldg(src + q);
      if (p > 0.0f) {
        float ks[4];
        dropout_scale4(seed, ebase4 + q, p, inv_keep, ks);
        v.x *= ks[0]; v.y *= ks[1]; v.z *= ks[2]; v.w *= ks[3];
      }
    }
    tc_split_store4<MODE>(out, plane_stride, Cp, row, q * 4, v);
  }
}

extern "C" int nnr_embed_gather_planes_fwd(const float* table, const int32_t* ids, const int32_t* len, const int32_t* off,
                                           int N, int L, int E, int V, int cap, float p_drop, uint64_t seed, int algo,
                                           void* planes, size_t planes_bytes, void* stream) {
  NNR_REQUIRE(table && ids && len && off && planes && N > 0 && L > 0 && E > 0 && V > 0 && cap > 0, NNR_ERR_ARG,
              "nnr_embed_gather_planes_fwd: bad arguments");
  NNR_REQUIRE(p_drop >= 0.0f && p_drop < 1.0f, NNR_ERR_ARG, "nnr_embed_gather_planes_fwd: p_drop=%f", p_drop);
  NNR_REQUIRE(E % 4 == 0 && nnr_aligned16(table) && nnr_aligned16(planes), NNR_ERR_ALIGN,
              "nnr_embed_gather_planes_fwd: E %% 4 == 0 and 16B-aligned table / planes required");
  NNR_REQUIRE(algo == NNR_GEMM_TC_TF32X3 || algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3, NNR_ERR_UNSUPPORTED,
              "nnr_embed_gather_planes_fwd: planes exist only for the tensor-core GEMM algorithms");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(cap, E, algo), NNR_ERR_WORKSPACE, "nnr_embed_gather_planes_fwd: planes buffer too small");
  const int mode = algo_mode(algo);
  const int Cp = (int)nnr_tc_split_pitch(E, algo);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t warps = (size_t)N * L + 64;
  const unsigned blocks = (unsigned)((warps * 32 + 255) / 256);
  const float inv_keep = 1.0f / (1.0f - p_drop);
  const size_t ps = (size_t)cap * Cp;
  if (mode == 1) embed_gather_planes_kernel<1><<<blocks, 256, 0, st>>>(table, ids, len, off, N, L, E, V, cap, Cp, planes, ps, p_drop, inv_keep, seed);
  else if (mode == 2) embed_gather_planes_kernel<2><<<blocks, 256, 0, st>>>(table, ids, len, off, N, L, E, V, cap, Cp, planes, ps, p_drop, inv_keep, seed);
  else embed_gather_planes_kernel<0><<<blocks, 256, 0, st>>>(table, ids, len, off, N, L, E, V, cap, Cp, planes, ps, p_drop, inv_keep, seed);
  NNR_LAUNCH_CHECK("embed_gather_planes_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// The recurrent input of every LSTM step (h_{t-1} forward, h_{t+1} reverse; zero at the sequence ends) as operand
// planes: nnr_lstm_shift_h + nnr_tc_split in one pass.  It is only ever the B operand of dW_hh = dz^T hprev.
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) lstm_shift_h_planes_kernel(const float* __restrict__ h, const int32_t* __restrict__ len,
                                                                  const int32_t* __restrict__ off, const int32_t* __restrict__ tok_row,
                                                                  int N, int H, int cap, int Cp, void* __restrict__ out, size_t plane_stride) {
  const int ntok = min(off[N], cap);
  const int rows = min(cap, (ntok + 63) / 64 * 64);
  const int H2 = 2 * H, hq = H >> 2, ncq = Cp >> 2, q_valid = H2 >> 2;
  const long long total = (long long)rows * ncq;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i / ncq), q = (int)(i - (long long)p * ncq);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p < ntok && q < q_valid) {
      const int r = tok_row[p];
      const int t = p - off[r];
      if (q < hq) { if (t > 0) v = __ldg(reinterpret_cast<const float4*>(h + (size_t)(p - 1) * H2) + q); }
      else { if (t < len[r] - 1) v = __ldg(reinterpret_cast<const float4*>(h + (size_t)(p + 1) * H2) + q); }
    }
    tc_split_store4<MODE>(out, plane_stride, Cp, p, q * 4, v);
  }
}

extern "C" int nnr_lstm_shift_h_planes(const float* h, const int32_t* len, const int32_t* off, const int32_t* tok_row, int N,
                                       int L, int H, int cap, int algo, void* planes, size_t planes_bytes, void* stream) {
  NNR_REQUIRE(h && len && off && tok_row && planes && N > 0 && L > 0 && H > 0 && cap > 0, NNR_ERR_ARG, "nnr_lstm_shift_h_planes: bad arguments");
  NNR_REQUIRE(H % 4 == 0 && nnr_aligned16(h) && nnr_aligned16(planes), NNR_ERR_ALIGN, "nnr_lstm_shift_h_planes: H %% 4 == 0, 16B alignment");
  NNR_REQUIRE(algo == NNR_GEMM_TC_TF32X3 || algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3, NNR_ERR_UNSUPPORTED,
              "nnr_lstm_shift_h_planes: planes exist only for the tensor-core GEMM algorithms");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(cap, 2 * H, algo), NNR_ERR_WORKSPACE, "nnr_lstm_shift_h_planes: planes buffer too small");
  const int mode = algo_mode(algo);
  const int Cp = (int)nnr_tc_split_pitch(2 * H, algo);
  const size_t ps = (size_t)cap * Cp;
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == 1) lstm_shift_h_planes_kernel<1><<<148 * 8, 256, 0, st>>>(h, len, off, tok_row, N, H, cap, Cp, planes, ps);
  else if (mode == 2) lstm_shift_h_planes_kernel<2><<<148 * 8, 256, 0, st>>>(h, len, off, tok_row, N, H, cap, Cp, planes, ps);
  else lstm_shift_h_planes_kernel<0><<<148 * 8, 256, 0, st>>>(h, len, off, tok_row, N, H, cap, Cp, planes, ps);
  NNR_LAUNCH_CHECK("lstm_shift_h_planes_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Selective-gate backward prologue, fused (nnr_gate_bwd_pre + nnr_tc_split + nnr_segment_colsum in one pass over the
// tokens): per news r, dz = dhg * h * g * (1 - g) leaves as operand planes (it feeds the dW_H and dh GEMMs), its sum over
// the news' tokens is dmproj[r] (gradient of the projected partner cell state), dh0 = dhg * g stays fp32.
// One CTA per news, a thread per 4-column group, tokens in order (the same summation order as segment_colsum_kernel).
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128) gate_bwd_planes_kernel(const float* __restrict__ dhg, const float* __restrict__ h,
                                                              const float* __restrict__ g, const int32_t* __restrict__ off, int N,
                                                              int D, int cap, int Cp, void* __restrict__ planes, size_t plane_stride,
                                                              float* __restrict__ dh0, float* __restrict__ dmproj, int64_t lddm) {
  const int r = blockIdx.x;
  const int ncq = Cp >> 2, dq = D >> 2;
  if (r >= N) {                                                  // zero row tail [ntok, round_up(ntok, 64)) of the planes
    const int ntok = min(off[N], cap);
    const int r1 = min(cap, (ntok + 63) / 64 * 64);
    for (int i = (r - N) * 128 + threadIdx.x; i < (r1 - ntok) * ncq; i += (gridDim.x - N) * 128)
      tc_split_store4<MODE>(planes, plane_stride, Cp, ntok + i / ncq, (i % ncq) * 4, make_float4(0.f, 0.f, 0.f, 0.f));
    return;
  }
  const int a = off[r], b = min(off[r + 1], cap);
  for (int cq = threadIdx.x; cq < ncq; cq += 128) {
    if (cq >= dq) {                                              // column pad
      for (int p = a; p < b; ++p) tc_split_store4<MODE>(planes, plane_stride, Cp, p, cq * 4, make_float4(0.f, 0.f, 0.f, 0.f));
      continue;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int p = a;
    auto one = [&](const float4 x, const float4 hh, const float4 gg, int pp) {
      float4 z, d0;      // explicit roundings: no contraction with the running sum, same bits as gate_bwd_pre_kernel
      z.x = __fmul_rn(__fmul_rn(__fmul_rn(x.x, hh.x), gg.x), __fsub_rn(1.f, gg.x)); d0.x = __fmul_rn(x.x, gg.x);
      z.y = __fmul_rn(__fmul_rn(__fmul_rn(x.y, hh.y), gg.y), __fsub_rn(1.f, gg.y)); d0.y = __fmul_rn(x.y, gg.y);
      z.z = __fmul_rn(__fmul_rn(__fmul_rn(x.z, hh.z), gg.z), __fsub_rn(1.f, gg.z)); d0.z = __fmul_rn(x.z, gg.z);
      z.w = __fmul_rn(__fmul_rn(__fmul_rn(x.w, hh.w), gg.w), __fsub_rn(1.f, gg.w)); d0.w = __fmul_rn(x.w, gg.w);
      *reinterpret_cast<float4*>(dh0 + (size_t)pp * D + cq * 4) = d0;
      tc_split_store4<MODE>(planes, plane_stride, Cp, pp, cq * 4, z);
      acc.x = __fadd_rn(acc.x, z.x); acc.y = __fadd_rn(acc.y, z.y); acc.z = __fadd_rn(acc.z, z.z); acc.w = __fadd_rn(acc.w, z.w);
    };
    for (; p + 4 <= b; p += 4) {                                 // twelve 16-byte loads in flight
      float4 x[4], hh[4], gg[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const size_t o = (size_t)(p + u) * D + cq * 4;
        x[u] = __ldg(reinterpret_cast<const float4*>(dhg + o));
        hh[u] = __ldg(reinterpret_cast<const float4*>(h + o));
        gg[u] = __ldg(reinterpret_cast<const float4*>(g + o));
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) one(x[u], hh[u], gg[u], p + u);
    }
    for (; p < b; ++p) {
      const size_t o = (size_t)p * D + cq * 4;
      one(__ldg(reinterpret_cast<const float4*>(dhg + o)), __ldg(reinterpret_cast<const float4*>(h + o)),
          __ldg(reinterpret_cast<const float4*>(g + o)), p);
    }
    *reinterpret_cast<float4*>(dmproj + (size_t)r * lddm + cq * 4) = acc;
  }
}

extern "C" int nnr_gate_bwd_planes(const float* dhg, const float* h, const float* g, const int32_t* off, int N, int D, int cap,
                                   int algo, void* dz_planes, size_t planes_bytes, float* dh0, float* dmproj, int64_t lddm,
                                   void* stream) {
  NNR_REQUIRE(dhg && h && g && off && dz_planes && dh0 && dmproj && N > 0 && D > 0 && cap > 0 && lddm >= D, NNR_ERR_ARG,
              "nnr_gate_bwd_planes: bad arguments");
  NNR_REQUIRE(D % 4 == 0 && lddm % 4 == 0 && nnr_aligned16(dhg) && nnr_aligned16(h) && nnr_aligned16(g) && nnr_aligned16(dz_planes) &&
                  nnr_aligned16(dh0) && nnr_aligned16(dmproj), NNR_ERR_ALIGN, "nnr_gate_bwd_planes: needs 16B alignment and D %% 4 == 0");
  NNR_REQUIRE(algo == NNR_GEMM_TC_TF32X3 || algo == NNR_GEMM_TC_BF16 || algo == NNR_GEMM_TC_BF16X3, NNR_ERR_UNSUPPORTED,
              "nnr_gate_bwd_planes: planes exist only for the tensor-core GEMM algorithms");
  NNR_REQUIRE(planes_bytes >= nnr_tc_split_bytes(cap, D, algo), NNR_ERR_WORKSPACE, "nnr_gate_bwd_planes: planes buffer too small");
  const int mode = algo_mode(algo);
  const int Cp = (int)nnr_tc_split_pitch(D, algo);
  const size_t ps = (size_t)cap * Cp;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)N + 8;
  if (mode == 1) gate_bwd_planes_kernel<1><<<blocks, 128, 0, st>>>(dhg, h, g, off, N, D, cap, Cp, dz_planes, ps, dh0, dmproj, lddm);
  else if (mode == 2) gate_bwd_planes_kernel<2><<<blocks, 128, 0, st>>>(dhg, h, g, off, N, D, cap, Cp, dz_planes, ps, dh0, dmproj, lddm);
  else gate_bwd_planes_kernel<0><<<blocks, 128, 0, st>>>(dhg, h, g, off, N, D, cap, Cp, dz_planes, ps, dh0, dmproj, lddm);
  NNR_LAUNCH_CHECK("gate_bwd_planes_kernel");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Operand planes of MANY small matrices in one launch (all weight matrices after an optimizer step: ~50 launches of
// 3-5 us each otherwise).  descs is a DEVICE array; up to TSM_PARTS CTAs per matrix (grid.y = matrix).
// ------------------------------------------------------------------------------------------------
#define TSM_PARTS 64
template <int MODE>
__global__ void __launch_bounds__(256) tc_split_many_kernel(const nnr_split_desc* __restrict__ descs, int n) {
  const int di = blockIdx.y, part = blockIdx.x;
  if (di >= n) return;
  const nnr_split_desc d = descs[di];
  const int Cp = (int)d.pitch;
  const int cq_per_row = Cp >> 2;
  const long long total = (long long)d.rows * cq_per_row;
  const bool vec = ((((uintptr_t)d.src) & 15) == 0) && (d.ld % 4 == 0);
  for (long long i = (long long)part * 256 + threadIdx.x; i < total; i += TSM_PARTS * 256) {
    const int r = (int)(i / cq_per_row), cq = (int)(i - (long long)r * cq_per_row) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* sp = d.src + (size_t)r * d.ld + cq;
    if (vec && cq + 3 < d.cols) x = __ldg(reinterpret_cast<const float4*>(sp));
    else {
      if (cq < d.cols) x.x = __ldg(sp);
      if (cq + 1 < d.cols) x.y = __ldg(sp + 1);
      if (cq + 2 < d.cols) x.z = __ldg(sp + 2);
      if (cq + 3 < d.cols) x.w = __ldg(sp + 3);
    }
    tc_split_store4<MODE>(d.planes, (size_t)d.rows * Cp, Cp, r, cq, x);
  }
}
extern "C" int nnr_tc_split_many(const nnr_split_desc* descs, int n, int algo, void* stream) {
  NNR_REQUIRE(descs && n > 0 && n <= 65535, NNR_ERR_ARG, "nnr_tc_split_many: bad arguments");
  const int mode = algo_mode(algo);
  cudaStream_t st = (cudaStream_t)stream;
  void* ph = nnr_prof_begin(1, 0.0, st);
  if (mode == 1) tc_split_many_kernel<1><<<dim3(TSM_PARTS, n), 256, 0, st>>>(descs, n);
  else if (mode == 2) tc_split_many_kernel<2><<<dim3(TSM_PARTS, n), 256, 0, st>>>(descs, n);
  else tc_split_many_kernel<0><<<dim3(TSM_PARTS, n), 256, 0, st>>>(descs, n);
  nnr_prof_end(ph, st);
  NNR_LAUNCH_CHECK("tc_split_many_kernel");
  return 0;
}

// phase stamps of the last gemm_tc_kernel launch (CTA 0; library built with -DNNR_TC_PROF), 16 clock64 values; returns 0 when
// the library was built without them
extern "C" int nnr_debug_tc_prof(unsigned long long* out) {
#ifdef NNR_TC_PROF
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out, g_tc_prof, sizeof(unsigned long long) * 16) == cudaSuccess ? 1 : 0;
#else
  (void)out;
  return 0;
#endif
}
