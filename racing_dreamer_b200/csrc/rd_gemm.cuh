// rd_gemm.cuh -- the dense layers of the Dreamer agent on the 5th-generation tensor cores (SURVEY.md §8-f2).
//
// One kernel, k_dense<EPI, NSLAB, NACC, STAGES>, computes a 128 x 64 tile of  act(A @ W + b)  for a batch of envs:
//   * A (activations, [envs][K] float32, K contiguous) and W (weights, stored transposed [N][K], K contiguous) are
//     streamed through a 4-stage shared-memory ring by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle, out-of-bounds
//     rows/columns zero-filled by the copy engine, so no padded copies of anything exist in HBM);
//   * one elected thread issues tcgen05.mma.kind::tf32 (M = 128, N = 64, K = 8 per instruction; float32 operands are
//     read as TF32, accumulation in float32) into tensor memory; tcgen05.commit hands each ring slot back to the
//     producer and, after the last K block, hands the accumulators to the epilogue warps;
//   * four epilogue warps read their 32 TMEM lanes (one env per thread) with tcgen05.ld and apply the layer's
//     epilogue in registers: bias + ELU, the Keras GRU cell gates, the RSSM posterior sample, or the actor head with
//     SampleDist.mode() -- so no pre-activation ever reaches HBM.
// Precision.  kind::tf32 reads 10 mantissa bits of each operand.  With GemmArgs-level "x3" operation every product is
// evaluated as  hi*hi + lo*hi + hi*lo  (hi = the TF32 rounding of the float32 value, lo = the TF32 rounding of the
// remainder; weights are split once at upload, activations by the epilogue that produces them): three passes over K
// into the same float32 accumulator, ~2^-21 relative error per product instead of 2^-11 -- float32-grade results,
// which is what the reference's TensorFlow computes in.
// The tensor core adds each instruction's products into the float32 accumulator with truncation, so a long K chain
// drifts by ~(chain length) x 2^-24 x |partial sum| (measured: 2e-3 on the 1280-term obs1 layer).  The K range of a
// layer is therefore cut into groups that accumulate in separate TMEM columns, and the epilogue adds the partial
// sums in round-to-nearest float32; the lo*hi / hi*lo passes get an accumulator of their own.
// A layer is described by up to twelve "phases" (K ranges with their own A source: concat([deter, embed]) @ W is two
// phases over one W) and up to three weight slabs per phase feeding up to four accumulators (the GRU's z, r and the
// two halves of the candidate gate).
//
// Replaces tf.keras Dense / GRUCell calls inside RSSM.obs_step / img_step and ActionDecoder.__call__
// [REF ros_agent/models/dreamer/models.py:63-90, 307-332].
#pragma once
#include <cuda.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "rd_common.cuh"

#define GM_BM 128
#define GM_BN 64
#define GM_BK 32                      // float32 elements per K block = one 128-byte swizzle row
#define GM_A_BYTES (GM_BM * 128)      // 16 KB
#define GM_W_BYTES (GM_BN * 128)      // 8 KB
#ifndef GM_EPI_GROUPS
#define GM_EPI_GROUPS 2               // epilogue warp groups: group p of 4 warps handles columns [p, p + 1) * 64 / GROUPS of the tile
#endif
#define GM_THREADS (64 + 128 * GM_EPI_GROUPS)   // warp 0: TMA producer, warp 1: TMEM allocator + MMA issuer, then the epilogue warps
#define GM_STOCH 30                   // RSSM stochastic state size of the shipped agents [REF racing_dreamer.py:20]

#define GM_MAX_PHASES 12
struct GemmMaps {   // tensor maps of one launch: A sources and weight matrices, hi parts and (x3 mode) lo parts
  CUtensorMap a[4];
  CUtensorMap w[4];
  CUtensorMap o[2];  // GemmArgs::tma_out: the output rows (hi, lo), box 32 columns x 128 rows -- the view the next layer loads
};
struct GemmPhase {
  int a_map, w_map; // indices into GemmMaps
  int k_blocks;     // number of 32-wide K blocks of this phase
  int a_k0;         // first K element in the phase's A tensor map
  int w_k0;         // first K element in the phase's W tensor map
  int nb;           // weight slabs per block (1..3)
  int w_row0[3];    // first W row of each slab (the CTA's n0 is added)
  int acc[3];       // accumulator fed by each slab
  // k_dense<..., X3 = true>: the K block also carries the lo parts of both operands (maps a_map_lo / w_map_lo) and feeds
  // three products: lo*hi and hi*lo into acc_small[i], hi*hi into acc[i]
  int a_map_lo, w_map_lo;
  int acc_small[3];
};

enum { EPI_DENSE = 0, EPI_GRU = 1, EPI_STOCH = 2, EPI_ACTOR = 3 };
enum { GM_NOISE_ZERO = 0, GM_NOISE_PHILOX = 1, GM_NOISE_EXPLICIT = 2 };
#define RD_STREAM_STOCH 0x53544f43u
#define RD_STREAM_ACTOR 0x41435452u
#define RD_STREAM_TRAIN 0x5452414eu   // training head: the action sample and its exploration noise (k_actor_train)

struct GemmArgs {
  int M, N;                 // rows (envs), valid output columns
  int n_phases;
  int n_acc;                // accumulators (64 TMEM columns each) per output: the epilogue adds them up (GRU: per gate)
  GemmPhase ph[GM_MAX_PHASES];
  const float* bias;        // [N]; GRU: [2][3N] (input side, recurrent side; gates z, r, h)
  float* out; int ldo;      // DENSE / GRU: output rows, TF32-rounded (they are only ever read as MMA operands)
  float* out_lo;            // x3 mode: TF32-rounded remainder of the same rows (same pitch), or null
  int act;                  // DENSE: 1 = ELU, 0 = linear
  int tma_out;              // DENSE / GRU: 1 = the tile leaves through shared memory and the copy engine (maps.o), see gm_stage_f4
  const float* hold; const float* hold_lo; int ldh;   // GRU: previous deterministic state (hi [+ lo])
  // STOCH / ACTOR
  int noise;                // GM_NOISE_*
  const float* eps; int ld_eps;   // explicit standard-normal draws: STOCH [M][30], ACTOR [M][n_samples*2]
  uint32_t key0, key1, step, gid0;
  float* dbg;               // STOCH: [M][60] mean | std; ACTOR: [M][8] mean0 mean1 std0 std1 a0 a1 logp index
  float* actions;           // ACTOR: [M][2] agent-facing action (what rd_step reads)
  float* feat; float* feat_lo; int ldf;   // STOCH: stoch -> feat[row][0..29]; ACTOR: action -> feat[row][30..31]
  const float* bn;          // ACTOR "normalized" head: [4][4] gamma, beta, moving_mean, moving_variance (or null)
  float raw_init_std, min_std, mean_scale, bn_eps;
  int n_samples;
};

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void gm_tma_2d(uint32_t dst_smem, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          dst_smem),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(rd_smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void gm_prefetch_map(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// bounded wait: a broken pipeline traps (the launch fails) instead of hanging the device
__device__ __forceinline__ void gm_mbar_wait(uint64_t* bar, uint32_t parity, bool backoff = false) {
  const uint32_t a = rd_smem_u32(bar);
  for (uint32_t spins = 0;; ++spins) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
    if (ok) return;
    // the four epilogue warps wait for the whole K loop: they must not take issue slots from the single issuer /
    // producer threads their schedulers also serve
    if (backoff) __nanosleep(256);
    if (spins > (1u << 24)) __trap();
  }
}
__device__ __forceinline__ void gm_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void gm_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void gm_tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(rd_smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void gm_tmem_free(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void gm_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(rd_smem_u32(bar))
               : "memory");
}
// One thread of a converged warp (the compiler then issues the tcgen05 / TMA instructions of the elected region
// directly instead of wrapping each one in a per-lane election loop).
__device__ __forceinline__ bool gm_elect_one() {
  uint32_t p;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(p));
  return p != 0;
}
// K-major operand tile in shared memory, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart
// (cute::UMMA::SmemDescriptor: start >> 4 | LBO 1 << 16 | SBO 64 << 32 | version 1 << 46 | SWIZZLE_128B 2 << 61)
__device__ __forceinline__ uint64_t gm_smem_desc(uint32_t addr) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// The descriptor's low word (start address >> 4 | LBO) and its constant high word (SBO, version, swizzle): the issuer
// thread steps the low word by plain additions (32 bytes of K = +2, next slab = +bytes / 16) instead of rebuilding
// the 64-bit value for every instruction -- its own instruction stream is what bounds a K block (see the kernel).
__device__ __forceinline__ uint32_t gm_desc_lo(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); }
#define GM_DESC_HI ((uint32_t)((64ull << 32 | 1ull << 46 | 2ull << 61) >> 32))
__device__ __forceinline__ uint64_t gm_desc(uint32_t lo) { return ((uint64_t)GM_DESC_HI << 32) | lo; }
// cute::UMMA::InstrDescriptor: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), both K-major, N >> 3 at bit 17, M >> 4 at 24
#define GM_IDESC_N(BN_) ((1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)((BN_) >> 3) << 17) | ((uint32_t)(GM_BM >> 4) << 24))
__device__ __forceinline__ void gm_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 bit x N columns: thread i of the warp receives TMEM lane (lane_base + i), N consecutive columns
__device__ __forceinline__ void gm_tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void gm_tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// the same columns of n_acc accumulators (GM_BN * stride columns apart), added in round-to-nearest float32
__device__ __forceinline__ void gm_tmem_sum16(uint32_t taddr, int n_acc, int stride, float (&v)[16], int bn = GM_BN) {
  gm_tmem_ld16(taddr, v);
  for (int a = 1; a < n_acc; ++a) {
    float t[16];
    gm_tmem_ld16(taddr + (uint32_t)(a * stride * bn), t);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += t[i];
  }
}
__device__ __forceinline__ void gm_tmem_sum8(uint32_t taddr, int n_acc, int stride, float (&v)[8]) {
  gm_tmem_ld8(taddr, v);
  for (int a = 1; a < n_acc; ++a) {
    float t[8];
    gm_tmem_ld8(taddr + (uint32_t)(a * stride * GM_BN), t);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] += t[i];
  }
}
__device__ __forceinline__ float gm_round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// tf.nn.elu; exp(x) - 1 instead of expm1: the absolute error (6e-8) is what matters for the next layer's dot products
__device__ __forceinline__ float gm_elu(float x) { return x > 0.f ? x : expf(x) - 1.0f; }
__device__ __forceinline__ float gm_softplus(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float gm_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }
// four standard normals from one Philox block (Box-Muller on (0,1] uniforms)
__device__ __forceinline__ void gm_normal4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                           float (&z)[4]) {
  uint32_t c[4] = {c0, c1, c2, c3};
  philox4x32_10(c, k0, k1);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float u1 = ((float)(c[2 * h] >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0, 1]
    const float u2 = (float)(c[2 * h + 1] >> 8) * (1.0f / 16777216.0f);        // [0, 1)
    const float r = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    z[2 * h] = r * cs;
    z[2 * h + 1] = r * sn;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Output tiles through the copy engine.  In the epilogue a thread owns a tile ROW (its TMEM lane), so a store from
// registers puts 16 bytes into each of 32 different rows per instruction: thousands of half-sector writes per CTA,
// measured at 8.5 us of a 16.5 us actor layer (profiles/r5b_dreamer_chain.txt).  Instead the warps build [128 rows]
// [32 columns] tiles in shared memory -- the ring is idle by then -- in the 128-byte-swizzled layout of the tensor
// map the NEXT layer loads these rows through, and one thread hands each tile to cp.async.bulk.tensor (rows >= M and
// columns >= N are clipped by the map).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void gm_stage_f4(uint32_t tile_smem, uint32_t r, int col_in_tile, const float4& v) {
  const uint32_t off = r * 128u + ((((uint32_t)col_in_tile >> 2) ^ (r & 7u)) << 4);   // SWIZZLE_128B
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tile_smem + off), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void gm_tile_store(const CUtensorMap* map, int x, int y, uint32_t tile_smem) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(x), "r"(y), "r"(tile_smem)
               : "memory");
}
// The warps that share a 32-column tile (n_threads of them, barrier `bar_id`) have staged it; `leader` stores it.
__device__ __forceinline__ void gm_tiles_out(int bar_id, int n_threads, bool leader, bool any, const CUtensorMap* m_hi,
                                             const CUtensorMap* m_lo, int x, int y, uint32_t s_hi, uint32_t s_lo) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the tiles were written through the generic proxy
  asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(n_threads) : "memory");
  if (leader && any) {
    gm_tile_store(m_hi, x, y, s_hi);
    if (m_lo) gm_tile_store(m_lo, x, y, s_lo);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory stays valid until the engine has read it
  }
}

// ---------------------------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------------------------
template <int EPI, int NSLAB, int NACC, int GM_STAGES, bool X3 = false, int EW = GM_EPI_GROUPS, int BN = GM_BN>
__global__ void __launch_bounds__(64 + 128 * EW, 1)
    k_dense(const __grid_constant__ GemmMaps maps, const GemmArgs g) {
  extern __shared__ uint8_t gm_smem_raw[];
  __shared__ uint64_t full_bar[GM_STAGES], empty_bar[GM_STAGES], acc_bar;
  __shared__ uint32_t tmem_slot;
#ifdef GM_CHAIN_TRACE   // per-role clock stamps (tools/gpu_chain_trace.sh)
  __shared__ long long trd[8];
#define GM_TRD(k) trd[k] = clock64()
#else
#define GM_TRD(k) do { } while (0)
#endif
  // X3: a ring stage holds the hi AND the lo tiles of a K block ([A_hi | W_hi slabs | A_lo | W_lo slabs]) and feeds all
  // three products of the float32-grade scheme from one load: two thirds of the operand bytes of three separate passes
  // and a third of the producer / issuer hand-offs.
  static_assert(BN % 16 == 0 && BN <= 256 && NACC * BN <= 512, "MMA N and the accumulators' TMEM columns");
  constexpr uint32_t W_BYTES = BN * 128, IDESC = GM_IDESC_N(BN);
  constexpr uint32_t SUB_BYTES = GM_A_BYTES + NSLAB * W_BYTES;
  constexpr uint32_t STAGE_BYTES = (X3 ? 2u : 1u) * SUB_BYTES;
  constexpr uint32_t TM_COLS = (NACC * BN <= 64) ? 64 : (NACC * BN <= 128 ? 128 : (NACC * BN <= 256 ? 256 : 512));
  const uint32_t smem_base = (rd_smem_u32(gm_smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B tiles: 1024-byte aligned
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * GM_BM, n0 = blockIdx.y * BN;

  if (threadIdx.x == 0) {
    for (int p = 0; p < g.n_phases; ++p) {
      gm_prefetch_map(&maps.a[g.ph[p].a_map]); gm_prefetch_map(&maps.w[g.ph[p].w_map]);
      if (X3) { gm_prefetch_map(&maps.a[g.ph[p].a_map_lo]); gm_prefetch_map(&maps.w[g.ph[p].w_map_lo]); }
    }
#pragma unroll
    for (int s = 0; s < GM_STAGES; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&full_bar[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&empty_bar[s])));
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&acc_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) gm_tmem_alloc(&tmem_slot, TM_COLS);
  gm_tc_fence_before();
  __syncthreads();
  gm_tc_fence_after();
  const uint32_t tmem = tmem_slot;
  // Programmatic dependent launch: the next k_dense of the stream may start its own set-up (barriers, TMEM, tensor-map
  // fetch) now; everything that touches global memory first waits for the previous kernel to have completed.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (threadIdx.x == 0) GM_TRD(0);

  if (warp == 0) {
    if (gm_elect_one()) {   // ===== TMA producer =====
      // like the issuer below, this thread's instruction stream bounds a K block: everything that does not change from
      // one K block to the next is set up per phase.
      // The weights do not depend on the kernel in front of this one: the weight tiles of the first GM_STAGES K blocks
      // are requested BEFORE griddepcontrol.wait (pass 0), the activation tiles of those K blocks and everything else
      // after it (pass 1) -- the ring is full of weights by the time the previous layer's outputs exist.
      for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1) { asm volatile("griddepcontrol.wait;" ::: "memory"); GM_TRD(1); }
        uint32_t it = 0;
        for (int p = 0; p < g.n_phases; ++p) {
          const GemmPhase& ph = g.ph[p];
          const CUtensorMap* ma = &maps.a[ph.a_map];
          const CUtensorMap* mw = &maps.w[ph.w_map];
          const int nb = ph.nb, kbs = ph.k_blocks;
          const CUtensorMap* ma2 = &maps.a[X3 ? ph.a_map_lo : ph.a_map];
          const CUtensorMap* mw2 = &maps.w[X3 ? ph.w_map_lo : ph.w_map];
          const uint32_t tx = (X3 ? 2u : 1u) * (GM_A_BYTES + (uint32_t)nb * W_BYTES);
          int ak = ph.a_k0, wk = ph.w_k0;
          const int r0 = ph.w_row0[0] + n0, r1 = ph.w_row0[1] + n0, r2 = ph.w_row0[2] + n0;
          for (int kb = 0; kb < kbs; ++kb, ++it, ak += GM_BK, wk += GM_BK) {
            if (pass == 0 && it >= (uint32_t)GM_STAGES) break;
            const uint32_t s = it % GM_STAGES, par = (it / GM_STAGES) & 1u;
            const bool early = it < (uint32_t)GM_STAGES;       // first use of the slot: nothing to wait for
            const bool do_w = pass == 0 || !early, do_a = pass == 1;
            const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + SUB_BYTES;
            if (!early) gm_mbar_wait(&empty_bar[s], par ^ 1u);
            if (do_w) {
              rd_mbar_expect_tx(&full_bar[s], tx);
              gm_tma_2d(sa + GM_A_BYTES, mw, wk, r0, &full_bar[s]);
              if (nb > 1) gm_tma_2d(sa + GM_A_BYTES + W_BYTES, mw, wk, r1, &full_bar[s]);
              if (nb > 2) gm_tma_2d(sa + GM_A_BYTES + 2 * W_BYTES, mw, wk, r2, &full_bar[s]);
              if (X3) {
                gm_tma_2d(sb + GM_A_BYTES, mw2, wk, r0, &full_bar[s]);
                if (nb > 1) gm_tma_2d(sb + GM_A_BYTES + W_BYTES, mw2, wk, r1, &full_bar[s]);
                if (nb > 2) gm_tma_2d(sb + GM_A_BYTES + 2 * W_BYTES, mw2, wk, r2, &full_bar[s]);
              }
            }
            if (do_a) {
              gm_tma_2d(sa, ma, ak, m0, &full_bar[s]);
              if (X3) gm_tma_2d(sb, ma2, ak, m0, &full_bar[s]);
            }
          }
          if (pass == 0 && it >= (uint32_t)GM_STAGES) break;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (gm_elect_one()) {   // ===== MMA issuer =====
      // A K block is four small MMAs per slab (128 x 64 x 8): ~130 tensor-pipe cycles.  What a CTA can sustain is set by
      // THIS thread's instruction stream (measured: ~860 cycles per K block whatever the ring depth, tile width or
      // operand source, profiles/r3t_dreamer_kdense_analysis.txt), so the loop is kept to the barrier wait, one
      // descriptor addition per instruction and the issue itself.
      uint32_t it = 0, touched = 0;
      const uint32_t lo_base = gm_desc_lo(smem_base);
      for (int p = 0; p < g.n_phases; ++p) {
        const GemmPhase& ph = g.ph[p];
        const int nb = ph.nb, kbs = ph.k_blocks;
        uint32_t dcol[3], fresh[3], dsm[3], fresh_sm[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int a = i < nb ? ph.acc[i] : 0;
          dcol[i] = tmem + (uint32_t)(a * BN);
          fresh[i] = i < nb ? (((touched >> a) & 1u) ^ 1u) : 0u;   // first instruction into this accumulator overwrites
          if (i < nb) touched |= 1u << a;
          const int b = (X3 && i < nb) ? ph.acc_small[i] : 0;
          dsm[i] = tmem + (uint32_t)(b * BN);
          fresh_sm[i] = (X3 && i < nb) ? (((touched >> b) & 1u) ^ 1u) : 0u;
          if (X3 && i < nb) touched |= 1u << b;
        }
        for (int kb = 0; kb < kbs; ++kb, ++it) {
          const uint32_t s = it % GM_STAGES, par = (it / GM_STAGES) & 1u;
          gm_mbar_wait(&full_bar[s], par);
          gm_tc_fence_after();
          if (it == 0) GM_TRD(2);
          const uint32_t a_lo = lo_base + s * (STAGE_BYTES >> 4);
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            if (i < nb) {
              const uint32_t w_lo = a_lo + ((GM_A_BYTES + i * W_BYTES) >> 4);
              const uint32_t acc0 = (kb > 0) ? 1u : (fresh[i] ^ 1u);
              if (X3) {   // the two cross products of this K block: A_lo W_hi, then A_hi W_lo, into the small accumulator
                const uint32_t a2 = a_lo + (SUB_BYTES >> 4), w2 = w_lo + (SUB_BYTES >> 4);
                const uint32_t sm0 = (kb > 0) ? 1u : (fresh_sm[i] ^ 1u);
#pragma unroll
                for (int k = 0; k < GM_BK / 8; ++k)
                  gm_mma_tf32(dsm[i], gm_desc(a2 + 2 * k), gm_desc(w_lo + 2 * k), IDESC, k > 0 ? 1u : sm0);
#pragma unroll
                for (int k = 0; k < GM_BK / 8; ++k)
                  gm_mma_tf32(dsm[i], gm_desc(a_lo + 2 * k), gm_desc(w2 + 2 * k), IDESC, 1u);
              }
#pragma unroll
              for (int k = 0; k < GM_BK / 8; ++k)   // UMMA_K = 8 TF32 = 32 bytes along the swizzled row
                gm_mma_tf32(dcol[i], gm_desc(a_lo + 2 * k), gm_desc(w_lo + 2 * k), IDESC, k > 0 ? 1u : acc0);
            }
          }
          gm_commit(&empty_bar[s]);   // the slot is free once these MMAs have read it
        }
      }
      gm_commit(&acc_bar);            // accumulators complete
      GM_TRD(3);
    }
    __syncwarp();
  } else {
    // ===== epilogue: warp w owns TMEM lanes 32*(w%4) .. +31 = tile rows; the GM_EPI_GROUPS warps that share a lane
    // quarter split the tile's columns.  (Per-CTA clock stamps: after the issuer fix the epilogue -- one warp per
    // scheduler working through 64 columns of bias / activation / TF32 split / row-strided stores -- was 6-7 us of a
    // 14 us actor layer and 21 us of the GRU cell, profiles/r3t_dreamer_kdense_analysis.txt.) =====
    const int q = warp & 3;
    const int part = (warp - 2) >> 2;                        // 0 .. EW - 1
    constexpr int PART_COLS = (EPI == EPI_DENSE ? BN : GM_BN) / EW;
    const int cbeg = part * PART_COLS, cend = cbeg + PART_COLS;
    const int row = m0 + q * 32 + lane;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const bool live = row < g.M;
    // What does not depend on the accumulators is done here, while the K loop runs: the posterior's normal draws
    // (Philox + Box-Muller: most of that epilogue's arithmetic) and the GRU's previous state (row-strided loads).
    [[maybe_unused]] float zpre[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    if constexpr (EPI == EPI_STOCH && EW == 4) {
      if (live && g.noise == GM_NOISE_PHILOX) {
        const uint32_t gid = g.gid0 + (uint32_t)row;
        gm_normal4(gid, g.step, (uint32_t)(8 * part), RD_STREAM_STOCH, g.key0, g.key1, zpre[0]);
        gm_normal4(gid, g.step, (uint32_t)(8 * part + 4), RD_STREAM_STOCH, g.key0, g.key1, zpre[1]);
      }
    }
    [[maybe_unused]] float hpre[16];
    if constexpr (EPI == EPI_GRU && EW == 4) {
#pragma unroll
      for (int c = 0; c < 16; c += 4) {
        const int col = n0 + part * 16 + c;
        float4 hp = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && col < g.N) {
          hp = *reinterpret_cast<const float4*>(g.hold + (size_t)row * g.ldh + col);
          if (g.hold_lo) {
            const float4 hl = *reinterpret_cast<const float4*>(g.hold_lo + (size_t)row * g.ldh + col);
            hp.x += hl.x; hp.y += hl.y; hp.z += hl.z; hp.w += hl.w;
          }
        }
        hpre[c] = hp.x; hpre[c + 1] = hp.y; hpre[c + 2] = hp.z; hpre[c + 3] = hp.w;
      }
    }
    gm_mbar_wait(&acc_bar, 0, true);
    gm_tc_fence_after();
    if (threadIdx.x == 64) GM_TRD(4);
    // tma_out: this part's 32-column staging tile (hi, lo) in the idle ring, and who shares it
    constexpr int TILE_PARTS = PART_COLS >= 32 ? 1 : 32 / PART_COLS;       // column parts per staging tile
    static_assert(PART_COLS == 16 || PART_COLS % 32 == 0, "staging tiles are 32 columns wide");
    const uint32_t rt = (uint32_t)(q * 32 + lane);                          // tile row
    if constexpr (EPI == EPI_DENSE) {
#pragma unroll 1
      for (int c0 = cbeg; c0 < cend; c0 += 16) {
        if (n0 + c0 >= g.N) break;   // warp-uniform
        float v[16];
        gm_tmem_sum16(tl + c0, g.n_acc, 1, v, BN);
        const uint32_t s_hi = smem_base + (uint32_t)(c0 >> 5) * (2u * GM_A_BYTES), s_lo = s_hi + GM_A_BYTES;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const int col = n0 + c0 + j;
          if ((live || g.tma_out) && col < g.N) {   // N % 4 == 0
            float4 o, ol;
            float* po = &o.x;
            float* pl = &ol.x;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              float x = v[j + t] + __ldg(g.bias + col + t);
              if (g.act) x = gm_elu(x);
              po[t] = gm_round_tf32(x);
              pl[t] = gm_round_tf32(x - po[t]);
            }
            if (g.tma_out) {
              gm_stage_f4(s_hi, rt, (c0 + j) & 31, o);
              if (g.out_lo) gm_stage_f4(s_lo, rt, (c0 + j) & 31, ol);
            } else {
              *reinterpret_cast<float4*>(g.out + (size_t)row * g.ldo + col) = o;
              if (g.out_lo) *reinterpret_cast<float4*>(g.out_lo + (size_t)row * g.ldo + col) = ol;
            }
          }
        }
      }
      if (g.tma_out) {
#pragma unroll 1
        for (int t0 = cbeg & ~31; t0 < cend; t0 += 32) {   // the 32-column tiles this part contributes to (one, unless PART_COLS > 32)
          const uint32_t s_hi = smem_base + (uint32_t)(t0 >> 5) * (2u * GM_A_BYTES);
          gm_tiles_out(1 + (t0 >> 5), 128 * TILE_PARTS, (part % TILE_PARTS) == 0 && q == 0 && lane == 0, n0 + t0 < g.N, &maps.o[0],
                       g.out_lo ? &maps.o[1] : nullptr, n0 + t0, m0, s_hi, s_hi + GM_A_BYTES);
        }
      }
    } else if constexpr (EPI == EPI_GRU) {
      // tf.keras GRUCell (reset_after=True): z, r, h gates; bias[0] input side, bias[1] recurrent side
      const int H = g.N;
      const float* bx = g.bias;
      const float* bh = g.bias + 3 * H;
#pragma unroll
      for (int c0 = cbeg; c0 < cend; c0 += 8) {   // (unrolled: hpre is indexed statically)
        if (n0 + c0 >= H) break;
        float az[8], ar[8], axh[8], arh[8];
        gm_tmem_sum8(tl + 0 * GM_BN + c0, g.n_acc, 4, az);    // accumulator a of gate q sits at column (4 a + q) * 64
        gm_tmem_sum8(tl + 1 * GM_BN + c0, g.n_acc, 4, ar);
        gm_tmem_sum8(tl + 2 * GM_BN + c0, g.n_acc, 4, axh);
        gm_tmem_sum8(tl + 3 * GM_BN + c0, g.n_acc, 4, arh);
#pragma unroll
        for (int j = 0; j < 8; j += 4) {
          const int col = n0 + c0 + j;
          if (live && col < H) {   // (rows >= M stage nothing: the copy engine clips them)
            float4 hp;
            if constexpr (EW == 4) {
              const int c = (c0 - cbeg + j) & 15;
              hp = make_float4(hpre[c], hpre[c + 1], hpre[c + 2], hpre[c + 3]);
            } else {
              hp = *reinterpret_cast<const float4*>(g.hold + (size_t)row * g.ldh + col);
              if (g.hold_lo) {
                const float4 hl = *reinterpret_cast<const float4*>(g.hold_lo + (size_t)row * g.ldh + col);
                hp.x += hl.x; hp.y += hl.y; hp.z += hl.z; hp.w += hl.w;
              }
            }
            const float* ph_ = &hp.x;
            float4 o, ol;
            float* po = &o.x;
            float* pl = &ol.x;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int c = col + t;
              const float z = gm_sigmoid((az[j + t] + __ldg(bx + c)) + __ldg(bh + c));
              const float r = gm_sigmoid((ar[j + t] + __ldg(bx + H + c)) + __ldg(bh + H + c));
              const float hh = tanhf((axh[j + t] + __ldg(bx + 2 * H + c)) + r * (arh[j + t] + __ldg(bh + 2 * H + c)));
              const float hn = z * ph_[t] + (1.f - z) * hh;
              po[t] = gm_round_tf32(hn);
              pl[t] = gm_round_tf32(hn - po[t]);
            }
            if (g.tma_out) {
              const uint32_t s_hi = smem_base + (uint32_t)(c0 >> 5) * (2u * GM_A_BYTES);
              gm_stage_f4(s_hi, rt, (c0 + j) & 31, o);
              if (g.out_lo) gm_stage_f4(s_hi + GM_A_BYTES, rt, (c0 + j) & 31, ol);
            } else {
              *reinterpret_cast<float4*>(g.out + (size_t)row * g.ldo + col) = o;
              if (g.out_lo) *reinterpret_cast<float4*>(g.out_lo + (size_t)row * g.ldo + col) = ol;
            }
          }
        }
      }
      if (g.tma_out) {
#pragma unroll 1
        for (int t0 = cbeg & ~31; t0 < cend; t0 += 32) {
          const uint32_t s_hi = smem_base + (uint32_t)(t0 >> 5) * (2u * GM_A_BYTES);
          gm_tiles_out(1 + (t0 >> 5), 128 * TILE_PARTS, (part % TILE_PARTS) == 0 && q == 0 && lane == 0, n0 + t0 < H, &maps.o[0],
                       g.out_lo ? &maps.o[1] : nullptr, n0 + t0, m0, s_hi, s_hi + GM_A_BYTES);
        }
      }
    } else if constexpr (EPI == EPI_STOCH) {
      // RSSM posterior [REF models.py:69-73]: mean, std = split(x); std = softplus(std) + 0.1; stoch = mean + std * eps
      if constexpr (EW == 4) {
        // part p owns latents 8p .. 8p + 7: their means are accumulator columns 8p .. 8p + 7, their raw deviations
        // columns 30 + 8p .. 37 + 8p = entries 6 .. 13 of the 16 columns from 24 + 8p; two TMEM reads per accumulator
        // instead of four, whole 16-byte stores (latent slots 30 / 31 of the row are the action's: k_actor_mode
        // fills them later in the step, the zero written here is never read as anything but a zero-weight input)
        float mu[8], sr[16];
        gm_tmem_sum8(tl + 8 * part, g.n_acc, 1, mu);
        gm_tmem_sum16(tl + 24 + 8 * part, g.n_acc, 1, sr);
        if (live) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int j0 = 8 * part + 4 * h;
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f), ol = o;
            float* po = &o.x;
            float* pl = &ol.x;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int j = j0 + t;
              if (j < GM_STOCH) {
                const float mean = mu[4 * h + t] + __ldg(g.bias + j);
                const float sd = gm_softplus(sr[6 + 4 * h + t] + __ldg(g.bias + GM_STOCH + j)) + 0.1f;
                float e = zpre[h][t];
                if (g.noise == GM_NOISE_EXPLICIT) e = g.eps[(size_t)row * g.ld_eps + j];
                const float sv = mean + sd * e;
                po[t] = gm_round_tf32(sv);
                pl[t] = gm_round_tf32(sv - po[t]);
                if (g.dbg) { g.dbg[(size_t)row * 2 * GM_STOCH + j] = mean; g.dbg[(size_t)row * 2 * GM_STOCH + GM_STOCH + j] = sd; }
              }
            }
            *reinterpret_cast<float4*>(g.feat + (size_t)row * g.ldf + j0) = o;
            if (g.feat_lo) *reinterpret_cast<float4*>(g.feat_lo + (size_t)row * g.ldf + j0) = ol;
          }
        }
      } else {
      float lo[32], hi[32];
      {
        float t[16];
        gm_tmem_sum16(tl + 0, g.n_acc, 1, t);
#pragma unroll
        for (int i = 0; i < 16; ++i) lo[i] = t[i];
        gm_tmem_sum16(tl + 16, g.n_acc, 1, t);
#pragma unroll
        for (int i = 0; i < 16; ++i) lo[16 + i] = t[i];
        gm_tmem_sum16(tl + 32, g.n_acc, 1, t);
#pragma unroll
        for (int i = 0; i < 16; ++i) hi[i] = t[i];
        gm_tmem_sum16(tl + 48, g.n_acc, 1, t);
#pragma unroll
        for (int i = 0; i < 16; ++i) hi[16 + i] = t[i];
      }
      if (live) {
        float* frow = g.feat + (size_t)row * g.ldf;
        const uint32_t gid = g.gid0 + (uint32_t)row;
#pragma unroll
        for (int j0 = 0; j0 < 32; j0 += 4) {
          if (j0 / (32 / EW) != part) continue;   // warp-uniform: this group's share of the 30 latents
          float z[4] = {0.f, 0.f, 0.f, 0.f};
          if (g.noise == GM_NOISE_PHILOX) gm_normal4(gid, g.step, (uint32_t)j0, RD_STREAM_STOCH, g.key0, g.key1, z);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int j = j0 + t;
            if (j < GM_STOCH) {
              const float mean = lo[j] + __ldg(g.bias + j);
              const float sraw = (j + GM_STOCH < 32 ? lo[(j + GM_STOCH) & 31] : hi[(j + GM_STOCH - 32) & 31]) + __ldg(g.bias + GM_STOCH + j);
              const float sd = gm_softplus(sraw) + 0.1f;
              float e = z[t];
              if (g.noise == GM_NOISE_EXPLICIT) e = g.eps[(size_t)row * g.ld_eps + j];
              const float sv = mean + sd * e;
              const float sh = gm_round_tf32(sv);
              frow[j] = sh;
              if (g.feat_lo) g.feat_lo[(size_t)row * g.ldf + j] = gm_round_tf32(sv - sh);
              if (g.dbg) { g.dbg[(size_t)row * 2 * GM_STOCH + j] = mean; g.dbg[(size_t)row * 2 * GM_STOCH + GM_STOCH + j] = sd; }
            }
          }
        }
      }
      }   // EW != 4
    } else {
      // hout: the four pre-activations of the ActionDecoder head, in full float32; the head itself and
      // SampleDist.mode() need many more threads than this tile has rows (k_actor_mode)
      float v[8];
      gm_tmem_sum8(tl, g.n_acc, 1, v);
      if (live && part == 0) {
        float4 o;
        o.x = v[0] + __ldg(g.bias + 0); o.y = v[1] + __ldg(g.bias + 1); o.z = v[2] + __ldg(g.bias + 2); o.w = v[3] + __ldg(g.bias + 3);
        *reinterpret_cast<float4*>(g.out + (size_t)row * 4) = o;
      }
    }
    gm_tc_fence_before();
    if (threadIdx.x == 64) GM_TRD(5);
  }
  __syncthreads();
  if (warp == 1) {
    gm_tc_fence_after();
    gm_tmem_free(tmem, TM_COLS);
  }
#ifdef GM_CHAIN_TRACE
  if (threadIdx.x == 0 && g.step == 40u && blockIdx.x % 16 == 0)
    printf("DENSE epi %d cta (%d,%d): inputs ready %lld | first full %lld | MMAs issued %lld | acc ready %lld | epilogue done %lld | end %lld\n",
           EPI, blockIdx.x, blockIdx.y, trd[1] - trd[0], trd[2] - trd[0], trd[3] - trd[0], trd[4] - trd[0], trd[5] - trd[0], clock64() - trd[0]);
#endif
#undef GM_TRD
}

// ActionDecoder distribution head [REF models.py:323-346]: mean and sd of the pre-tanh Normal from hout's
// pre-activations g.out[row][0..3]
__device__ __forceinline__ void gm_actor_dist(const GemmArgs& g, int row, float (&mean)[2], float (&sd)[2]) {
  const float4 x4 = *reinterpret_cast<const float4*>(g.out + (size_t)row * 4);
  float x[4] = {x4.x, x4.y, x4.z, x4.w};
  if (g.bn) {   // 'normalized_tanhtransformed_normal': BatchNormalization in inference mode, linear mean
#pragma unroll
    for (int t = 0; t < 4; ++t)
      x[t] = (x[t] - __ldg(g.bn + 8 + t)) * (__ldg(g.bn + t) * rsqrtf(__ldg(g.bn + 12 + t) + g.bn_eps)) + __ldg(g.bn + 4 + t);
    mean[0] = x[0]; mean[1] = x[1];
    sd[0] = gm_softplus(x[2]) + g.min_std; sd[1] = gm_softplus(x[3]) + g.min_std;
  } else {      // 'tanh_normal'
    mean[0] = g.mean_scale * tanhf(x[0] / g.mean_scale); mean[1] = g.mean_scale * tanhf(x[1] / g.mean_scale);
    sd[0] = gm_softplus(x[2] + g.raw_init_std) + g.min_std; sd[1] = gm_softplus(x[3] + g.raw_init_std) + g.min_std;
  }
}
// the chosen action -> g.actions[row] and the latent's action slots (TF32 hi [+ lo]), which the next img1 reads
__device__ __forceinline__ void gm_actor_store(const GemmArgs& g, int row, float a0, float a1) {
  g.actions[2 * (size_t)row] = a0;
  g.actions[2 * (size_t)row + 1] = a1;
  float* frow = g.feat + (size_t)row * g.ldf;
  const float h0 = gm_round_tf32(a0), h1 = gm_round_tf32(a1);
  frow[GM_STOCH] = h0;
  frow[GM_STOCH + 1] = h1;
  if (g.feat_lo) {
    g.feat_lo[(size_t)row * g.ldf + GM_STOCH] = gm_round_tf32(a0 - h0);
    g.feat_lo[(size_t)row * g.ldf + GM_STOCH + 1] = gm_round_tf32(a1 - h1);
  }
}

// ActionDecoder distribution head + SampleDist.mode() [REF ros_agent/helpers/tools.py:70-73]:
// one warp per env, lanes over pairs of draws (one Philox block = the four normals of two draws), warp arg-max.
// `g.out` holds hout's pre-activations [M][4] (k_dense<EPI_ACTOR>); the other fields are the ACTOR ones of GemmArgs.
__global__ void __launch_bounds__(256) k_actor_mode(const GemmArgs g) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= g.M) return;
  // Launched while the head's k_dense still runs (programmatic dependent launch): the normal draws -- Philox and
  // Box-Muller, most of this kernel's arithmetic -- depend on nothing it produces and are made before the wait.
  constexpr int PRE = 4;   // draws 2 lane + 64 it, it < PRE, kept in registers; beyond 256 draws they are made in the loop
  float zp[PRE][4];
  if (g.noise == GM_NOISE_PHILOX) {
#pragma unroll
    for (int it = 0; it < PRE; ++it)
      if (2 * lane + 64 * it < g.n_samples)
        gm_normal4(g.gid0 + (uint32_t)row, g.step, (uint32_t)(2 * lane + 64 * it), RD_STREAM_ACTOR, g.key0, g.key1, zp[it]);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  float mean[2], sd[2];
  gm_actor_dist(g, row, mean, sd);
  // mode(): argmax over n_samples draws of log_prob(tanh(u)), u ~ N(mean, sd): the Normal's log density minus the tanh
  // bijector's forward log-det-Jacobian 2 (log 2 - u - softplus(-2u)), summed over the two actions
  const float log2f_ = 0.69314718f, half_log_2pi = 0.91893853f;
  const uint32_t gid = g.gid0 + (uint32_t)row;
  float best = -INFINITY, bu0 = mean[0], bu1 = mean[1];
  int bi = 0x7fffffff;
  if (g.noise == GM_NOISE_ZERO) {
    bi = 0;
    best = 0.f;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      const float u = mean[d];
      best += (-logf(sd[d]) - half_log_2pi) - 2.f * ((log2f_ - u) - gm_softplus(-2.f * u));
    }
  } else {
    int it = 0;
#pragma unroll 1
    for (int s0 = 2 * lane; s0 < g.n_samples; s0 += 64, ++it) {
      float z[4] = {0.f, 0.f, 0.f, 0.f};
      if (g.noise == GM_NOISE_PHILOX) {
        if (it < PRE) {
#pragma unroll
          for (int k = 0; k < PRE; ++k)
            if (k == it) { z[0] = zp[k][0]; z[1] = zp[k][1]; z[2] = zp[k][2]; z[3] = zp[k][3]; }
        } else {
          gm_normal4(gid, g.step, (uint32_t)s0, RD_STREAM_ACTOR, g.key0, g.key1, z);
        }
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int s = s0 + h;
        if (s >= g.n_samples) break;
        float lp = 0.f, u[2];
#pragma unroll
        for (int d = 0; d < 2; ++d) {
          const float e = (g.noise == GM_NOISE_EXPLICIT) ? g.eps[(size_t)row * g.ld_eps + 2 * s + d] : z[2 * h + d];
          u[d] = mean[d] + sd[d] * e;
          lp += ((-0.5f * e * e - logf(sd[d])) - half_log_2pi) - 2.f * ((log2f_ - u[d]) - gm_softplus(-2.f * u[d]));
        }
        if (lp > best) { best = lp; bu0 = u[0]; bu1 = u[1]; bi = s; }   // ascending s per lane: first maximum
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {   // tf.argmax: the first maximum over all draws
      const float ob = __shfl_xor_sync(0xffffffffu, best, off), o0 = __shfl_xor_sync(0xffffffffu, bu0, off),
                  o1 = __shfl_xor_sync(0xffffffffu, bu1, off);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (ob > best || (ob == best && oi < bi)) { best = ob; bu0 = o0; bu1 = o1; bi = oi; }
    }
  }
  if (lane == 0) {
    const float a0 = tanhf(bu0), a1 = tanhf(bu1);
    gm_actor_store(g, row, a0, a1);
    if (g.dbg) {
      float* d = g.dbg + (size_t)row * 8;
      d[0] = mean[0]; d[1] = mean[1]; d[2] = sd[0]; d[3] = sd[1]; d[4] = a0; d[5] = a1; d[6] = best; d[7] = (float)bi;
    }
  }
}

// Dreamer.policy(training=True)'s head [REF dreamer/dreamer.py, Dreamer.policy and _exploration]: ONE draw of the
// ActionDecoder distribution, a = tanh(mean + sd e1) (`actor(feat).sample()`), then the additive Gaussian exploration
// a' = clip(a + amount e2, -1, 1), rounded once per operation so that a' is reproducible bit for bit from a.  a' is the
// executed action and the one the latent keeps for the next obs_step.  One thread per env; noise: Philox block
// (env id, step, 0, RD_STREAM_TRAIN) -> e1 = z0..1, e2 = z2..3, zero (a = tanh(mean), a' = a) or explicit
// (g.eps [M][2] = e1, eps_expl [M][2] = e2).  Debug row: mean, sd, a (before exploration), log_prob(a), index 0.
__global__ void __launch_bounds__(256) k_actor_train(const GemmArgs g, const float* __restrict__ eps_expl, float amount) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= g.M) return;
  float z[4] = {0.f, 0.f, 0.f, 0.f};
  // made before the wait, as in k_actor_mode: the draws do not depend on the head's k_dense
  if (g.noise == GM_NOISE_PHILOX) gm_normal4(g.gid0 + (uint32_t)row, g.step, 0u, RD_STREAM_TRAIN, g.key0, g.key1, z);
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (g.noise == GM_NOISE_EXPLICIT) {
    z[0] = g.eps[2 * (size_t)row]; z[1] = g.eps[2 * (size_t)row + 1];
    z[2] = eps_expl[2 * (size_t)row]; z[3] = eps_expl[2 * (size_t)row + 1];
  }
  float mean[2], sd[2];
  gm_actor_dist(g, row, mean, sd);
  const float log2f_ = 0.69314718f, half_log_2pi = 0.91893853f;
  float a[2], x[2], lp = 0.f;
#pragma unroll
  for (int d = 0; d < 2; ++d) {
    const float e = z[d], u = mean[d] + sd[d] * e;
    lp += ((-0.5f * e * e - logf(sd[d])) - half_log_2pi) - 2.f * ((log2f_ - u) - gm_softplus(-2.f * u));
    a[d] = tanhf(u);
    x[d] = fminf(fmaxf(__fadd_rn(a[d], __fmul_rn(amount, z[2 + d])), -1.f), 1.f);
  }
  gm_actor_store(g, row, x[0], x[1]);
  if (g.dbg) {
    float* d = g.dbg + (size_t)row * 8;
    d[0] = mean[0]; d[1] = mean[1]; d[2] = sd[0]; d[3] = sd[1]; d[4] = a[0]; d[5] = a[1]; d[6] = lp; d[7] = 0.f;
  }
}

// Weight refresh (rd_policy_dreamer_set_weights): checkpoint arrays -> the policy's packed operands, on the device.
// Job j: src [in][out] -> dst (o, kmap(i)) = tf32(x) and, if lo, tf32(x - tf32(x)), kmap(i) = i >= k_from ? i + k_shift
// : i (dr_upload_t's layout; the K slots it skips keep their zeros); raw jobs copy [out] values as they are (biases,
// BN).  The rounding is dr_tf32's integer one, so the packed bits equal the host packing of rd_policy_dreamer_init.
#define GM_PACK_MAX 32
struct PackJob {
  const float* src; float* hi; float* lo;
  int in, out, ld, k_from, k_shift, raw;
  long long begin;         // first element of the job in the launch's flat index
};
struct PackArgs { int n_jobs; long long total; PackJob job[GM_PACK_MAX]; };
__device__ __forceinline__ float gm_tf32_bits(float x) {   // == dr_tf32 (rd_dreamer.cuh)
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & ~0x1fffu);
}
__global__ void __launch_bounds__(256) k_pack_weights(const __grid_constant__ PackArgs a) {
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < a.total; t += (long long)gridDim.x * blockDim.x) {
    int j = 0;
    while (j + 1 < a.n_jobs && t >= a.job[j + 1].begin) ++j;
    const PackJob& J = a.job[j];
    const long long e = t - J.begin;
    const float x = J.src[e];
    if (J.raw) { J.hi[e] = x; continue; }
    const int i = (int)(e / J.out), o = (int)(e % J.out);
    const size_t f = (size_t)o * J.ld + (i >= J.k_from ? i + J.k_shift : i);
    const float h = gm_tf32_bits(x);
    J.hi[f] = h;
    if (J.lo) J.lo[f] = gm_tf32_bits(__fsub_rn(x, h));
  }
}

// RacingDreamer._preprocess_lidar [REF ros_agent/models/dreamer/racing_dreamer.py:45-52] in its own float32 arithmetic
// (clip to [0, 15], / 15, - 0.5; `normalise` = 0 when the env already emits that), then the TF32 split (hi, lo) the
// tensor-core passes read; lo may be null (single-pass mode).  count % 4 == 0.
__global__ void __launch_bounds__(256) k_embed_lidar(const float4* __restrict__ src, float4* __restrict__ hi,
                                                     float4* __restrict__ lo, size_t count4, int normalise) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 x4 = src[i];
    const float* x = &x4.x;
    float4 h4, l4;
    float* h = &h4.x;
    float* l = &l4.x;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float v = x[t];
      if (normalise) {
        v = fminf(fmaxf(v, 0.0f), 15.0f);
        v = __fsub_rn(__fdiv_rn(__fsub_rn(v, 0.0f), 15.0f), 0.5f);
      }
      h[t] = gm_round_tf32(v);
      l[t] = gm_round_tf32(v - h[t]);
    }
    hi[i] = h4;
    if (lo) lo[i] = l4;
  }
}
// latent rows <-> the reference's state tuple.  dir 0: out = hi + lo; dir 1: (hi, lo) = split(in)
__global__ void __launch_bounds__(256) k_latent_copy(float* __restrict__ feat, float* __restrict__ feat_lo, int ldf, int col0,
                                                      int width, float* __restrict__ ext, int n, int dir) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n * width) return;
  const int e = (int)(i / width), c = (int)(i % width);
  const size_t f = (size_t)e * ldf + col0 + c;
  if (dir == 0) {
    ext[i] = feat[f] + (feat_lo ? feat_lo[f] : 0.f);
  } else {
    const float x = ext[i], h = gm_round_tf32(x);
    feat[f] = h;
    if (feat_lo) feat_lo[f] = gm_round_tf32(x - h);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// k_dense_chain: a stack of equally wide Dense + ELU layers (the ActionDecoder trunk [REF models.py:321-322]) in ONE
// launch.  The arithmetic of every layer is k_dense<EPI_DENSE, 1, 4, STAGES, X3 = true, EW, BN>'s, instruction for
// instruction (same K blocks, same accumulator groups, same epilogue), so the results are bitwise those of the
// per-layer launches; what goes away is, per layer, a launch, a CTA set-up (barriers, TMEM, tensor maps) and the
// drain / fill of the whole grid around a kernel boundary.
//   * grid (N tiles, row-block groups): CTA (x, y) owns output columns [x BN, (x + 1) BN) of the 128-env row blocks
//     y, y + gridDim.y, ...  The N tiles of a row block are launched as ONE thread-block cluster, so the hardware runs
//     the CTAs that wait for each other together whatever else occupies the SMs (33 such clusters fit a B200 at once;
//     the host sizes the grid to that to keep the work in one wave).
//   * layer l + 1 of a row block reads what ALL N tiles of layer l wrote for that row block: each CTA bumps the
//     counter flags[l][row block] (stores -> __threadfence -> CTA barrier of the epilogue warps -> atomic) and the
//     producer thread of each CTA waits for it to reach `target[l]` (acquire load, then fence.proxy.async before the
//     TMA reads) -- no grid-wide barrier, row blocks run ahead of each other freely.  Counters only ever grow
//     (the host passes the value they must reach in this launch), so nothing has to be cleared between launches.
//   * while waiting, the producer has already filled the ring with the weight tiles of the layer's first K blocks
//     (weights depend on nothing); the accumulators are handed back and forth between the issuer and the epilogue
//     warps through acc_bar / tmem_free_bar.
// Waits are bounded (trap instead of hang), like gm_mbar_wait.
// ---------------------------------------------------------------------------------------------------------------
#define GM_CHAIN_MAX 4
struct ChainMaps {   // [layer][hi, lo]; layer l stores its output through a[l + 1] (the same rows), the last one through o_last
  CUtensorMap a[GM_CHAIN_MAX][2];
  CUtensorMap w[GM_CHAIN_MAX][2];
  CUtensorMap o_last[2];
  CUtensorMap wh[2];          // ChainArgs::head: the head's weights [4][K] (hi, lo), box 32 x 64 rows
};
struct ChainLayer {
  int kb_total;            // K blocks of the layer
  int n_groups;            // accumulator groups of the hi*hi products (the cross products go to accumulator n_groups)
  int grp_blocks[3];       // K blocks per group
  const float* bias;
  float* out; float* out_lo;
  unsigned target;         // value flags[layer][row block] reaches when every column part of every N tile of this launch
                           // has stored the layer (EW parts per CTA)
};
struct ChainArgs {
  int M, N, ldo, n_layers, row_blocks;
  unsigned* flags;         // [GM_CHAIN_MAX][row_blocks]
  ChainLayer L[GM_CHAIN_MAX];
  // Fused output head (ActionDecoder hout, 4 columns): cluster launches with one row block per cluster only.  The last
  // layer's output tiles never leave shared memory: every CTA multiplies its own 128 columns -- staged as MMA-ready
  // 128-byte-swizzled tiles anyway -- with its K slice of the head's weights, and the cluster's first CTA adds the
  // four partial [128][4] products (distributed shared memory) and the bias.
  int head;
  const float* head_bias;  // [4]
  float* head_out;         // [M][4] pre-activations (k_actor_mode reads them)
};

__device__ __forceinline__ void gm_flag_wait(const unsigned* flag, unsigned target) {
  for (uint32_t spins = 0;; ++spins) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if ((int)(v - target) >= 0) break;
    if (spins > (1u << 22)) __trap();
  }
  asm volatile("fence.proxy.async;" ::: "memory");   // the rows were written through the generic proxy, TMA reads them
}

template <int GM_STAGES, int EW, int BN>
__global__ void __launch_bounds__(64 + 128 * EW, 1)
    k_dense_chain(const __grid_constant__ ChainMaps maps, const ChainArgs g) {
  extern __shared__ uint8_t gm_smem_raw[];
  __shared__ uint64_t full_bar[GM_STAGES], empty_bar[GM_STAGES], acc_bar, tmem_free_bar, epi_done_bar;
  __shared__ uint64_t head_full_bar, stage_ready_bar, head_acc_bar;   // fused head (g.head)
  __shared__ float4 head_red[4][GM_BM];                              // CTA 0 of the cluster: the four partial products
  __shared__ uint32_t tmem_slot;
#ifdef GM_CHAIN_TRACE   // per-role clock stamps of the first row block (tools/gpu_chain_trace.sh)
  __shared__ long long tr[GM_CHAIN_MAX][16];
  __shared__ long long tr0;
#define GM_TR(l, k) do { if (mb == (int)blockIdx.y) tr[l][k] = clock64(); } while (0)
#else
#define GM_TR(l, k) do { } while (0)
#endif
  static_assert(BN % 16 == 0 && BN <= 256 && 4 * BN <= 512, "MMA N and the accumulators' TMEM columns");
  constexpr uint32_t W_BYTES = BN * 128, IDESC = GM_IDESC_N(BN);
  constexpr uint32_t SUB_BYTES = GM_A_BYTES + W_BYTES, STAGE_BYTES = 2u * SUB_BYTES;
  constexpr uint32_t TM_COLS = 512;
  const uint32_t smem_base = (rd_smem_u32(gm_smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN;
  // fused head: this CTA's live 32-column parts, and where the ring stands after the last K block (g.head implies one
  // row block per CTA, so the K blocks of the launch are those of its layers)
  const int head_parts = g.head ? min(EW, (g.N - n0 + 31) / 32) : 0;
  uint32_t head_it = 0;
  for (int l = 0; l < g.n_layers; ++l) head_it += (uint32_t)g.L[l].kb_total;
  // staging tile of part p (see the epilogue) and the idle weight slot that receives the head's K slice for it
  auto head_a_hi = [&](int p) -> uint32_t {
    const uint32_t st = p < 2 ? (head_it + (uint32_t)p) % 3u : (head_it + 2u) % 3u;
    return smem_base + st * STAGE_BYTES + (p == 3 ? GM_A_BYTES : 0u);
  };
  auto head_w_hi = [&](int p) -> uint32_t {   // parts 0, 1 -> W slots of stage head_it % 3; parts 2, 3 -> of the next stage
    const uint32_t st = (head_it + (uint32_t)(p >> 1)) % 3u;
    return smem_base + st * STAGE_BYTES + GM_A_BYTES + (uint32_t)(p & 1) * SUB_BYTES;
  };

  if (threadIdx.x == 0) {
    if (g.head) { gm_prefetch_map(&maps.wh[0]); gm_prefetch_map(&maps.wh[1]); }
    for (int l = 0; l < g.n_layers; ++l) {
      gm_prefetch_map(&maps.a[l][0]); gm_prefetch_map(&maps.a[l][1]);
      gm_prefetch_map(&maps.w[l][0]); gm_prefetch_map(&maps.w[l][1]);
    }
#pragma unroll
    for (int s = 0; s < GM_STAGES; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&full_bar[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&empty_bar[s])));
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&acc_bar)));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rd_smem_u32(&tmem_free_bar)), "r"(4 * EW));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rd_smem_u32(&epi_done_bar)), "r"(EW));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&head_full_bar)));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rd_smem_u32(&stage_ready_bar)), "r"(EW));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rd_smem_u32(&head_acc_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) gm_tmem_alloc(&tmem_slot, TM_COLS);
  gm_tc_fence_before();
  __syncthreads();
  gm_tc_fence_after();
  const uint32_t tmem = tmem_slot;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef GM_CHAIN_TRACE
  if (threadIdx.x == 0) tr0 = clock64();
#endif

  if (warp == 0) {
    if (gm_elect_one()) {   // ===== TMA producer =====
      uint32_t it = 0, tile = 0;
      bool first = true;
      for (int mb = blockIdx.y; mb < g.row_blocks; mb += gridDim.y) {
        const int m0 = mb * GM_BM;
        for (int l = 0; l < g.n_layers; ++l) {
          const CUtensorMap* ma = &maps.a[l][0];
          const CUtensorMap* ma2 = &maps.a[l][1];
          const CUtensorMap* mw = &maps.w[l][0];
          const CUtensorMap* mw2 = &maps.w[l][1];
          const int kbs = g.L[l].kb_total;
          const int pre = kbs < GM_STAGES - 1 ? kbs : GM_STAGES - 1;
          // weight tiles of the first K blocks: they depend on nothing but a free ring slot (the last stage and the
          // activation slots of these ones are the staging space of the epilogue that may still be running)
          for (int j = 0; j < pre; ++j) {
            const uint32_t i = it + (uint32_t)j, s = i % GM_STAGES, par = (i / GM_STAGES) & 1u;
            const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + SUB_BYTES;
            if (i >= (uint32_t)GM_STAGES) gm_mbar_wait(&empty_bar[s], par ^ 1u);
            rd_mbar_expect_tx(&full_bar[s], STAGE_BYTES);
            gm_tma_2d(sa + GM_A_BYTES, mw, j * GM_BK, n0, &full_bar[s]);
            gm_tma_2d(sb + GM_A_BYTES, mw2, j * GM_BK, n0, &full_bar[s]);
          }
          GM_TR(l, 0);
          // the layer's input rows: the kernel in front of this one (first layer) or every N tile of the layer before
          if (first) { asm volatile("griddepcontrol.wait;" ::: "memory"); first = false; }
          if (tile > 0) gm_mbar_wait(&epi_done_bar, (tile - 1) & 1u);   // the copy engine has read the staged tiles
          GM_TR(l, 14);
          if (l > 0) gm_flag_wait(g.flags + (size_t)(l - 1) * g.row_blocks + mb, g.L[l - 1].target);
          GM_TR(l, 1);
          for (int j = 0; j < pre; ++j) {
            const uint32_t s = (it + (uint32_t)j) % GM_STAGES;
            const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + SUB_BYTES;
            gm_tma_2d(sa, ma, j * GM_BK, m0, &full_bar[s]);
            gm_tma_2d(sb, ma2, j * GM_BK, m0, &full_bar[s]);
          }
          for (int j = pre; j < kbs; ++j) {
            const uint32_t i = it + (uint32_t)j, s = i % GM_STAGES, par = (i / GM_STAGES) & 1u;
            const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + SUB_BYTES;
            gm_mbar_wait(&empty_bar[s], par ^ 1u);
            rd_mbar_expect_tx(&full_bar[s], STAGE_BYTES);
            gm_tma_2d(sa + GM_A_BYTES, mw, j * GM_BK, n0, &full_bar[s]);
            gm_tma_2d(sb + GM_A_BYTES, mw2, j * GM_BK, n0, &full_bar[s]);
            gm_tma_2d(sa, ma, j * GM_BK, m0, &full_bar[s]);
            gm_tma_2d(sb, ma2, j * GM_BK, m0, &full_bar[s]);
          }
          it += (uint32_t)kbs;
          ++tile;
        }
      }
      if (g.head) {
        // the head's weights go into ring slots no staging tile uses; the ring is idle once the last MMAs are complete
        gm_mbar_wait(&acc_bar, (tile - 1) & 1u);
        rd_mbar_expect_tx(&head_full_bar, (uint32_t)head_parts * 2u * GM_W_BYTES);
        for (int p = 0; p < head_parts; ++p) {
          const uint32_t w = head_w_hi(p);
          gm_tma_2d(w, &maps.wh[0], n0 + 32 * p, 0, &head_full_bar);
          gm_tma_2d(w + GM_W_BYTES, &maps.wh[1], n0 + 32 * p, 0, &head_full_bar);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (gm_elect_one()) {   // ===== MMA issuer =====
      uint32_t it = 0, tile = 0;
      const uint32_t lo_base = gm_desc_lo(smem_base);
      for (int mb = blockIdx.y; mb < g.row_blocks; mb += gridDim.y) {
        for (int l = 0; l < g.n_layers; ++l, ++tile) {
          if (tile > 0) {   // the epilogue warps have read the accumulators of the tile before
            gm_mbar_wait(&tmem_free_bar, (tile - 1) & 1u);
            gm_tc_fence_after();
          }
          const ChainLayer& L = g.L[l];
          const uint32_t dsm = tmem + (uint32_t)(L.n_groups * BN);
          bool small_fresh = true;
          for (int grp = 0; grp < L.n_groups; ++grp) {
            const uint32_t dcol = tmem + (uint32_t)(grp * BN);
            const int kbs = L.grp_blocks[grp];
            for (int kb = 0; kb < kbs; ++kb, ++it) {
              const uint32_t s = it % GM_STAGES, par = (it / GM_STAGES) & 1u;
              gm_mbar_wait(&full_bar[s], par);
              gm_tc_fence_after();
              if (grp == 0 && kb == 0) GM_TR(l, 2);
              const uint32_t a_lo = lo_base + s * (STAGE_BYTES >> 4);
              const uint32_t w_lo = a_lo + (GM_A_BYTES >> 4);
              const uint32_t a2 = a_lo + (SUB_BYTES >> 4), w2 = w_lo + (SUB_BYTES >> 4);
              const uint32_t sm0 = small_fresh ? 0u : 1u;
              small_fresh = false;
#pragma unroll
              for (int k = 0; k < GM_BK / 8; ++k)
                gm_mma_tf32(dsm, gm_desc(a2 + 2 * k), gm_desc(w_lo + 2 * k), IDESC, k > 0 ? 1u : sm0);
#pragma unroll
              for (int k = 0; k < GM_BK / 8; ++k)
                gm_mma_tf32(dsm, gm_desc(a_lo + 2 * k), gm_desc(w2 + 2 * k), IDESC, 1u);
#pragma unroll
              for (int k = 0; k < GM_BK / 8; ++k)
                gm_mma_tf32(dcol, gm_desc(a_lo + 2 * k), gm_desc(w_lo + 2 * k), IDESC, (k > 0 || kb > 0) ? 1u : 0u);
              gm_commit(&empty_bar[s]);
            }
          }
          gm_commit(&acc_bar);
          GM_TR(l, 3);
        }
      }
      if (g.head) {
        // hout's partial product over this CTA's K slice, straight from the staged output tiles: hi*hi into TMEM
        // columns 0..15, the two cross products into columns 16..31 (N = 16: the head's 4 rows + zero-filled ones)
        gm_mbar_wait(&tmem_free_bar, (tile - 1) & 1u);   // the last layer's accumulators have been read
        gm_mbar_wait(&stage_ready_bar, 0);                // its output tiles are staged (and fenced for the async proxy)
        gm_mbar_wait(&head_full_bar, 0);                  // the weights' K slice has landed
        gm_tc_fence_after();
        constexpr uint32_t IDESC16 = GM_IDESC_N(16);
        for (int p = 0; p < head_parts; ++p) {
          const uint32_t a_hi = gm_desc_lo(head_a_hi(p)), a_lo = a_hi + (SUB_BYTES >> 4);
          const uint32_t w_hi = gm_desc_lo(head_w_hi(p)), w_lo = w_hi + (GM_W_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < GM_BK / 8; ++k)
            gm_mma_tf32(tmem + 16u, gm_desc(a_lo + 2 * k), gm_desc(w_hi + 2 * k), IDESC16, (p > 0 || k > 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < GM_BK / 8; ++k)
            gm_mma_tf32(tmem + 16u, gm_desc(a_hi + 2 * k), gm_desc(w_lo + 2 * k), IDESC16, 1u);
#pragma unroll
          for (int k = 0; k < GM_BK / 8; ++k)
            gm_mma_tf32(tmem, gm_desc(a_hi + 2 * k), gm_desc(w_hi + 2 * k), IDESC16, (p > 0 || k > 0) ? 1u : 0u);
        }
        gm_commit(&head_acc_bar);
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue (k_dense's EPI_DENSE with ELU), then the row block's counter =====
    // Thread = tile row (TMEM lane), so storing straight from registers would put 16 bytes into each of 32 different rows
    // per instruction: 8192 half-sector writes per CTA and layer, measured at 8.5 us of a 16.5 us layer (clock stamps,
    // profiles/r5b_dreamer_chain.txt).  Instead the four warps of a column part build their [128 rows][32 columns]
    // hi and lo tiles in shared memory, in the 128-byte-swizzled layout of the tensor maps the NEXT layer loads its
    // A operand through, and one thread hands each tile to the copy engine (cp.async.bulk.tensor store; rows >= M and
    // columns >= N are clipped by the map).  Staging space: the ring itself -- the producer only prefetches WEIGHT
    // tiles of GM_STAGES - 1 K blocks while an epilogue runs, so their activation slots and the whole remaining stage
    // are idle (it waits for epi_done_bar before it loads activations again).
    const int q = warp & 3;
    const int part = (warp - 2) >> 2;
    constexpr int PART_COLS = BN / EW;
    static_assert(PART_COLS == 32 && GM_STAGES == 3 && EW == 4 && W_BYTES == GM_A_BYTES, "staging tiles overlay a 3-stage ring");
    const int cbeg = part * PART_COLS, cend = cbeg + PART_COLS;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t r = (uint32_t)(q * 32 + lane);     // tile row
    asm volatile("griddepcontrol.wait;" ::: "memory");
    uint32_t tile = 0, it_end = 0;
    for (int mb = blockIdx.y; mb < g.row_blocks; mb += gridDim.y) {
      for (int l = 0; l < g.n_layers; ++l, ++tile) {
        const ChainLayer& L = g.L[l];
        it_end += (uint32_t)L.kb_total;
        // stages it_end % 3 and (it_end + 1) % 3 receive the next tile's first weight tiles; stage (it_end + 2) % 3 is idle
        const uint32_t st = part < 2 ? (it_end + (uint32_t)part) % 3u : (it_end + 2u) % 3u;
        const uint32_t s_hi = smem_base + st * STAGE_BYTES + (part == 3 ? GM_A_BYTES : 0u), s_lo = s_hi + SUB_BYTES;
        const bool any = n0 + cbeg < g.N;   // warp-uniform (and uniform over the part's four warps)
        gm_mbar_wait(&acc_bar, tile & 1u, true);
        gm_tc_fence_after();
        if (threadIdx.x == 64) GM_TR(l, 4);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cend; c0 += 16) {
          if (n0 + c0 >= g.N) break;   // warp-uniform
          float v[16];
          gm_tmem_sum16(tl + c0, L.n_groups + 1, 1, v, BN);
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const int col = n0 + c0 + j;
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f), ol = o;
            if (col < g.N) {   // N % 4 == 0
              float* po = &o.x;
              float* pl = &ol.x;
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float x = gm_elu(v[j + t] + __ldg(L.bias + col + t));
                po[t] = gm_round_tf32(x);
                pl[t] = gm_round_tf32(x - po[t]);
              }
            }
            const uint32_t chunk = (uint32_t)((c0 - cbeg + j) >> 2);                 // 16-byte chunk of the 128-byte row
            const uint32_t off = r * 128u + ((chunk ^ (r & 7u)) << 4);               // SWIZZLE_128B
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(s_hi + off), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(s_lo + off), "f"(ol.x), "f"(ol.y), "f"(ol.z), "f"(ol.w) : "memory");
          }
        }
        gm_tc_fence_before();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the tiles were written through the generic proxy
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(rd_smem_u32(&tmem_free_bar)) : "memory");
        asm volatile("bar.sync %0, 128;" ::"r"(1 + part) : "memory");    // the part's four warps
        const bool to_head = g.head && l + 1 == g.n_layers;   // the tiles feed the fused head instead of leaving the SM
        if (q == 0 && lane == 0 && to_head) {
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(rd_smem_u32(&stage_ready_bar)) : "memory");
        } else if (q == 0 && lane == 0) {
          if (any) {
            const CUtensorMap* mo = l + 1 < g.n_layers ? &maps.a[l + 1][0] : &maps.o_last[0];
            const CUtensorMap* mo2 = l + 1 < g.n_layers ? &maps.a[l + 1][1] : &maps.o_last[1];
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                             reinterpret_cast<uint64_t>(mo)), "r"(n0 + cbeg), "r"(mb * GM_BM), "r"(s_hi) : "memory");
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                             reinterpret_cast<uint64_t>(mo2)), "r"(n0 + cbeg), "r"(mb * GM_BM), "r"(s_lo) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            GM_TR(l, 6 + part);
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          }
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(rd_smem_u32(&epi_done_bar)) : "memory");
          if (l + 1 < g.n_layers) {
            if (any) {
              asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
              asm volatile("fence.proxy.async;" ::: "memory");
            }
            GM_TR(l, 10 + part);
            __threadfence();
            atomicAdd(g.flags + (size_t)l * g.row_blocks + mb, 1u);
          }
        }
        if (threadIdx.x == 64) GM_TR(l, 5);
      }
    }
    if (q == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the last tile's stores
    if (g.head && part == 0) {
      // this CTA's partial [128][4] of hout -> slot blockIdx.x of the cluster's first CTA (distributed shared memory).
      // NOTE (why the fused head is opt-in): nothing but the co-scheduling of a cluster and the row-block counters this
      // CTA has consumed tells it that the first CTA is running; the programming model wants a cluster barrier before the
      // first remote access (a plain arrive + wait right after the set-up would do), and racecheck says so.  That
      // variant is not shipped because it could not be re-validated on a GPU (profiles/r5b_dreamer_chain.txt).
      gm_mbar_wait(&head_acc_bar, 0, true);
      gm_tc_fence_after();
      float m8[8], s8[8];
      gm_tmem_ld8(tl, m8);
      gm_tmem_ld8(tl + 16u, s8);
      const float4 v = make_float4(m8[0] + s8[0], m8[1] + s8[1], m8[2] + s8[2], m8[3] + s8[3]);
      uint32_t remote;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(rd_smem_u32(&head_red[blockIdx.x][r])), "r"(0));
      asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    }
    gm_tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    gm_tc_fence_after();
    gm_tmem_free(tmem, TM_COLS);
  }
  if (g.head) {
    // every thread of the cluster arrives; the first CTA waits for the other three's partials, adds them in CTA order
    // and stores hout's pre-activations (the others may exit: nobody writes into their shared memory)
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    if (blockIdx.x == 0) {
      asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
      if (warp >= 2 && ((warp - 2) >> 2) == 0) {
        const int rr = (warp & 3) * 32 + lane;
        const int row = (int)blockIdx.y * GM_BM + rr;
        if (row < g.M) {
          float4 o = head_red[0][rr];
          for (int x = 1; x < (int)gridDim.x; ++x) { const float4 t = head_red[x][rr]; o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
          o.x += __ldg(g.head_bias + 0); o.y += __ldg(g.head_bias + 1); o.z += __ldg(g.head_bias + 2); o.w += __ldg(g.head_bias + 3);
          *reinterpret_cast<float4*>(g.head_out + (size_t)row * 4) = o;
        }
      }
    }
  }
#ifdef GM_CHAIN_TRACE
  if (threadIdx.x == 0 && g.L[0].target == 40u * gridDim.x * EW && (blockIdx.y % 8) == 0)
    for (int l = 0; l < g.n_layers; ++l)
      printf("CHAIN cta (%d,%d) layer %d: W issued %lld | staged tiles read %lld | A issued %lld | first full %lld | MMAs issued %lld | acc ready %lld | "
             "stores issued %lld %lld %lld %lld | stores complete %lld %lld %lld %lld | part 0 counted %lld\n",
             blockIdx.x, blockIdx.y, l, tr[l][0] - tr0, tr[l][14] - tr0, tr[l][1] - tr0, tr[l][2] - tr0, tr[l][3] - tr0, tr[l][4] - tr0,
             tr[l][6] - tr0, tr[l][7] - tr0, tr[l][8] - tr0, tr[l][9] - tr0, tr[l][10] - tr0, tr[l][11] - tr0, tr[l][12] - tr0,
             tr[l][13] - tr0, tr[l][5] - tr0);
#endif
#undef GM_TR
}

// ---------------------------------------------------------------------------------------------------------------
// host side: tensor maps and launches
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*gm_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled through the runtime's driver entry point: the library keeps no link-time dependency on
// libcuda, so it still loads (and exports its symbols) on a machine without a driver.
static inline gm_encode_fn gm_get_encoder() {
  static gm_encode_fn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (gm_encode_fn)p;
  }
  return fn;
}

// float32 matrix [rows][inner] with row pitch ld (elements); box = 32 x box_rows, 128-byte swizzle, zero fill
static inline bool gm_make_map(CUtensorMap* m, const float* base, uint64_t inner, uint64_t rows, uint64_t ld, uint32_t box_rows) {
  gm_encode_fn enc = gm_get_encoder();
  if (!enc) return false;
  if (((uintptr_t)base & 15u) || ((ld * 4) & 15u)) return false;
  cuuint64_t gdim[2] = {inner, rows};
  cuuint64_t gstr[1] = {ld * 4};
  cuuint32_t box[2] = {GM_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int EPI, int NSLAB, int NACC, int GM_STAGES, bool X3 = false, int EW = GM_EPI_GROUPS, int BN = GM_BN>
static inline cudaError_t gm_launch(const GemmMaps& maps, const GemmArgs& g, cudaStream_t s) {
  constexpr size_t smem = (size_t)GM_STAGES * (X3 ? 2 : 1) * (GM_A_BYTES + NSLAB * BN * 128) + 1024;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(k_dense<EPI, NSLAB, NACC, GM_STAGES, X3, EW, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((g.M + GM_BM - 1) / GM_BM), (unsigned)((g.N + BN - 1) / BN));
  cfg.blockDim = dim3(64 + 128 * EW);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // see griddepcontrol in k_dense
  attrs[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_dense<EPI, NSLAB, NACC, GM_STAGES, X3, EW, BN>, maps, g);
}

template <int GM_STAGES, int EW, int BN>
// g.head != 0 asks for the fused output head; *head_fused tells whether this launch could take it (cluster launch, one
// row block per cluster) -- if not, the caller runs the head as a k_dense launch of its own.
static inline cudaError_t gm_launch_chain(const ChainMaps& maps, const ChainArgs& g_in, int sm_count, bool cluster, cudaStream_t s,
                                          bool* head_fused) {
  ChainArgs g = g_in;
  constexpr size_t smem = (size_t)GM_STAGES * 2 * (GM_A_BYTES + BN * 128) + 1024;
  static bool attr = false;
  static int max_clusters = -1;   // co-resident clusters of this shape on this device (cluster launches)
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(k_dense_chain<GM_STAGES, EW, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  const int nt = (g.N + BN - 1) / BN;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(64 + 128 * EW);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attrs[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  // The CTAs of a row block wait for each other's counters, so they must run together.  As a thread-block cluster
  // (the N tiles of a row block = one cluster) the hardware guarantees exactly that, whatever else occupies the SMs;
  // the grid is then sized to the clusters that fit at once only to keep the work in one wave.  Without clusters the
  // guarantee is the grid size (one CTA per SM, whole row-block groups, CTAs dispatched in index order).
  int groups = std::max(1, std::min(g.row_blocks, sm_count / nt));
  if (cluster && nt <= 8) {
    attrs[1].id = cudaLaunchAttributeClusterDimension;
    attrs[1].val.clusterDim.x = (unsigned)nt; attrs[1].val.clusterDim.y = 1; attrs[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
    if (max_clusters < 0) {
      cfg.gridDim = dim3((unsigned)nt, (unsigned)groups);
      int q = 0;
      cudaError_t e = cudaOccupancyMaxActiveClusters(&q, k_dense_chain<GM_STAGES, EW, BN>, &cfg);
      if (e != cudaSuccess) return e;
      max_clusters = std::max(1, q);
      if (std::getenv("RD_DREAMER_DEBUG")) std::fprintf(stderr, "k_dense_chain: %d clusters of %d CTAs fit at once\n", max_clusters, nt);
    }
    groups = std::min(groups, max_clusters);
  }
  g.head = (g.head && cfg.numAttrs == 2 && groups == g.row_blocks && nt <= 4) ? 1 : 0;
  if (head_fused) *head_fused = g.head != 0;
  cfg.gridDim = dim3((unsigned)nt, (unsigned)groups);
  return cudaLaunchKernelEx(&cfg, k_dense_chain<GM_STAGES, EW, BN>, maps, g);
}
