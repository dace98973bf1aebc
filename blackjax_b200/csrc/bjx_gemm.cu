// Batched dense linear map for the large-D dense metric / dense Gaussian target (SURVEY K8, VERDICT N1):
//   Y[R, N] = epilogue( X[R, K] . A[N, K]^T , Cin[R, N] )            (A symmetric: M^-1, precision; or L^-T)
// = the reference's `linear_map(M^-1, p)` / `-P x` / `L^-T z` (blackjax/util.py:23-61, lax.dot with
// precision="highest"; call sites mcmc/integrators.py:242, mcmc/metrics.py:263-270) for all chains at once.
//
// Hand-written sm_100a kernel: TMA (cp.async.bulk.tensor) operand loads into 128B-swizzled shared memory, one thread
// issuing tcgen05.mma.cta_group::2 (a CTA pair shares one 256 x 256 accumulator tile: 128 rows per CTA in TMEM, each
// CTA stages half of the constant matrix's rows), two TMEM accumulator buffers so the epilogue of tile i runs under
// the MMAs of tile i+1, epilogue through tcgen05.ld -> registers -> swizzled shared memory -> TMA stores.
//
// float32 accuracy on the fp16 tensor-core path.  One TF32/BF16/FP16 MMA (11/8/11-bit significands) cannot meet the
// 1e-5 parity tolerance, so every float32 operand is split into two binary16 terms x = x1 + x2 (+ a residual below
// 2^-22 |x|) and the three cross products above that residual are accumulated in float32 in TMEM:
//     x.a  ~=  x1 a1 + x2 a1 + x1 a2                      (dropped: x2 a2 and the residuals, each <= 2^-22 |x a|)
// Operand planes are stored [rows, 2, KP] = (x1 | x2): per 64-deep K block the producer stages FOUR tiles
// (x1, x2, a1, a2) and the issuer runs the THREE products on them -- 2/3 of the shared-memory fill and L2 traffic of
// a plain K' = 3K GEMM over (x1|x2|x1).(a1|a1|a2), and 2/3 of the plane bytes in HBM.
// binary16 has a 5-bit exponent, so rows / matrices are lifted by a power of two before the split; the per-row
// epilogue factor alpha_r = coef_r * 2^-s_r * 2^-s_A undoes both exactly (and carries per-chain step sizes).
//
// Fused epilogue (the separate operand-split pass of round 1 is gone from the leapfrog loop):
//   lincomb      : y = alpha_r * acc + beta * Cin                 (q <- q + eps_c (p M^-1); v = M^-1 p; g = -(q P))
//   double kick  : y = alpha_r * acc + (alpha_r * acc + Cin)      (two half kicks between leapfrog steps,
//                                                                  integrators.py:134-141,235-239; two rounded FMAs)
//   planes       : the (x1 | x2) planes of y for the NEXT product, lifted by 2^s_r chosen from the row maximum the
//                  previous production of the same variable recorded (any lift that lands the true row maximum in
//                  [2^-3, 2^15.5) is exact to 2^-22 of the row maximum, an 18-binade window; rows that leave it are
//                  re-split by k_planes_fixup in bjx_dense.cu), plus this production's row maximum (atomic max).
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdlib>
#include <mutex>

#include "bjx_gemm.h"

namespace bjx {
namespace {

constexpr int kBM = 128;                 // rows of X per CTA (256 per CTA pair)
constexpr int kBN = 256;                 // output columns per CTA pair
constexpr int kUmmaK = 16;
constexpr int kSub = 32;                 // epilogue sub-tile: 32 float32 columns = one 128-byte swizzle row
constexpr int kNSub = kBN / kSub;
constexpr int kThreads = 256;
constexpr uint32_t kTmemCols = 512;      // two [128 lanes x 256 columns] float32 accumulators
constexpr int kYSlab = 32 * kSub * 4;    // 4 KB: one epilogue warp's 32 rows x 32 float32 columns
constexpr int kPSlab = 32 * kSub * 2;    // 2 KB: the same block as one binary16 plane

// Shared-memory plan of one configuration: BK-deep operand stages (x1, x2, a1, a2 tiles of [128 x BK] binary16 each)
// and, per epilogue warp, a ring of NY float32 slabs (Cin lands in them, y is formed in place and stored from them)
// and NP slabs of plane pairs.
template <int BK, int STAGES, int NY, int NP>
struct Plan {
  static constexpr int kTileBytes = kBM * BK * 2;
  static constexpr int kStageBytes = 4 * kTileBytes;
  static constexpr int kOffY = STAGES * kStageBytes;
  static constexpr int kOffP = kOffY + 4 * NY * kYSlab;
  static constexpr int kOffBar = kOffP + 4 * NP * 2 * kPSlab;
  // barriers: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], cin[4 warps][NY], then the TMEM base slot
  static constexpr int kNumBars = 2 * STAGES + 4 + 4 * NY;
  static constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 16 + 1024;  // + slack to align the base to 1024
  static_assert(kSmemBytes <= 232448, "over the 227 KB dynamic shared memory limit");
  static_assert(BK == 64 || BK == 32, "one swizzle row per tile row: 128-byte or 64-byte swizzle");
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {  // arrivals come from the peer CTA too
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// operand tile [64 x 1 x 128] of a [K, 2, rows] plane tensor into this CTA's shared memory; completion is signalled on
// the LEADER CTA's barrier (cta_group::2: the MMA that consumes both CTAs' tiles is issued there)
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t leader_bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T, 256 x 256 x 16 over the CTA pair
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this shared-memory offset in BOTH CTAs once every MMA issued so far by this thread is done
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float4 lds_f4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

// Shared-memory matrix descriptor of a K-major [rows x BK] binary16 tile in the swizzle TMA writes it in (one swizzle
// row per tile row: 128-byte for BK = 64, 64-byte for BK = 32): 8-row groups 8 * 2BK bytes apart (stride byte offset),
// descriptor version 1 (Blackwell), layout type SWIZZLE_128B (2) / SWIZZLE_64B (4).
template <int BK>
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  const uint32_t lo = ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16);
  const uint32_t hi = ((8u * BK * 2u) >> 4) | (1u << 14) | ((BK == 64 ? 2u : 4u) << 29);
  return (uint64_t)lo | ((uint64_t)hi << 32);
}
// kind::f16 instruction descriptor: D float32, A/B binary16, both K-major, N = 256, M = 256 (over the pair)
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }

}  // namespace

// Cycle counters for timing experiments (GemmEpilogue::debug & 16): where the single-thread roles and epilogue warp 0
// of every CTA spend their time.  Read back through bjx_debug_gemm_counters (not part of the public ABI).
__device__ unsigned long long g_gemm_prof[16];
__device__ __forceinline__ unsigned long long clk() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t));
  return t;
}
#define BJX_PROF_BEGIN(var) unsigned long long var = prof ? clk() : 0ull
#define BJX_PROF_END(var, acc) \
  if (prof) acc += clk() - var

// ---- the kernel ---------------------------------------------------------------------------------------------
// Warp roles (256 threads, one CTA per SM, CTA pairs):
//   warp 0    TMA producer (one thread): this CTA's 128 activation rows and its 128 rows of the constant matrix
//   warp 1    MMA issuer (one thread of the leader CTA)
//   warp 2    TMEM allocation / release
//   warps 4-7 epilogue; warp w owns TMEM lanes [32 (w%4), +32) = 32 rows of this CTA's 128 and runs its OWN pipeline
//             on them: its lane 0 loads Cin slabs by TMA (NY - NP sub-tiles ahead), the warp forms y in place,
//             splits it into planes, and lane 0 stores the slabs by TMA -- no CTA-level barrier in the epilogue.
template <int BK, int STAGES, int NY, int NP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
k_gemm_f16x3(const __grid_constant__ CUtensorMap tm_x,   // [K, 2, M]  binary16 planes of the activations
             const __grid_constant__ CUtensorMap tm_a,   // [K, 2, N]  binary16 planes of the constant matrix
             const __grid_constant__ CUtensorMap tm_c,   // [N, M]     float32 Cin (unused when !has_cin)
             const __grid_constant__ CUtensorMap tm_y,   // [N, M]     float32 Y
             const __grid_constant__ CUtensorMap tm_p,   // [N, 2, M]  binary16 planes of Y (unused when !planes)
             const GemmEpilogue E, const int M, const int N, const int K, const int tiles_n, const int n_tiles) {
  using P = Plan<BK, STAGES, NY, NP>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar0 = base + P::kOffBar;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * STAGES + 2 + a); };
  auto cin_bar = [&](int q, int slot) { return bar0 + 8u * (2 * STAGES + 4 + q * NY + slot); };
  const uint32_t tmem_slot = bar0 + 8u * P::kNumBars;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int nkb = (K + BK - 1) / BK;
  const bool prof = (E.debug & 16) != 0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_x);
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_y);
    if (E.has_cin) prefetch_tmap(&tm_c);
    if (E.planes) prefetch_tmap(&tm_p);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);    // the leader's producer arrives once (+ the bytes of both CTAs' tiles)
      mbar_init(empty_bar(s), 1);   // one multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);   // one multicast tcgen05.commit per tile
      mbar_init(tempty_bar(a), 8);  // 4 epilogue warps x 2 CTAs (the leader's copy is the one waited on)
    }
    for (int q = 0; q < 4; ++q)
      for (int i = 0; i < NY; ++i) mbar_init(cin_bar(q, i), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {  // TMEM: both CTAs of the pair allocate all 512 columns (one CTA per SM: nobody else wants them)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  // Programmatic dependent launch: everything above (descriptor prefetch, barrier init, TMEM allocation, cluster
  // rendezvous) may run while the previous kernel of the stream drains; nothing below touches its outputs earlier.
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp == 0) {
    // ===== TMA producer: four tiles per stage
    if (lane == 0) {
      const uint32_t leader_full0 = mapa(full_bar(0), 0);
      int s = 0;
      uint32_t ph = 0;
      unsigned long long w_empty = 0;
      for (int t = pair; t < n_tiles; t += n_pairs) {
        const int m0 = (t / tiles_n) * (2 * kBM) + (int)rank * kBM;
        const int n0 = (t % tiles_n) * kBN + (int)rank * (kBN / 2);
        for (int kb = 0; kb < nkb; ++kb) {
          BJX_PROF_BEGIN(t0);
          mbar_wait(empty_bar(s), ph ^ 1u);
          BJX_PROF_END(t0, w_empty);
          if (rank == 0) mbar_expect_tx(full_bar(s), 2u * P::kStageBytes);
          const uint32_t st = base + (uint32_t)s * P::kStageBytes;
          const uint32_t fb = leader_full0 + 8u * s;
          tma_load_3d_2sm(st, &tm_x, fb, kb * BK, 0, m0);
          tma_load_3d_2sm(st + 2 * P::kTileBytes, &tm_a, fb, kb * BK, 0, n0);
          tma_load_3d_2sm(st + P::kTileBytes, &tm_x, fb, kb * BK, 1, m0);
          tma_load_3d_2sm(st + 3 * P::kTileBytes, &tm_a, fb, kb * BK, 1, n0);
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
      if (prof) atomicAdd(&g_gemm_prof[3], w_empty);
      // tail: do not leave while commits from the leader's issuer can still arrive on this CTA's barriers
      for (int i = 0; i < STAGES; ++i) {
        mbar_wait(empty_bar(s), ph ^ 1u);
        if (++s == STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread of the leader CTA
    if (rank == 0 && lane == 0) {
      int s = 0, as = 0;
      uint32_t ph = 0, aph = 0;
      unsigned long long w_tempty = 0, w_full = 0;
      BJX_PROF_BEGIN(t_all);
      for (int t = pair; t < n_tiles; t += n_pairs) {
        BJX_PROF_BEGIN(t0);
        mbar_wait_cluster(tempty_bar(as), aph ^ 1u);  // both CTAs' epilogues have drained this accumulator
        BJX_PROF_END(t0, w_tempty);
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)as * kBN;
        for (int kb = 0; kb < nkb; ++kb) {
          BJX_PROF_BEGIN(t1);
          mbar_wait(full_bar(s), ph);
          BJX_PROF_END(t1, w_full);
          tc_fence_after();
          const uint32_t st = base + (uint32_t)s * P::kStageBytes;
          const uint64_t dx1 = umma_desc<BK>(st), dx2 = umma_desc<BK>(st + P::kTileBytes);
          const uint64_t da1 = umma_desc<BK>(st + 2 * P::kTileBytes), da2 = umma_desc<BK>(st + 3 * P::kTileBytes);
#pragma unroll
          for (int k = 0; k < BK / kUmmaK; ++k)  // +32 bytes per 16-element K step inside the swizzle row
            umma_f16_2sm(d, dx1 + 2u * k, da1 + 2u * k, kIdesc, (kb | k) != 0);
#pragma unroll
          for (int k = 0; k < BK / kUmmaK; ++k) umma_f16_2sm(d, dx2 + 2u * k, da1 + 2u * k, kIdesc, 1u);
#pragma unroll
          for (int k = 0; k < BK / kUmmaK; ++k) umma_f16_2sm(d, dx1 + 2u * k, da2 + 2u * k, kIdesc, 1u);
          umma_commit_2sm(empty_bar(s));  // frees the stage in both CTAs when these MMAs have read it
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        umma_commit_2sm(tfull_bar(as));  // accumulator complete: both CTAs' epilogues may read their halves
        if (++as == 2) { as = 0; aph ^= 1u; }
      }
      if (prof) {
        atomicAdd(&g_gemm_prof[0], w_tempty);
        atomicAdd(&g_gemm_prof[1], w_full);
        atomicAdd(&g_gemm_prof[2], clk() - t_all);
        atomicAdd(&g_gemm_prof[9], 1ull);
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: four independent per-warp pipelines over (tile, sub-tile) pairs, numbered i = 8 * local tile + j
    const int q = warp & 3;
    const uint32_t ybuf = base + P::kOffY + (uint32_t)q * NY * kYSlab;
    const uint32_t pbuf = base + P::kOffP + (uint32_t)q * NP * 2 * kPSlab;
    const uint32_t leader_tempty0 = mapa(tempty_bar(0), 0);
    const float mat_unscale = E.mat_unscale ? E.mat_unscale[0] : 1.0f;
    const int my_tiles = pair < n_tiles ? (n_tiles - pair + n_pairs - 1) / n_pairs : 0;
    const int n_sub = my_tiles * kNSub;
    const int row_off = (int)rank * kBM + q * 32;  // this warp's first row inside a pair tile
    // coordinates of sub-tile i: column n0 + 32 j, row m0 of this warp's slab
    auto sub_n = [&](int i) { return ((pair + (i / kNSub) * n_pairs) % tiles_n) * kBN + (i % kNSub) * kSub; };
    auto sub_m = [&](int i) { return ((pair + (i / kNSub) * n_pairs) / tiles_n) * (2 * kBM) + row_off; };
    auto load_cin = [&](int i) {  // lane 0 only; sub-tiles past the last column just flip the barrier's phase
      const uint32_t bar = cin_bar(q, i % NY);
      if (sub_n(i) >= N || (E.debug & 1)) {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
        return;
      }
      mbar_expect_tx(bar, kYSlab);
      tma_load_2d(ybuf + (uint32_t)(i % NY) * kYSlab, &tm_c, bar, sub_n(i), sub_m(i));
    };
    constexpr int kAhead = NY - NP;  // Cin slabs in flight ahead of the one being processed
    if (E.has_cin && lane == 0)
      for (int i = 0; i < kAhead && i < n_sub; ++i) load_cin(i);

    int as = 0;
    uint32_t aph = 0;
    unsigned long long w_tfull = 0, w_cin = 0, w_rd = 0, w_work = 0;
    BJX_PROF_BEGIN(t_all);
    float al = 0.f, sc = 1.f, amax = 0.f;
    int r = 0;
    bool live = false;
    uint32_t tacc = 0;
    for (int i = 0; i < n_sub; ++i) {
      const int j = i % kNSub;
      const int n0s = sub_n(i), m0s = sub_m(i);
      if (lane == 0) {
        // stores up to sub-tile i - NP have been read out of shared memory: their plane slabs and float32 slab are free
        BJX_PROF_BEGIN(t0);
        tma_store_wait_read<NP - 1>();
        BJX_PROF_END(t0, w_rd);
        if (E.has_cin && i + kAhead < n_sub) load_cin(i + kAhead);
      }
      __syncwarp();
      if (j == 0) {  // new tile: per-row factors, then wait for its accumulator
        r = m0s + lane;
        live = r < M;
        // per-row epilogue factor (same expression as the standalone split pass of round 1) and the lift of this row's planes
        al = E.alpha;
        if (live) {
          if (E.alpha_dev) al = E.alpha_dev[r] * E.alpha;
          al = al * (E.x_unscale ? E.x_unscale[r] : 1.0f) * mat_unscale;
        }
        sc = 1.0f;
        if (E.planes && live) sc = plane_lift(E.stale_max[r]);
        amax = 0.f;
        BJX_PROF_BEGIN(t0);
        mbar_wait(tfull_bar(as), aph);
        BJX_PROF_END(t0, w_tfull);
        tc_fence_after();
        tacc = tmem_base + (uint32_t)as * kBN + ((uint32_t)(q * 32) << 16);
      }
      uint32_t acc[32];
      tmem_ld32(tacc + (uint32_t)(j * kSub), acc);
      const bool in_cols = n0s < N;
      BJX_PROF_BEGIN(t2);
      if (E.has_cin) mbar_wait(cin_bar(q, i % NY), (uint32_t)((i / NY) & 1));
      BJX_PROF_END(t2, w_cin);
      tmem_ld_wait();
      BJX_PROF_BEGIN(t3);
      if (j == kNSub - 1) {  // the accumulator has been read: hand it back to the issuer
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(leader_tempty0 + 8u * as);
        if (++as == 2) { as = 0; aph ^= 1u; }
      }
      const uint32_t yb = ybuf + (uint32_t)(i % NY) * kYSlab;
      const uint32_t p1b = pbuf + (uint32_t)(i % NP) * 2 * kPSlab, p2b = p1b + kPSlab;
      uint32_t h1lo0 = 0, h1lo1 = 0, h2lo0 = 0, h2lo1 = 0;
      if (!(E.debug & 8))
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint32_t yo = yb + (uint32_t)lane * 128u + (uint32_t)((c ^ (lane & 7)) << 4);
        float4 y;
        const float a0 = __uint_as_float(acc[4 * c]), a1 = __uint_as_float(acc[4 * c + 1]);
        const float a2 = __uint_as_float(acc[4 * c + 2]), a3 = __uint_as_float(acc[4 * c + 3]);
        if (E.has_cin) {
          const float4 cv = lds_f4(yo);
          if (E.double_kick) {
            y.x = fmaf(al, a0, fmaf(al, a0, cv.x));
            y.y = fmaf(al, a1, fmaf(al, a1, cv.y));
            y.z = fmaf(al, a2, fmaf(al, a2, cv.z));
            y.w = fmaf(al, a3, fmaf(al, a3, cv.w));
          } else {
            y.x = fmaf(al, a0, E.beta * cv.x);
            y.y = fmaf(al, a1, E.beta * cv.y);
            y.z = fmaf(al, a2, E.beta * cv.z);
            y.w = fmaf(al, a3, E.beta * cv.w);
          }
        } else {
          y = make_float4(al * a0, al * a1, al * a2, al * a3);
        }
        sts_f4(yo, y);
        if (E.planes) {
          // past the last column the slab holds no Cin (nothing is loaded there): whatever an earlier sub-tile, tile or
          // kernel left in it must not reach the row maximum
          if (in_cols) amax = fmaxf(fmaxf(amax, fmaxf(fabsf(y.x), fabsf(y.y))), fmaxf(fabsf(y.z), fabsf(y.w)));
          const float s0 = y.x * sc, s1 = y.y * sc, s2 = y.z * sc, s3 = y.w * sc;
          const uint32_t ha = pack_h2(s0, s1), hb = pack_h2(s2, s3);
          const float2 fa = unpack_h2(ha), fb = unpack_h2(hb);
          const uint32_t ra = pack_h2(s0 - fa.x, s1 - fa.y), rb = pack_h2(s2 - fb.x, s3 - fb.y);
          if ((c & 1) == 0) {
            h1lo0 = ha; h1lo1 = hb; h2lo0 = ra; h2lo1 = rb;
          } else {  // eight columns = one 16-byte chunk of the 64-byte-swizzled plane rows
            const uint32_t po = (uint32_t)lane * 64u + (uint32_t)(((c >> 1) ^ ((lane >> 1) & 3)) << 4);
            sts_u4(p1b + po, h1lo0, h1lo1, ha, hb);
            sts_u4(p2b + po, h2lo0, h2lo1, ra, rb);
          }
        }
      }
      fence_proxy_async();  // generic-proxy writes above -> visible to the TMA engine
      __syncwarp();
      BJX_PROF_END(t3, w_work);
      // Invariant: lane 0 commits exactly one bulk group per sub-tile, so the wait_read<NP - 1> above frees the slabs
      // of sub-tile i - NP.  A sub-tile past the last column stores nothing and commits an empty group (valid in the
      // PTX ISA); skipping its commit would let the count of groups fall behind the count of sub-tiles, and the wait
      // would then pass while the last in-column store still reads a slab that is about to be overwritten.
      if (lane == 0) {
        if (in_cols) {
          if (!(E.debug & 4)) tma_store_2d(&tm_y, yb, n0s, m0s);
          if (E.planes && !(E.debug & 2)) {
            tma_store_3d(&tm_p, p1b, n0s, 0, m0s);
            tma_store_3d(&tm_p, p2b, n0s, 1, m0s);
          }
        }
        tma_store_commit();
      }
      if (j == kNSub - 1 && E.planes && live) {
        atomicMax(reinterpret_cast<int*>(E.next_max) + r, __float_as_int(amax));
        E.zero_max[r] = 0.f;
        if (n0s < kBN) E.out_unscale[r] = 1.0f / sc;  // the tile of the first column block writes the lift
      }
    }
    if (lane == 0) tma_store_wait_all();
    if (prof && q == 0 && lane == 0) {
      atomicAdd(&g_gemm_prof[4], w_tfull);
      atomicAdd(&g_gemm_prof[5], w_cin);
      atomicAdd(&g_gemm_prof[6], w_rd);
      atomicAdd(&g_gemm_prof[7], w_work);
      atomicAdd(&g_gemm_prof[8], clk() - t_all);
      atomicAdd(&g_gemm_prof[10], 1ull);
    }
  }

  // teardown: nobody leaves (or frees TMEM) while the peer may still touch this CTA's shared memory / TMEM
  tc_fence_before();
  cluster_sync();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

namespace {
// ---- host side ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// planes tensor [rows, 2, KP] binary16 seen as (K, 2, rows): box (box_k, 1, box_rows)
bool make_plane_map(CUtensorMap* m, const void* ptr, int rows, int K, int KP, int box_k, int box_rows, CUtensorMapSwizzle sw) {
  const cuuint64_t dims[3] = {(cuuint64_t)K, 2, (cuuint64_t)rows};
  const cuuint64_t strides[2] = {(cuuint64_t)KP * 2, (cuuint64_t)KP * 4};
  const cuuint32_t box[3] = {(cuuint32_t)box_k, 1, (cuuint32_t)box_rows};
  const cuuint32_t es[3] = {1, 1, 1};
  return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// float32 [rows, N] seen as (N, rows): box (32, 32) = one epilogue warp's slab, 128-byte swizzle
bool make_row_map(CUtensorMap* m, const void* ptr, int rows, int N) {
  const cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)N * 4};
  const cuuint32_t box[2] = {(cuuint32_t)kSub, 32};
  const cuuint32_t es[2] = {1, 1};
  return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool pdl_enabled() {  // BJX_GEMM_PDL=0 switches programmatic dependent launch off (measurement)
  static const bool on = [] { const char* e = getenv("BJX_GEMM_PDL"); return !(e && e[0] == '0'); }();
  return on;
}

template <int BK, int STAGES, int NY, int NP>
struct Variant {
  using P = Plan<BK, STAGES, NY, NP>;
  static int max_pairs() {
    static int cached = 0;
    static std::once_flag once;
    std::call_once(once, [] {
      int dev = 0, sms = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      cudaFuncSetAttribute(k_gemm_f16x3<BK, STAGES, NY, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, P::kSmemBytes);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(2 * (sms > 0 ? sms : 2));
      cfg.blockDim = dim3(kThreads);
      cfg.dynamicSmemBytes = P::kSmemBytes;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, k_gemm_f16x3<BK, STAGES, NY, NP>, &cfg) == cudaSuccess && n > 0) cached = n;
      else cached = sms / 2 > 0 ? sms / 2 : 1;
      cudaGetLastError();
    });
    return cached;
  }
  static int run(const GemmCall& g, cudaStream_t stream) {
    CUtensorMap tx, ta, tc, ty, tp;
    const CUtensorMapSwizzle sw = BK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    if (!make_plane_map(&tx, g.x_planes, g.M, g.K, g.KP, BK, kBM, sw)) return 3;
    if (!make_plane_map(&ta, g.a_planes, g.N, g.K, g.KP, BK, kBM, sw)) return 4;
    if (!make_row_map(&ty, g.Y, g.M, g.N)) return 5;
    tc = ty;
    if (g.epi.has_cin && g.Cin != g.Y && !make_row_map(&tc, g.Cin, g.M, g.N)) return 6;
    tp = tx;
    if (g.epi.planes && !make_plane_map(&tp, g.planes_out, g.M, g.N, g.KP_out, kSub, 32, CU_TENSOR_MAP_SWIZZLE_64B)) return 7;
    const int tiles_m = (g.M + 2 * kBM - 1) / (2 * kBM), tiles_n = (g.N + kBN - 1) / kBN;
    const int n_tiles = tiles_m * tiles_n;
    const int pairs = n_tiles < max_pairs() ? n_tiles : max_pairs();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = P::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // prologue overlaps the previous kernel's tail
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, k_gemm_f16x3<BK, STAGES, NY, NP>, tx, ta, tc, ty, tp, g.epi, g.M, g.N, g.K,
                                             tiles_n, n_tiles);
    return e == cudaSuccess ? 0 : 8;
  }
};

int variant_id() {  // BJX_GEMM_VARIANT selects an alternative shared-memory plan (measurements in DESIGN.md)
  static int v = [] {
    const char* e = getenv("BJX_GEMM_VARIANT");
    return e ? atoi(e) : 0;
  }();
  return v;
}

}  // namespace

}  // namespace bjx
extern "C" int bjx_debug_gemm_counters(unsigned long long* out16, int reset) {
  cudaDeviceSynchronize();
  if (out16 && cudaMemcpyFromSymbol(out16, bjx::g_gemm_prof, sizeof(bjx::g_gemm_prof)) != cudaSuccess) return 1;
  if (reset) {
    unsigned long long z[16] = {0};
    if (cudaMemcpyToSymbol(bjx::g_gemm_prof, z, sizeof(z)) != cudaSuccess) return 2;
  }
  return 0;
}
namespace bjx {

int gemm_f16x3(const GemmCall& g, cudaStream_t stream) {
  if (!encode_fn()) return 1;
  static const int dbg = [] { const char* e = getenv("BJX_GEMM_DEBUG"); return e ? atoi(e) : 0; }();
  if (dbg) const_cast<GemmCall&>(g).epi.debug = dbg;
  if (g.M <= 0 || g.N <= 0 || g.K <= 0 || (g.N & 3) || (g.KP & 7) || (g.KP_out & 7)) return 2;
  switch (variant_id()) {
    case 1: return Variant<64, 2, 4, 2>::run(g, stream);
    case 2: return Variant<32, 5, 3, 1>::run(g, stream);
    case 3: return Variant<64, 3, 1, 1>::run(g, stream);  // three 64-deep stages leave room for no epilogue ring
    default: return Variant<32, 4, 4, 2>::run(g, stream);
  }
}

}  // namespace bjx
