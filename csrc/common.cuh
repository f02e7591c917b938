// Shared sm_100a device helpers: mbarrier, TMA, tcgen05/TMEM, cluster/DSMEM,
// system-scope flags for the NVLink piece handoff.  Everything is inline PTX —
// no CUTLASS dependency.  Bit layouts follow the PTX ISA tcgen05 descriptors.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2b {

#ifndef B2B_SPIN_LIMIT
#define B2B_SPIN_LIMIT (1u << 27)   // bounded waits: a protocol bug traps instead of hanging the GPU
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() {
  asm volatile("fence.proxy.async;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > B2B_SPIN_LIMIT) { __trap(); }
  }
}

// ---------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tiled load: coordinates are (c0 = innermost/K element index, c1 = row index).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
      "r"(c1)
      : "memory");
}
// Same with an L2 cache-policy hint (weights are streamed once: evict_first).
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* m,
                                                 uint64_t* bar, int c0, int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
      "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// ------------------------------------------------------------ tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM cols: pow2 in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate; single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// fp8 (e4m3) inputs, fp32 accumulate (kind::f8f6f4, non block-scaled).
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// MX block-scaled fp8: e4m3 x e4m3 with one UE8M0 scale per 32 K elements; the scale factors live in
// TMEM (4 columns per 128 rows x 4 k-blocks; the descriptor's sf-id fields pick the k-block byte).
__device__ __forceinline__ void umma_mxf8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate, uint32_t sfa_tmem, uint32_t sfb_tmem) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf8f6f4.block_scale [%0], %1, %2, %3, [%5], [%6], p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(sfa_tmem), "r"(sfb_tmem)
      : "memory");
}
// smem -> TMEM copy of 32 rows x 16 bytes, replicated into the four 32-lane subpartitions (scale factors).
__device__ __forceinline__ void tmem_cp_32x128b_warpx4(uint32_t taddr, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.32x128b.warpx4 [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
// un-swizzled K-major descriptor of a contiguous [32 rows][16 bytes] scale-factor chunk (8-row atoms 128 B apart)
__device__ __forceinline__ uint64_t make_sf_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(128 >> 4) << 32;               // SBO: next 8-row atom
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}
// 1D bulk copy global -> shared with mbarrier transaction accounting (size multiple of 16 bytes)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// tcgen05.commit: arrive on an mbarrier once all previously issued MMAs retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// Each thread of the warp reads its own TMEM lane (warp%4 selects the 32-lane
// quarter via the address), 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major, 128B-swizzled shared-memory operand descriptor (rows of 128 bytes,
// 8-row x 128B swizzle atoms stacked every 1024 bytes).
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);   // start address   [0,14)
  d |= static_cast<uint64_t>(1) << 16;                       // LBO (ignored for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;               // SBO = 1024 B    [32,46)
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
  return d;
}
// Instruction descriptor, kind::f16: bf16 x bf16 -> fp32, both K-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4)      // D format  = F32
       | (1u << 7)      // A format  = BF16
       | (1u << 10)     // B format  = BF16
       | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// kind::f8f6f4 with e4m3 x e4m3 -> fp32 (format code 0 for both).
__host__ __device__ constexpr uint32_t make_idesc_e4m3(uint32_t m, uint32_t n) {
  return (1u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// kind::mxf8f6f4.block_scale, e4m3 x e4m3, UE8M0 scales: [4,6) b_sf_id, [23] scale format E8M0, [29,31) a_sf_id
__host__ __device__ constexpr uint32_t make_idesc_mxf8(uint32_t m, uint32_t n) {
  return ((n >> 3) << 17) | (1u << 23) | ((m >> 4) << 24);
}

// ------------------------------------------------------------ cluster / DSMEM
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive_release() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait_acquire() {
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_smem(uint32_t local_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void st_dsmem_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ void st_dsmem_u64(uint32_t cluster_addr, unsigned long long v) {
  asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(cluster_addr), "l"(v) : "memory");
}
__device__ __forceinline__ uint2 ld_dsmem_v2u32(uint32_t cluster_addr) {
  uint2 v;
  asm volatile("ld.shared::cluster.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(cluster_addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_dsmem_f32(uint32_t cluster_addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_dsmem_v4(uint32_t cluster_addr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(cluster_addr), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// ------------------------------------------- system-scope flags (NVLink handoff)
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_release_sys_add(uint32_t* p, uint32_t v) {
  asm volatile("red.release.sys.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Mesh abort word (device memory, one per process / GPU; set through set_wait_policy() of every translation unit that
// waits on handoff flags).  A wait that exceeds the time bound does NOT trap the GPU (round 1: a late or dead peer took
// all 8 contexts down): it raises the abort word and returns; every later wait of this process returns at once, so the
// pipeline drains with garbage in microseconds, the token read-back kernel reports the word to the host and the engine
// fails the in-flight requests with a clean error while the process (and its control plane) stays alive.
static __device__ uint32_t* g_abort_word = nullptr;
static __device__ unsigned long long g_wait_limit_ns = 0;

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Slow path of a flag wait: out of line on purpose -- the decode GEMMs are sensitive to their code size (a bisect in
// round 2 attributed 1-2 % of the step to a few hundred extra SASS instructions per kernel), and this is inlined nowhere.
static __device__ __noinline__ void wait_flag_slow(const uint32_t* flag, uint32_t target) {
  volatile uint32_t* ab = g_abort_word;
  if (ab != nullptr && *ab != 0u) return;                                        // mesh aborted: drain
  uint32_t spins = 0;
  unsigned long long t0 = 0;
  while (static_cast<int32_t>(ld_acquire_sys(flag) - target) < 0) {
    __nanosleep(20);
    ++spins;
    if (ab != nullptr) {
      if ((spins & 127u) == 0u) {
        if (*ab != 0u) return;                                                   // another waiter gave up
        const unsigned long long now = globaltimer_ns();
        if (t0 == 0) t0 = now;
        else if (now - t0 > g_wait_limit_ns) {
          *ab = 1u;
          __threadfence_system();
          return;
        }
      }
    } else if (spins > B2B_SPIN_LIMIT) {
      __trap();
    }
  }
}

// Spin until *flag >= target (monotonic counters; wrap-safe compare); bounded, see above.
__device__ __forceinline__ void wait_flag_ge(const uint32_t* flag, uint32_t target) {
  if (static_cast<int32_t>(ld_acquire_sys(flag) - target) >= 0) return;          // fast path: already published
  wait_flag_slow(flag, target);
}

// Programmatic dependent launch: wait for (and see the memory of) all prerequisite grids /
// allow the dependent grid to start launching.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ float bf16_round(float x) {
  return __bfloat162float(__float2bfloat16_rn(x));
}

}  // namespace b2b
