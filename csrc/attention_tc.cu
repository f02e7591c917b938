// Prefill (and chunked-prefill) attention on the 5th-gen tensor cores: flash-attention forward over
// the paged KV cache with tcgen05.mma, accumulators in TMEM, operands staged by TMA.
//
// One CTA = (sequence, kv head, block of QB = 128/G queries).  The G query heads that share the kv
// head are stacked into the 128 MMA rows (row = g*QB + i), so every K/V page is fetched once per
// group.  Per KV tile of BKV keys:
//     S = Q K^T      tcgen05.mma  (A = Q tile, B = K tile, both K-major 128B-swizzled)  -> TMEM, double buffered
//     P = softmax    4 warps, one TMEM lane (= row) per thread, online max with lazy rescaling
//     O += P V       tcgen05.mma  (A = P written back to TMEM as bf16 over the S columns it came from, B = V tile
//                                  read MN-major: the cache keeps V as [token, d], i.e. N-contiguous)
// Warp roles: 0 = TMA producer, 1 = TMEM owner + MMA issuer, 2..5 = softmax / correction / epilogue.
// q is pre-scaled by 1/sqrt(d) and rotated by the QKV GEMM epilogue; K is rotated when appended.
//
// Layouts: q/out [tokens, n_q, D]; K/V cache [pages, 64, n_kv, D]; block_table [seqs, max_pages].
// Reference parity: torch SDPA under `transformers.generate` (bee2bee/hf.py:42-43).
#include "kernels.h"

#include <cuda.h>
#include <cuda_fp8.h>

#include <type_traits>

#include "common.cuh"
#include "launch.cuh"

namespace b2b {

int make_tmap_shared(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     int elt_bytes);

namespace {

constexpr int APAGE = 64;
constexpr int ATC_THREADS = 192;
constexpr float LOG2E = 1.4426950408889634f;

struct AttnTcParams {
  __nv_bfloat16* out;
  const int* block_table;
  const int* q_start;
  const int* q_len;
  const int* kv_len;
  int max_pages, n_q, n_kv, window;
  float softcap;
  // split-KV decode (q_len == 1): grid.x = splits, CTA `split` covers a contiguous range of the 64-key tiles and writes
  // its unnormalised partial (O, running max, row sum) to the workspace the CUDA-core kernel's merge pass reads:
  // ws[((seq * n_kv + kvh) * splits + split) * ws_rows + head_in_group][D + 2]
  int splits, ws_rows;
  float* ws;
  // fused MX quantisation of the output for the O-proj GEMM (mxfp8 pieces): every thread owns whole 32-feature blocks of
  // its (token, head) row, so the block maximum is a register reduction: e4m3 bytes + UE8M0 scale in the consumer's
  // tcgen05.cp chunk layout (token tile q_bn).  Not available in split-KV mode (the merge pass writes the output).
  uint8_t* q_out8;
  uint8_t* q_sf;
  int q_bn;
};

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
      "%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,"
      "%31,%32};"
      ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
        "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
        "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
        "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
        "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])), "r"(__float_as_uint(v[16])),
        "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])),
        "r"(__float_as_uint(v[23])), "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])),
        "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])), "r"(__float_as_uint(v[28])),
        "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// D[tmem] (+)= A[tmem] * B[smem] -- the A operand (P) is read from tensor memory: lane = row, 16-bit elements packed
// two per 32-bit column (element 2j in the low half).
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st32_bits(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,"
      "%31,%32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
        "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
        "r"(v[30]), "r"(v[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// MN-major 128B-swizzled operand (rows = K index, 128-byte rows of 64 contiguous N elements):
// LBO = distance between 64-element N blocks, SBO = distance between 8-row K groups (1024 B).
__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// issue-only TMEM load of 32 columns (this thread's lane); pair with tmem_ld_fence() before reading r[]
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
      "%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// wait for all outstanding TMEM loads; the "+r" operands keep every use of r[] after the wait
__device__ __forceinline__ void tmem_ld_fence(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]),
                 "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]),
                 "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

template <int D>
struct AtcCfg {
  static constexpr int BKV = 64;                                  // keys per tile == one KV page
  static constexpr int kQBytes = 128 * D * 2;
  static constexpr int kKVBytes = BKV * D * 2;
  static constexpr int kPBytes = 128 * BKV * 2;   // P lives in TMEM; the bytes stay: the footprint sets the CTAs per SM
  static constexpr int kSmemBytes = kQBytes + 4 * kKVBytes + kPBytes + 256;
  static constexpr int kTmemCols = (2 * BKV + D <= 256) ? 256 : 512;   // S double buffer + O
  static constexpr int kMinCtas = (D <= 128) ? 2 : 1;                  // two CTAs per SM: one's softmax hides the other's MMAs
};

// P stays in tensor memory (written over the first BKV/2 columns of the S buffer it was computed from) and feeds the PV
// MMA as a TMEM A operand.
template <int D, bool SOFTCAP>
__global__ void __launch_bounds__(ATC_THREADS, AtcCfg<D>::kMinCtas)
attn_prefill_tc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                       const __grid_constant__ CUtensorMap tm_v, const AttnTcParams p, const int G, const int QB) {
  using Cfg = AtcCfg<D>;
  constexpr int BKV = Cfg::BKV;
  constexpr int DB = D / 64;            // 64-column (128 B) blocks of the head dim
  constexpr uint32_t S_COL = 0, O_COL = 2 * BKV;
  constexpr uint32_t TCOLS = Cfg::kTmemCols;

  // ---- set-up that reads nothing an earlier kernel wrote (barriers, tensor memory, descriptor prefetch): under PDL the CTA
  // is resident while the QKV GEMM still drains, so all of this is off the critical path; only then wait for the producer
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();             // the swizzled tiles need 1024-byte alignment
  uint8_t* q_s = smem;
  uint8_t* k_s = q_s + Cfg::kQBytes;                       // [2][kKVBytes]
  uint8_t* v_s = k_s + 2 * Cfg::kKVBytes;                  // [2][kKVBytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(v_s + 2 * Cfg::kKVBytes + Cfg::kPBytes);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;     // [2]
  uint64_t* v_full = bars + 3;     // [2]
  uint64_t* k_empty = bars + 5;    // [2]
  uint64_t* v_empty = bars + 7;    // [2]
  uint64_t* s_full = bars + 9;     // [2]
  uint64_t* p_ready = bars + 11;
  uint64_t* pv_done = bars + 12;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1); mbar_init(&v_full[i], 1); mbar_init(&k_empty[i], 1); mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
    }
    mbar_init(p_ready, 4);
    mbar_init(pv_done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tm_q); tma_prefetch_desc(&tm_k); tma_prefetch_desc(&tm_v);
  }
  if (warp == 1) tmem_alloc<TCOLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // dependents (the O-proj GEMM) may become resident from here on: every CTA of this grid already owns its tensor memory,
  // so an early O-proj CTA that takes TMEM columns and then waits for this grid can never starve one of its CTAs
  pdl_launch_dependents();
  pdl_wait();                                               // q / K / V and the metadata below come from earlier kernels
  const int seq = blockIdx.z, kvh = blockIdx.y;
  const bool split_mode = p.splits > 1;
  const int qblk = split_mode ? 0 : gridDim.x - 1 - blockIdx.x;   // longest (latest) query blocks first
  const int qlen = p.q_len[seq], kvlen = p.kv_len[seq];
  const int q0 = qblk * QB;
  bool active = q0 < qlen;                                  // CTA-uniform; an idle CTA only runs the tear-down below
  const int nq_here = min(QB, qlen - q0);
  const int qtok0 = p.q_start[seq] + q0;
  const int pos0 = kvlen - qlen + q0;                       // absolute position of query 0 of this block
  const int kv_hi = min(kvlen, pos0 + nq_here);
  const int kv_lo = p.window > 0 ? max(0, pos0 - p.window + 1) : 0;
  int t_lo = kv_lo / BKV, t_hi = (kv_hi + BKV - 1) / BKV;
  if (active && split_mode) {
    // this CTA's share of the key tiles (may be empty: it then publishes an empty partial, m = -inf, l = 0)
    const int per = (t_hi - t_lo + p.splits - 1) / p.splits;
    t_lo = min(t_hi, t_lo + static_cast<int>(blockIdx.x) * per);
    t_hi = min(t_hi, t_lo + per);
    if (t_hi <= t_lo) {
      // empty share (short sequence, many splits): publish an empty partial; no TMA / MMA is ever issued by this CTA
      if (threadIdx.x < G) {
        float* w = p.ws + (((static_cast<size_t>(seq) * p.n_kv + kvh) * p.splits + blockIdx.x) * p.ws_rows + threadIdx.x) * (D + 2);
        for (int c = 0; c < D; ++c) w[c] = 0.f;
        w[D] = -INFINITY;
        w[D + 1] = 0.f;
      }
      active = false;
    }
  }
  const int nt = t_hi - t_lo;

  if (!active) {
    // nothing to compute (inactive row / empty split share)
  } else if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, Cfg::kQBytes);
      for (int g = 0; g < G; ++g)
        for (int c = 0; c < DB; ++c)
          tma_load_2d(q_s + c * (128 * 128) + g * QB * 128, &tm_q, q_full, (kvh * G + g) * D + c * 64, qtok0);
      const int* bt = p.block_table + static_cast<size_t>(seq) * p.max_pages;
      for (int n = 0; n < nt; ++n) {
        const int s = n & 1;
        const uint32_t ph = static_cast<uint32_t>((n >> 1) & 1);
        const int page = bt[t_lo + n];
        mbar_wait(&k_empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&k_full[s], Cfg::kKVBytes);
#pragma unroll
        for (int c = 0; c < DB; ++c)
          tma_load_2d(k_s + s * Cfg::kKVBytes + c * (BKV * 128), &tm_k, &k_full[s], kvh * D + c * 64, page * APAGE);
        mbar_wait(&v_empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&v_full[s], Cfg::kKVBytes);
#pragma unroll
        for (int c = 0; c < DB; ++c)
          tma_load_2d(v_s + s * Cfg::kKVBytes + c * (BKV * 128), &tm_v, &v_full[s], kvh * D + c * 64, page * APAGE);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc_s = make_idesc_bf16(128, BKV);
    constexpr uint32_t idesc_o = make_idesc_bf16(128, D) | (1u << 16);        // B operand (V) is MN-major
    auto issue_qk = [&](int n) {
      const int s = n & 1;
      mbar_wait(&k_full[s], static_cast<uint32_t>((n >> 1) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d_tmem = tmem + S_COL + static_cast<uint32_t>(s) * BKV;
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk) {
          const uint64_t a = make_sw128_kmajor_desc(smem_u32(q_s + (kk / 4) * (128 * 128))) + static_cast<uint64_t>((kk % 4) * 2);
          const uint64_t b = make_sw128_kmajor_desc(smem_u32(k_s + s * Cfg::kKVBytes + (kk / 4) * (BKV * 128))) +
                             static_cast<uint64_t>((kk % 4) * 2);
          umma_bf16(d_tmem, a, b, idesc_s, kk > 0 ? 1u : 0u);
        }
        umma_commit(&k_empty[s]);
        umma_commit(&s_full[s]);
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0);
    if (nt > 0) issue_qk(0);
    for (int n = 0; n < nt; ++n) {
      if (n + 1 < nt) issue_qk(n + 1);                    // S(n+1) runs on the tensor pipe while softmax(n) runs
      const int s = n & 1;
      mbar_wait(&v_full[s], static_cast<uint32_t>((n >> 1) & 1));
      mbar_wait(p_ready, static_cast<uint32_t>(n & 1));
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < BKV / 16; ++kk) {
          const uint64_t b = make_sw128_mnmajor_desc(smem_u32(v_s + s * Cfg::kKVBytes + kk * (16 * 128)), BKV * 128);
          // 16 keys of P = 8 packed columns of the S buffer this tile came from
          umma_bf16_ts(tmem + O_COL, tmem + S_COL + static_cast<uint32_t>(s) * BKV + kk * 8, b, idesc_o, (n > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(&v_empty[s]);
        umma_commit(pv_done);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ softmax / correction / epilogue
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int g = row / QB, i = row % QB;
    const bool row_valid = (g < G) && (i < nq_here);
    const int qpos = pos0 + i;
    const uint32_t lane_addr = tmem + (static_cast<uint32_t>(quarter * 32) << 16);
    const float cap = p.softcap;
    const float inv_cap = SOFTCAP ? 1.f / cap : 0.f;
    float m_ref = -INFINITY, l = 0.f;

    auto tile = [&](int n, auto masked) {
      const int t = t_lo + n, b = n & 1;
      mbar_wait(&s_full[b], static_cast<uint32_t>((n >> 1) & 1));
      tc_fence_after();
      const uint32_t s_addr = lane_addr + S_COL + static_cast<uint32_t>(b) * BKV;
      // the whole score row of this tile lives in registers: one TMEM read, one wait
      uint32_t r[BKV];
      tmem_ld32_issue(s_addr, r);
      tmem_ld32_issue(s_addr + 32, r + 32);
      tmem_ld_fence(r);
      tmem_ld_fence(r + 32);
      float mrow = -INFINITY;
#pragma unroll
      for (int e = 0; e < BKV; ++e) {
        float sc = __uint_as_float(r[e]);
        if constexpr (SOFTCAP) sc = cap * tanhf(sc * inv_cap);
        sc *= LOG2E;
        if constexpr (decltype(masked)::value) {
          const int kvpos = t * BKV + e;
          const bool ok = row_valid && kvpos <= qpos && kvpos < kvlen && (p.window <= 0 || kvpos > qpos - p.window);
          sc = ok ? sc : -INFINITY;
        }
        r[e] = __float_as_uint(sc);
        mrow = fmaxf(mrow, sc);
      }
      // lazy rescaling: keep the reference max while the new maximum is within 2^8 of it
      float alpha = 1.f;
      if (mrow > m_ref + 8.f || (m_ref == -INFINITY && mrow > -INFINITY)) {
        alpha = (m_ref == -INFINITY) ? 0.f : exp2f(m_ref - mrow);
        m_ref = mrow;
      }
      if (n > 0) {
        mbar_wait(pv_done, static_cast<uint32_t>((n - 1) & 1));        // O is free again
        tc_fence_after();
        if (__any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll 1
          for (int c = 0; c < D; c += 32) {
            float o[32];
            tmem_ld32(lane_addr + O_COL + c, o);
#pragma unroll
            for (int e = 0; e < 32; ++e) o[e] *= alpha;
            tmem_st32(lane_addr + O_COL + c, o);
          }
        }
      }
      // P = exp2(s - m_ref) -> bf16 pairs -> TMEM (A operand of the PV MMA)
      const float mr = (m_ref == -INFINITY) ? 0.f : m_ref;          // fully masked so far: exp2(-inf - 0) = 0
      float lsum = 0.f;
      uint32_t pk[BKV / 2];              // bf16 pairs: key 2j in the low half of column j
#pragma unroll
      for (int j = 0; j < BKV / 2; ++j) {
        const float p0 = exp2f(__uint_as_float(r[2 * j]) - mr);
        const float p1 = exp2f(__uint_as_float(r[2 * j + 1]) - mr);
        lsum += p0 + p1;
        const __nv_bfloat162 h = __floats2bfloat162_rn(p0, p1);
        pk[j] = *reinterpret_cast<const uint32_t*>(&h);
      }
      static_assert(BKV == 64, "one 64-key tile of P packs into 32 TMEM columns");
      tmem_st32_bits(s_addr, pk);        // over the (already consumed) scores of this tile
      l = l * alpha + lsum;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_ready);
    };

    for (int n = 0; n < nt; ++n) {
      const int t = t_lo + n;
      // a tile needs no predicate when every key of it is visible to every (valid) query row of the block
      const bool full = nq_here == QB && (t + 1) * BKV - 1 <= pos0 && (t + 1) * BKV <= kvlen &&
                        (p.window <= 0 || t * BKV > pos0 + nq_here - 1 - p.window);
      if (full) tile(n, std::false_type{}); else tile(n, std::true_type{});
    }

    // epilogue: O / l -> out[token, head, :]
    if (nt > 0) {
      mbar_wait(pv_done, static_cast<uint32_t>((nt - 1) & 1));
      tc_fence_after();
    }
    const float inv = l > 0.f ? 1.f / l : 0.f;
    __nv_bfloat16* dst = p.out + (static_cast<size_t>(qtok0 + i) * p.n_q + kvh * G + g) * D;
    float* wsrow = split_mode ? p.ws + (((static_cast<size_t>(seq) * p.n_kv + kvh) * p.splits + blockIdx.x) * p.ws_rows + g) *
                                           (D + 2) : nullptr;
    if (split_mode && row_valid) {
      wsrow[D] = (m_ref == -INFINITY) ? -INFINITY : m_ref * 0.6931471805599453f;     // natural-log domain for the merge pass
      wsrow[D + 1] = l;
    }
#pragma unroll 1
    for (int c = 0; c < D; c += 32) {
      float o[32];
      if (nt > 0) {
        tmem_ld32(lane_addr + O_COL + c, o);
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) o[e] = 0.f;
      }
      if (split_mode) {
        if (row_valid) {
#pragma unroll
          for (int e = 0; e < 32; e += 2)      // rows are (D + 2) floats apart: 8-byte, not 16-byte, aligned
            *reinterpret_cast<float2*>(wsrow + c + e) = make_float2(o[e], o[e + 1]);
        }
        continue;
      }
      if (row_valid && p.q_out8 != nullptr) {
        // e4m3 + block scale of these 32 features (what a separate quantiser would compute from the bf16 output)
        float amax = 0.f;
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          o[e] = __bfloat162float(__float2bfloat16_rn(o[e] * inv));
          amax = fmaxf(amax, fabsf(o[e]));
        }
        const uint32_t u = __float_as_uint(amax * (1.f / 448.f));
        int ex = static_cast<int>(u >> 23) - 127 + ((u & 0x7FFFFFu) ? 1 : 0);
        ex = max(-126, min(127, ex));
        const float sc = __uint_as_float(static_cast<uint32_t>(127 - ex) << 23);
        const int tok = qtok0 + i, feat = (kvh * G + g) * D + c, ldq = p.n_q * D;
        uint32_t w8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint32_t b = 0;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            b |= static_cast<uint32_t>(__nv_cvt_float_to_fp8(o[4 * j + e] * sc, __NV_SATFINITE, __NV_E4M3)) << (8 * e);
          w8[j] = b;
        }
        uint4* q4 = reinterpret_cast<uint4*>(p.q_out8 + static_cast<size_t>(tok) * ldq + feat);
        q4[0] = make_uint4(w8[0], w8[1], w8[2], w8[3]);
        q4[1] = make_uint4(w8[4], w8[5], w8[6], w8[7]);
        const int tile = tok / p.q_bn, n = tok - tile * p.q_bn, rr = n & 127;
        p.q_sf[(static_cast<size_t>(tile) * (ldq >> 7) + (feat >> 7)) * (p.q_bn > 128 ? 1024 : 512) + (n >> 7) * 512 +
               (rr & 31) * 16 + (rr >> 5) * 4 + ((feat >> 5) & 3)] = static_cast<uint8_t>(ex + 127);
      } else if (row_valid) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t w[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const __nv_bfloat162 h = __floats2bfloat162_rn(o[8 * j + 2 * e] * inv, o[8 * j + 2 * e + 1] * inv);
            w[e] = *reinterpret_cast<const uint32_t*>(&h);
          }
          *reinterpret_cast<uint4*>(dst + c + 8 * j) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TCOLS>(tmem);
  }
}

template <int D, bool SOFTCAP>
int launch_tc_cap(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcParams& p, int G, int QB,
                  int seqs, int qblocks, cudaStream_t s) {
  using Cfg = AtcCfg<D>;
  static bool set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 64 && !set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(attn_prefill_tc_kernel<D, SOFTCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes);
    if (e != cudaSuccess) return static_cast<int>(e);
    set[dev] = true;
  }
  return static_cast<int>(launch_kernel(attn_prefill_tc_kernel<D, SOFTCAP>,
                                        dim3(p.splits > 1 ? p.splits : qblocks, p.n_kv, seqs), dim3(ATC_THREADS),
                                        Cfg::kSmemBytes, s, 1, tq, tk, tv, p, G, QB));
}

template <int D>
int launch_tc(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcParams& p, int G, int QB,
              int seqs, int qblocks, cudaStream_t s) {
  return p.softcap > 0.f ? launch_tc_cap<D, true>(tq, tk, tv, p, G, QB, seqs, qblocks, s)
                         : launch_tc_cap<D, false>(tq, tk, tv, p, G, QB, seqs, qblocks, s);
}

}  // namespace

bool attention_tc_supported(int n_q, int n_kv, int head_dim) {
  if (n_kv <= 0 || n_q % n_kv) return false;
  const int G = n_q / n_kv;
  if (G != 1 && G != 2 && G != 4 && G != 8 && G != 16) return false;
  return head_dim == 64 || head_dim == 128 || head_dim == 256;
}

// Prefill path: every sequence contributes q_len >= 1 new tokens, kv_len includes them.
int launch_attention_tc(const void* q, const void* k_cache, const void* v_cache, void* out, const int* block_table,
                        const int* q_start, const int* q_len, const int* kv_len, int seqs, int max_q, int max_pages,
                        int n_tokens, int n_pages, int n_q, int n_kv, int head_dim, int window, float softcap,
                        int splits, float* ws, void* q_out8, void* q_sf, int q_bn, cudaStream_t s) {
  if (!attention_tc_supported(n_q, n_kv, head_dim)) return -2;
  const int G = n_q / n_kv, QB = 128 / G;
  CUtensorMap tq, tk, tv;
  int r = make_tmap_shared(&tq, q, static_cast<uint64_t>(n_tokens), static_cast<uint64_t>(n_q) * head_dim,
                           static_cast<uint64_t>(n_q) * head_dim, static_cast<uint32_t>(QB), 2);
  if (r) return r;
  const uint64_t kv_rows = static_cast<uint64_t>(n_pages) * APAGE, kv_cols = static_cast<uint64_t>(n_kv) * head_dim;
  if ((r = make_tmap_shared(&tk, k_cache, kv_rows, kv_cols, kv_cols, APAGE, 2))) return r;
  if ((r = make_tmap_shared(&tv, v_cache, kv_rows, kv_cols, kv_cols, APAGE, 2))) return r;
  AttnTcParams p;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.block_table = block_table; p.q_start = q_start; p.q_len = q_len; p.kv_len = kv_len;
  p.max_pages = max_pages; p.n_q = n_q; p.n_kv = n_kv; p.window = window; p.softcap = softcap;
  p.splits = (max_q == 1 && splits > 1 && ws != nullptr) ? splits : 1;
  p.ws = ws;
  p.ws_rows = attn_rows(G, 1);
  p.q_out8 = p.splits > 1 ? nullptr : static_cast<uint8_t*>(q_out8);
  p.q_sf = static_cast<uint8_t*>(q_sf);
  p.q_bn = q_bn > 0 ? q_bn : 32;
  if (q_out8 != nullptr && p.splits > 1) return -8;       // the merge pass writes bf16: use the stand-alone quantiser
  const int qblocks = (max_q + QB - 1) / QB;
  int rc;
  switch (head_dim) {
    case 64: rc = launch_tc<64>(tq, tk, tv, p, G, QB, seqs, qblocks, s); break;
    case 128: rc = launch_tc<128>(tq, tk, tv, p, G, QB, seqs, qblocks, s); break;
    case 256: rc = launch_tc<256>(tq, tk, tv, p, G, QB, seqs, qblocks, s); break;
    default: return -3;
  }
  if (rc == 0 && p.splits > 1)
    rc = launch_attention_merge(out, q_start, ws, seqs, n_q, n_kv, head_dim, p.splits, s);
  return rc;
}

}  // namespace b2b
