// tcgen05 / TMEM / TMA "swap-AB" GEMM for sm_100a.
//
//   out[t, n] = epilogue( sum_k X[t, k] * W[n, k] )
//
// The WEIGHT matrix is the 128-row MMA "A" operand (UMMA_M = 128 output features
// per CTA, one TMEM lane per feature) and the TOKENS are the MMA "N" dimension
// (BN = 16..256 TMEM columns).  Decode batches of 1..32 tokens therefore cost
// 16..32 tensor-core columns instead of a padded 128-row tile, the kernel streams
// W exactly once through a TMA -> smem ring, and the whole op sits on the HBM
// roofline.  Small problems get their parallelism from split-K across a
// thread-block cluster whose partial accumulators are reduced through DSMEM.
//
// Roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2..5 = epilogue (TMEM -> registers -> fused epilogue -> global / peer).
//
// Fused epilogues: residual add, SwiGLU/GeGLU, bias+GELU, RMSNorm scale of the
// *input* (gamma folded into W; per-token 1/rms computed by the idle epilogue
// warps during the main loop), RoPE + paged-KV append for the QKV projection,
// and the NVLink piece handoff: the tail GEMM of piece i stores its tiles straight
// into piece i+1's input buffer on the peer GPU and publishes a release flag; the
// head GEMM of piece i+1 prefetches its weight tiles, acquires the flag, then
// TMA-loads the freshly written activations.
//
// Reference parity: replaces the JSON/WebSocket hidden-state hop of
// bee2bee/node.py:249-277 and the cuBLAS calls under bee2bee/hf.py:42-43.
#include "gemm_tc.cuh"

#include <cuda_fp8.h>

#include <cstdio>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "launch.cuh"

namespace b2b {

constexpr int BM = 128;   // weight rows per CTA == UMMA_M
constexpr int BK = 64;    // bf16 elements per 128B swizzle row (fp8: 128 elements, same 128 bytes)
constexpr int ROW_BYTES = 128;
constexpr int A_STAGE_BYTES = BM * ROW_BYTES;

template <int BN>
struct GemmCfg {
  static constexpr int kStages = (BN <= 32) ? 5 : (BN == 64 ? 4 : (BN == 128 ? 6 : 4));
  static constexpr int kStageBytes = A_STAGE_BYTES + BN * ROW_BYTES;
  static constexpr int kTmemCols = BN < 32 ? 32 : BN;
  // MX (block-scaled fp8): the UE8M0 scale factors of a stage (one 512-byte chunk per 128 rows x 128 K)
  // are staged in smem next to the ring and copied to TMEM columns behind the accumulator.
  static constexpr int kSfaBytes = 512;
  static constexpr int kSfbBytes = BN > 128 ? 1024 : 512;
  static constexpr int kSfBytes = kSfaBytes + kSfbBytes;
  static constexpr int kSfCol = kTmemCols;                      // first scale-factor column (2 x 16 columns)
  static constexpr int kTmemColsMx = BN <= 32 ? 64 : (BN == 64 ? 128 : (BN == 128 ? 256 : 512));
  static constexpr int smem_bytes(int stages) { return stages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + BN * 12 + stages * kSfBytes; }
  static constexpr int kSmemBytes = smem_bytes(kStages);
};

__device__ __forceinline__ float gelu_tanh(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  return 0.5f * x * (1.f + tanhf(u));
}
__device__ __forceinline__ float silu(float x) { return x / (1.f + __expf(-x)); }

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define B2B_DBG(slot)                                                                                          \
  do {                                                                                                         \
    if (p.dbg != nullptr)                                                                                      \
      p.dbg[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 + (slot)] = gtime();          \
  } while (0)

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// QM: 0 = bf16, 1 = fp8 e4m3 with per-row / per-token fp32 scales, 2 = MX fp8 (e4m3 + UE8M0 scale per 32 K)
template <int BN, int EPI, int QM>
__global__ void __launch_bounds__(192) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_w,
                                                      const __grid_constant__ CUtensorMap tmap_x,
                                                      const GemmParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr bool FP8 = QM != 0;
  constexpr bool MX = QM == 2;
  const int STAGES = p.stages;            // ring depth (runtime: 2..Cfg::kStages; fewer stages = more CTAs per SM)
  constexpr int STAGE_BYTES = Cfg::kStageBytes;
  constexpr uint32_t TX_BYTES = STAGE_BYTES + (MX ? Cfg::kSfBytes : 0);
  constexpr uint32_t TCOLS = MX ? Cfg::kTmemColsMx : Cfg::kTmemCols;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* rstd_s = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + 256);
  int* pos_s = reinterpret_cast<int*>(rstd_s + BN);               // [BN] token positions (QKV/RoPE epilogue)
  int* slot_s = pos_s + BN;                                       // [BN] KV-cache slots
  uint8_t* sf_s = smem + STAGES * STAGE_BYTES + 256 + BN * 12;    // [STAGES][kSfBytes]: SFA chunk, SFB chunk(s)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) B2B_DBG(0);
  const int tile_n = blockIdx.x;             // 128-row block of W
  const int tok0 = blockIdx.y * BN;          // first token of this CTA
  const int splitk = p.splitk;
  const int krank = (splitk > 1) ? static_cast<int>(cluster_ctarank()) : 0;
  // split-K reduce-scatter: this CTA finishes token columns [col0, col0 + ncol) of the tile (launcher: splitk | BN)
  const int ncol = BN / splitk;
  const int col0 = krank * ncol;

  constexpr int BKE = FP8 ? 128 : 64;       // K elements per 128-byte k-block
  const int nkb_total = p.k / BKE;
  const int kb_begin = static_cast<int>((static_cast<long long>(nkb_total) * krank) / splitk);
  const int kb_end = static_cast<int>((static_cast<long long>(nkb_total) * (krank + 1)) / splitk);
  const int nkb = kb_end - kb_begin;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_w);
    tma_prefetch_desc(&tmap_x);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&empty_bar[s], 1);
      }
      mbar_init(tmem_full_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc<TCOLS>(tmem_ptr_s);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  pdl_launch_dependents();     // the next kernel may start its own set-up / weight prefetch now
  if (threadIdx.x == 0) B2B_DBG(1);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      const uint64_t pol_w = l2_policy_evict_first();   // weights: streamed once
      const uint64_t pol_x = l2_policy_evict_last();    // activations: re-read by every CTA
      // Weight tiles depend on no earlier kernel: fill the ring with them first, THEN wait for
      // the producer of the activations (previous kernel via PDL, upstream piece via its flag).
      const int npre = nkb < STAGES ? nkb : STAGES;
      const uint8_t* sfa_g = MX ? p.sfa + (static_cast<size_t>(tile_n) * nkb_total + kb_begin) * Cfg::kSfaBytes : nullptr;
      const uint8_t* sfb_g = MX ? p.sfb + (static_cast<size_t>(blockIdx.y) * nkb_total + kb_begin) * Cfg::kSfbBytes : nullptr;
      for (int i = 0; i < npre; ++i) {
        mbar_arrive_expect_tx(&full_bar[i], TX_BYTES);
        tma_load_2d_hint(smem + i * STAGE_BYTES, &tmap_w, &full_bar[i], (kb_begin + i) * BKE, tile_n * BM, pol_w);
        if constexpr (MX) bulk_load(sf_s + i * Cfg::kSfBytes, sfa_g + static_cast<size_t>(i) * Cfg::kSfaBytes, Cfg::kSfaBytes, &full_bar[i]);
      }
      pdl_wait();
      if (p.wait_flag != nullptr) {
        const uint32_t target = *reinterpret_cast<const volatile uint32_t*>(p.wait_epoch) + 1;
        wait_flag_ge(p.wait_flag, target);
        fence_proxy_async_all();   // peer-written (generic proxy) data -> TMA (async proxy) reads
      }
      for (int i = 0; i < npre; ++i) {
        tma_load_2d_hint(smem + i * STAGE_BYTES + A_STAGE_BYTES, &tmap_x, &full_bar[i], (kb_begin + i) * BKE, tok0,
                         pol_x);
        if constexpr (MX)
          bulk_load(sf_s + i * Cfg::kSfBytes + Cfg::kSfaBytes, sfb_g + static_cast<size_t>(i) * Cfg::kSfbBytes, Cfg::kSfbBytes, &full_bar[i]);
      }
      int kb = npre;
      B2B_DBG(2);
      int s = 0;                 // kb % STAGES
      uint32_t ph = 1;           // (kb / STAGES) & 1 -- first refill round
      for (; kb < nkb; ++kb) {
        mbar_wait(&empty_bar[s], ph ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], TX_BYTES);
        tma_load_2d_hint(smem + s * STAGE_BYTES, &tmap_w, &full_bar[s], (kb_begin + kb) * BKE,
                         tile_n * BM, pol_w);
        tma_load_2d_hint(smem + s * STAGE_BYTES + A_STAGE_BYTES, &tmap_x, &full_bar[s],
                         (kb_begin + kb) * BKE, tok0, pol_x);
        if constexpr (MX) {
          bulk_load(sf_s + s * Cfg::kSfBytes, sfa_g + static_cast<size_t>(kb) * Cfg::kSfaBytes, Cfg::kSfaBytes, &full_bar[s]);
          bulk_load(sf_s + s * Cfg::kSfBytes + Cfg::kSfaBytes, sfb_g + static_cast<size_t>(kb) * Cfg::kSfbBytes, Cfg::kSfbBytes, &full_bar[s]);
        }
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer
    constexpr uint32_t idesc = MX ? make_idesc_mxf8(BM, BN) : (FP8 ? make_idesc_e4m3(BM, BN) : make_idesc_bf16(BM, BN));
    int s = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < nkb; ++kb) {
      mbar_wait(&full_bar[s], ph);
      tc_fence_after();
      if (lane == 0) {
        if (kb == 0) B2B_DBG(3);
        const uint64_t adesc = make_sw128_kmajor_desc(smem_u32(smem + s * STAGE_BYTES));
        const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(smem + s * STAGE_BYTES + A_STAGE_BYTES));
        uint32_t sfa_t = 0, sfb_t = 0;
        if constexpr (MX) {
          // scale factors of this stage: smem -> TMEM (tcgen05.cp executes in issue order with the MMAs below);
          // two column sets alternate so that the copy for stage kb+1 never races the MMAs of stage kb
          sfa_t = tmem_base + Cfg::kSfCol + static_cast<uint32_t>(kb & 1) * 16;
          sfb_t = sfa_t + 4;
          const uint32_t sf_addr = smem_u32(sf_s + s * Cfg::kSfBytes);
          tmem_cp_32x128b_warpx4(sfa_t, make_sf_desc(sf_addr));
          tmem_cp_32x128b_warpx4(sfb_t, make_sf_desc(sf_addr + Cfg::kSfaBytes));
          if constexpr (BN > 128) tmem_cp_32x128b_warpx4(sfb_t + 4, make_sf_desc(sf_addr + Cfg::kSfaBytes + 512));
        }
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // advance 16 bf16 = 32 B along K inside the swizzle atom: +2 in the (addr>>4) field
          // one MMA consumes 32 bytes of K per row (16 bf16 / 32 e4m3): +2 in the (addr >> 4) field
          if constexpr (MX)
            umma_mxf8(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc | (static_cast<uint32_t>(k) << 4) | (static_cast<uint32_t>(k) << 29),
                      (kb > 0 || k > 0) ? 1u : 0u, sfa_t, sfb_t);
          else if constexpr (FP8) umma_f8(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          else umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty_bar[s]);                    // frees the smem slot when the MMAs retire
        if (kb == nkb - 1) { umma_commit(tmem_full_bar); B2B_DBG(4); }   // accumulator complete
      }
      __syncwarp();
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
  } else {
    // ---------------------------------------- epilogue warps: prologue work
    // Every CTA of a split-K cluster finishes its own slice of token columns [col0, col0 + ncol)
    // (reduce-scatter, see below), so each CTA only needs the per-token inputs of that slice.
    const int et = threadIdx.x - 64;   // 0..127
    pdl_wait();                        // everything below reads / writes memory of earlier kernels
    {
      if constexpr (EPI == EPI_QKV_ROPE) {
        // per-token metadata -> smem once: global loads inside the store loop of the epilogue serialise on L2
        // latency (the compiler cannot hoist them above stores that may alias): +8 us at 32 tokens
        for (int t = col0 + et; t < col0 + ncol; t += 128) {
          const int tok = tok0 + t;
          pos_s[t] = (p.positions != nullptr && tok < p.m_tok) ? p.positions[tok] : 0;
          slot_s[t] = (tok < p.m_tok) ? p.slots[tok] : -1;
        }
      }
      if (p.norm_src != nullptr) {
        if (p.wait_flag != nullptr) {
          const uint32_t target = *reinterpret_cast<const volatile uint32_t*>(p.wait_epoch) + 1;
          wait_flag_ge(p.wait_flag, target);
        }
        // one warp per token, FOUR tokens x FOUR row segments in flight per lane (the loop is L2-latency
        // bound: 16 independent 128-bit loads are issued before the first use)
        const int kv8 = p.k / 8;
        for (int tr = warp - 2; tr < ncol; tr += 16) {
          float ss[4] = {0.f, 0.f, 0.f, 0.f};
          const uint4* rowp[4];
          bool live[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int tok = tok0 + col0 + tr + 4 * u;
            live[u] = (tr + 4 * u < ncol) && tok < p.m_tok;
            rowp[u] = reinterpret_cast<const uint4*>(p.norm_src + static_cast<size_t>(live[u] ? tok : tok0) * p.k);
          }
          for (int i0 = lane; i0 < kv8; i0 += 128) {
            uint4 v[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int u = 0; u < 4; ++u)
                v[j][u] = (live[u] && i0 + 32 * j < kv8) ? rowp[u][i0 + 32 * j] : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v[j][u]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float2 f = __bfloat1622float2(h[e]);
                  ss[u] += f.x * f.x + f.y * f.y;
                }
              }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ss[u] += __shfl_xor_sync(0xffffffffu, ss[u], o);
            if (lane == 0 && tr + 4 * u < ncol)
              rstd_s[col0 + tr + 4 * u] = live[u] ? rsqrtf(ss[u] / static_cast<float>(p.k) + p.eps) : 0.f;
          }
        }
      } else {
        if constexpr (MX) {
          if (p.sumsq != nullptr && p.wait_flag != nullptr) {
            // piece head fed by a quantised hop: the sums of squares were accumulated by the upstream piece's tail GEMM
            const uint32_t target = *reinterpret_cast<const volatile uint32_t*>(p.wait_epoch) + 1;
            wait_flag_ge(p.wait_flag, target);
          }
        }
        for (int t = col0 + et; t < col0 + ncol; t += 128) {
          const int tok = tok0 + t;
          float r = (p.rstd != nullptr && tok < p.m_tok) ? p.rstd[tok] : 1.f;
          if constexpr (MX) {
            if (p.sumsq != nullptr && tok < p.m_tok)      // RMSNorm statistics accumulated by the producing GEMM's epilogue
              r *= rsqrtf(p.sumsq[tok] / static_cast<float>(p.k) + p.eps);
          }
          rstd_s[t] = r;
        }
        if constexpr (MX) {
          if (p.zero_buf != nullptr && blockIdx.x == 0 && blockIdx.z == 0)
            for (int t = et; t < BN; t += 128)
              if (tok0 + t < p.m_tok) p.zero_buf[tok0 + t] = 0.f;
        }
      }
      epi_bar_sync();
    }
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    if (threadIdx.x == 64) B2B_DBG(5);
  }

  // ------------------------------------- split-K reduce-scatter through DSMEM
  // After barrier #1 every CTA's main loop has retired, so all stage rings are free.  CTA r of the cluster owns
  // the token columns [r*CW, (r+1)*CW): every CTA scatters its partial accumulator column slices into the owners'
  // landing zones (its own slice included), barrier #2, then every CTA adds the `splitk` partials of its slice and
  // runs the fused epilogue for those CW tokens only.  Compared with "everything to the leader" the epilogue work
  // (residual / RoPE / stores) is spread over the cluster and no CTA idles.
  const int q = warp & 3;
  const int row = q * 32 + lane;                 // TMEM lane == weight row within the tile
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  float* red = reinterpret_cast<float*>(smem);   // landing zone [splitk][128 rows][CW + 4]
  const int CWP = ncol + 4;                      // row pitch in floats (16-byte aligned rows, bank spread)
  if (splitk > 1) {
    cluster_arrive_release();
    cluster_wait_acquire();
    if (warp >= 2) {
      const uint32_t zone = smem_u32(red) + static_cast<uint32_t>(((krank * BM + row) * CWP) * 4);
#pragma unroll 1
      for (int c = 0; c < BN; c += 16) {
        float v[16];
        tmem_ld16(taddr + c, v);
        if (ncol >= 4) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const int col = c + i, d = col / ncol, off = col - d * ncol;
            st_dsmem_v4(mapa_smem(zone, static_cast<uint32_t>(d)) + static_cast<uint32_t>(off * 4),
                        make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int col = c + i, d = col / ncol, off = col - d * ncol;
            st_dsmem_f32(mapa_smem(zone, static_cast<uint32_t>(d)) + static_cast<uint32_t>(off * 4), v[i]);
          }
        }
      }
    }
    cluster_arrive_release();
    cluster_wait_acquire();
  }

  // ------------------------------------------------------------ fused epilogue
  if (warp >= 2) {
    const int n_glob = tile_n * BM + row;
    float* xch = red + (splitk > 1 ? splitk * BM * CWP : 0);   // GLU exchange buffer [ncol][64] (behind the landing zone, if any)
    const float bias_v = (p.bias != nullptr) ? p.bias[n_glob] : 0.f;
    // fp8: per-output-row weight scale (the per-token activation scale rides in rstd_s)
    const float wsc = (FP8 && p.w_scale != nullptr) ? p.w_scale[n_glob] : 1.f;
    const float wsc_up = (FP8 && EPI == EPI_GLU && p.w_scale != nullptr && row < 64) ? p.w_scale[n_glob + 64] : 1.f;

    if (p.free_flag != nullptr) {
      // back-pressure: the consumer must have drained the previous payload of this slot
      const uint32_t e = *reinterpret_cast<const volatile uint32_t*>(p.signal_epoch);
      wait_flag_ge(p.free_flag, e - p.free_lag);
    }

    // QKV section bookkeeping (uniform per CTA)
    int sect = 0, f_in_sect = 0;
    float inv_freq = 0.f;
    const int q_dim = p.n_q_heads * p.head_dim, kv_dim = p.n_kv_heads * p.head_dim;
    if constexpr (EPI == EPI_QKV_ROPE) {
      const int f = n_glob;
      sect = (f < q_dim) ? 0 : (f < q_dim + kv_dim ? 1 : 2);
      f_in_sect = f - (sect == 0 ? 0 : (sect == 1 ? q_dim : q_dim + kv_dim));
      if (sect < 2 && p.rope_theta > 0.f) {
        const int j = (f_in_sect % p.head_dim) >> 1;   // rotary pair index (rows are pair-interleaved)
        inv_freq = exp2f(-(2.f * j / static_cast<float>(p.head_dim)) * log2f(p.rope_theta));
      }
    }

    // Fused MX quantisation of a CHUNK of 16 tokens: every lane holds its feature's value for each token of the chunk
    // (32 lanes = 32 consecutive features = one MX block per token).  The per-token block maximum and sum of squares are
    // computed with a transpose-reduce (8 + 4 + 2 + 1 + 1 shuffles for all 16 tokens instead of 5 dependent shuffles per
    // token): afterwards lanes 2t and 2t+1 hold the totals of token t.
    const int q_nkc = MX ? (p.ld_q >> 7) : 0;
    const int q_chunk = (MX && p.q_bn > 128) ? 1024 : 512;
    auto emit_q_chunk = [&](const float* qv, int tok_base, int nvalid, int feat) {
      float r[16], am[16], ss[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        r[i] = (i < nvalid) ? bf16_round(qv[i]) : 0.f;     // what a separate quantiser would read back from memory
        am[i] = fabsf(r[i]);
        ss[i] = r[i] * r[i];
      }
#pragma unroll
      for (int s = 16, n = 8; n >= 1; s >>= 1, n >>= 1) {
        const bool upper = (lane & s) != 0;
#pragma unroll
        for (int j = 0; j < n; ++j) {
          const float sa = upper ? am[j] : am[j + n], ka = upper ? am[j + n] : am[j];
          const float sq = upper ? ss[j] : ss[j + n], kq = upper ? ss[j + n] : ss[j];
          am[j] = fmaxf(ka, __shfl_xor_sync(0xffffffffu, sa, s));
          ss[j] = kq + __shfl_xor_sync(0xffffffffu, sq, s);
        }
      }
      am[0] = fmaxf(am[0], __shfl_xor_sync(0xffffffffu, am[0], 1));
      ss[0] += __shfl_xor_sync(0xffffffffu, ss[0], 1);
      // this lane's token: t = (lane >> 1) & 15; e = ceil(log2(amax / 448)) clamped to the UE8M0 range
      const uint32_t u = __float_as_uint(am[0] * (1.f / 448.f));
      int e_mine = static_cast<int>(u >> 23) - 127 + ((u & 0x7FFFFFu) ? 1 : 0);
      e_mine = max(-126, min(127, e_mine));
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int e = __shfl_sync(0xffffffffu, e_mine, 2 * i);
        if (i < nvalid) {
          const float inv = __uint_as_float(static_cast<uint32_t>(127 - e) << 23);
          p.q_out8[static_cast<size_t>(tok_base + i) * p.ld_q + feat] =
              static_cast<uint8_t>(__nv_cvt_float_to_fp8(r[i] * inv, __NV_SATFINITE, __NV_E4M3));
        }
      }
      const int t = lane >> 1;
      if ((lane & 1) == 0 && t < nvalid) {
        const int tok = tok_base + t;
        const int tile = tok / p.q_bn, n = tok - tile * p.q_bn, rr = n & 127;
        p.q_sf[(static_cast<size_t>(tile) * q_nkc + (feat >> 7)) * q_chunk + (n >> 7) * 512 + (rr & 31) * 16 + (rr >> 5) * 4 +
               ((feat >> 5) & 3)] = static_cast<uint8_t>(e_mine + 127);
        if (p.sumsq_out != nullptr) {
          if (p.signal_flag != nullptr) atomicAdd_system(&p.sumsq_out[tok], ss[0]);   // tail GEMM: the counter lives in the peer's memory
          else atomicAdd(&p.sumsq_out[tok], ss[0]);
        }
      }
    };

    // accumulators of up to 16 columns starting at local column c (slice-relative)
    auto load_acc = [&](int c, int n, float* v) {
      if (splitk == 1) {
        tmem_ld16(taddr + c, v);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = 0.f;
        for (int r = 0; r < splitk; ++r) {
          const float* pr = red + (r * BM + row) * CWP + c;
          if (n >= 4) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              if (i < n) {
                const float4 q4 = *reinterpret_cast<const float4*>(pr + i);
                v[i] += q4.x; v[i + 1] += q4.y; v[i + 2] += q4.z; v[i + 3] += q4.w;
              }
            }
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < n) v[i] += pr[i];
          }
        }
      }
    };

    if constexpr (EPI == EPI_GLU) {
      // phase A: the "up" half (rows 64..127) parks its values in shared memory
      if (row >= 64) {
#pragma unroll 1
        for (int c = 0; c < ncol; c += 16) {
          const int n = min(16, ncol - c);
          float v[16];
          load_acc(c, n, v);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < n) xch[(c + i) * 64 + (row - 64)] = v[i];
        }
      }
      epi_bar_sync();
    }

#pragma unroll 1
    for (int c = 0; c < ncol; c += 16) {
      if (EPI == EPI_GLU && row >= 64) break;
      if (tok0 + col0 + c >= p.m_tok) break;
      const int n = min(16, ncol - c);
      // residual values of the whole chunk first: 16 independent loads in flight (one L2 round trip) instead of
      // one per token between dependent stores
      __nv_bfloat16 resid[16];
      if constexpr (EPI == EPI_RESIDUAL) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int tok = tok0 + col0 + c + i;
          resid[i] = (i < n && tok < p.m_tok) ? p.residual[static_cast<size_t>(tok) * p.ld_res + n_glob] : __float2bfloat16_rn(0.f);
        }
      }
      float v[16];
      load_acc(c, n, v);
      float qv[16];                              // outputs of this chunk for the fused quantiser
      int q_valid = 0;

#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int lc = col0 + c + i;             // column within the CTA's token tile
        const int tok = tok0 + lc;
        if (i >= n || tok >= p.m_tok) continue;  // warp-uniform: padded token columns do no work
        const float rs = rstd_s[lc];
        const float a = v[i] * rs * wsc + bias_v;
        if constexpr (EPI == EPI_PLAIN) {
          if (p.out_fp32) reinterpret_cast<float*>(p.out)[static_cast<size_t>(tok) * p.ld_out + n_glob] = a;
          else reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<size_t>(tok) * p.ld_out + n_glob] = __float2bfloat16_rn(a);
        } else if constexpr (EPI == EPI_GELU) {
          reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<size_t>(tok) * p.ld_out + n_glob] =
              __float2bfloat16_rn(gelu_tanh(a));
        } else if constexpr (EPI == EPI_RESIDUAL) {
          const float rv = a + __bfloat162float(resid[i]);
          const __nv_bfloat16 r16 = __float2bfloat16_rn(rv);
          reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<size_t>(tok) * p.ld_out + n_glob] = r16;
          if (p.out2 != nullptr)
            reinterpret_cast<__nv_bfloat16*>(p.out2)[static_cast<size_t>(tok) * p.ld_out + n_glob] = r16;
          if constexpr (MX) {      // (anything of the fused quantiser left in the bf16 instantiations cost 50 us per step)
            qv[i] = rv;
            q_valid = i + 1;
          }
        } else if constexpr (EPI == EPI_GLU) {
          const float u = xch[(c + i) * 64 + row] * rs * wsc_up;
          const float g = p.act_gelu ? gelu_tanh(a) : silu(a);
          if (!MX || p.out != nullptr)
            reinterpret_cast<__nv_bfloat16*>(p.out)[static_cast<size_t>(tok) * p.ld_out + tile_n * 64 + row] =
                __float2bfloat16_rn(g * u);
          if constexpr (MX) {
            qv[i] = g * u;
            q_valid = i + 1;
          }
        } else {   // EPI_QKV_ROPE
          float o = a;
          if (sect < 2 && p.rope_theta > 0.f) {
            // lanes (2j, 2j+1) hold (x_j, x_{j+hd/2}) thanks to the offline row interleave
            const float partner = __shfl_xor_sync(0xffffffffu, a, 1);
            float sn, cs;
            sincosf(static_cast<float>(pos_s[lc]) * inv_freq, &sn, &cs);
            o = (lane & 1) ? (a * cs + partner * sn) : (a * cs - partner * sn);
          }
          if (sect == 0) {
            p.q_out[static_cast<size_t>(tok) * q_dim + f_in_sect] = __float2bfloat16_rn(o * p.q_scale);
          } else {
            const int slot = slot_s[lc];
            __nv_bfloat16* dst = (sect == 1 ? p.k_cache : p.v_cache);
            if (slot >= 0) dst[static_cast<size_t>(slot) * kv_dim + f_in_sect] = __float2bfloat16_rn(o);
          }
        }
      }
      if constexpr (MX && (EPI == EPI_RESIDUAL || EPI == EPI_GLU)) {     // (only the MX instantiations pay the registers)
        if (p.q_out8 != nullptr)        // warp-uniform: the valid tokens of a chunk are a prefix
          emit_q_chunk(qv, tok0 + col0 + c, q_valid, EPI == EPI_GLU ? tile_n * 64 + row : n_glob);
      }
    }

    if (threadIdx.x == 64) B2B_DBG(6);
    // ------------------------------------------------ handoff publication
    if (p.signal_flag != nullptr || p.bump_epoch != nullptr) {
      __threadfence_system();            // my (possibly peer-directed) stores are performed
      epi_bar_sync();
      if (threadIdx.x == 64) {
        const uint32_t total = gridDim.x * gridDim.y * gridDim.z;   // every CTA of a split-K cluster stores a slice
        const uint32_t prev = atomicAdd(p.done_counter, 1u);
        if (prev == total - 1) {
          __threadfence_system();
          *p.done_counter = 0;
          if (p.signal_flag != nullptr) {
            const uint32_t e = *reinterpret_cast<volatile uint32_t*>(p.signal_epoch) + 1;
            *reinterpret_cast<volatile uint32_t*>(p.signal_epoch) = e;
            st_release_sys(p.signal_flag, e);
          }
          if (p.bump_epoch != nullptr) {
            const uint32_t e = *reinterpret_cast<volatile uint32_t*>(p.bump_epoch) + 1;
            *reinterpret_cast<volatile uint32_t*>(p.bump_epoch) = e;
            if (p.ack_flag != nullptr) st_release_sys(p.ack_flag, e);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TCOLS>(tmem_base);
  }
  if (threadIdx.x == 0) B2B_DBG(7);
}

// ============================================================== host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

// 2D bf16 row-major [rows, cols] (row stride ld elements), box = [box_rows, 64], 128B swizzle.
static int make_tmap(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, int elt_bytes) {
  using Key = std::tuple<const void*, uint64_t, uint64_t, uint64_t, uint32_t, int>;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> g(mu);
  Key key{ptr, rows, cols, ld, box_rows, elt_bytes};
  auto it = cache.find(key);
  if (it != cache.end()) { *m = it->second; return 0; }
  PFN_encodeTiled enc = get_encode();
  if (!enc) return -1;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * static_cast<uint64_t>(elt_bytes)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(ROW_BYTES / elt_bytes), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, elt_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return static_cast<int>(r);
  if (cache.size() > 65536) cache.clear();
  cache[key] = *m;
  return 0;
}

int make_tmap_shared(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     int elt_bytes) {
  return make_tmap(m, ptr, rows, cols, ld, box_rows, elt_bytes);
}

template <int BN, int EPI, int QM>
static int launch_bn_epi(const GemmParams& p, const CUtensorMap& tw, const CUtensorMap& tx, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  static bool attr_set[64] = {};      // per device: one process may drive several GPUs (enable_peer_access path)
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, QM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::kSmemBytes);
    if (e != cudaSuccess) return static_cast<int>(e);
    if (dev < 64) attr_set[dev] = true;
  }
  return static_cast<int>(launch_kernel(gemm_tc_kernel<BN, EPI, QM>, dim3(p.n_out / BM, (p.m_tok + BN - 1) / BN, p.splitk),
                                        dim3(192), Cfg::smem_bytes(p.stages), stream, static_cast<unsigned>(p.splitk), tw, tx, p));
}

// one compact kernel per (token tile, epilogue): a runtime `switch` in the 16x-unrolled epilogue
// loop made the kernel instruction-fetch bound (5.4 us epilogue, see profiles/gemm_timeline.md)
template <int BN>
static int launch_bn(const GemmParams& p, const CUtensorMap& tw, const CUtensorMap& tx, cudaStream_t stream) {
#define B2B_EPI_CASE(E)                                                                              \
  case E:                                                                                            \
    if (p.fp8 && p.sfa != nullptr) {                                                                 \
      if constexpr (BN >= 32) return launch_bn_epi<BN, E, 2>(p, tw, tx, stream);                     \
      else return -7;   /* MX scale-factor chunks are laid out for token tiles of >= 32 */           \
    }                                                                                                \
    return p.fp8 ? launch_bn_epi<BN, E, 1>(p, tw, tx, stream) : launch_bn_epi<BN, E, 0>(p, tw, tx, stream);
  switch (p.epi) {
    B2B_EPI_CASE(EPI_PLAIN)
    B2B_EPI_CASE(EPI_RESIDUAL)
    B2B_EPI_CASE(EPI_GLU)
    B2B_EPI_CASE(EPI_QKV_ROPE)
    B2B_EPI_CASE(EPI_GELU)
    default: return -4;
  }
#undef B2B_EPI_CASE
}

template <int BN, int EPI, int QM>
static int set_attr_one() {
  return static_cast<int>(cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, QM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               GemmCfg<BN>::kSmemBytes));
}
template <int BN, int EPI>
static int set_attr_epi() {
  int r = 0;
  if ((r = set_attr_one<BN, EPI, 0>()) || (r = set_attr_one<BN, EPI, 1>())) return r;
  if constexpr (BN >= 32) r = set_attr_one<BN, EPI, 2>();
  return r;
}
template <int BN>
static int set_attr_bn() {
  int r = 0;
  if ((r = set_attr_epi<BN, EPI_PLAIN>()) || (r = set_attr_epi<BN, EPI_RESIDUAL>()) || (r = set_attr_epi<BN, EPI_GLU>()) ||
      (r = set_attr_epi<BN, EPI_QKV_ROPE>()) || (r = set_attr_epi<BN, EPI_GELU>()))
    return r;
  return 0;
}
// Opt every instantiation into its dynamic shared memory size up front (so the first real
// launch may happen inside a CUDA-graph capture).
int gemm_tc_init() {
  int r = 0;
  if ((r = set_attr_bn<16>())) return r;
  if ((r = set_attr_bn<32>())) return r;
  if ((r = set_attr_bn<64>())) return r;
  if ((r = set_attr_bn<128>())) return r;
  if ((r = set_attr_bn<256>())) return r;
  return get_encode() ? 0 : -1;
}

int gemm_tc_default_stages(int bn) {
  switch (bn) {
    case 16: return GemmCfg<16>::kStages;
    case 32: return GemmCfg<32>::kStages;
    case 64: return GemmCfg<64>::kStages;
    case 128: return GemmCfg<128>::kStages;
    default: return GemmCfg<256>::kStages;
  }
}

int gemm_tc_max_splitk(int bn, int epi, int stages) {
  // reduce-scatter landing zone in every CTA's stage ring: S * 128 rows * (BN/S + 4) floats (+ GLU exchange BN/S * 256 B)
  int stage_bytes;
  const int dflt = gemm_tc_default_stages(bn);
  if (stages <= 0 || stages > dflt) stages = dflt;
  switch (bn) {
    case 16: stage_bytes = GemmCfg<16>::kStageBytes; break;
    case 32: stage_bytes = GemmCfg<32>::kStageBytes; break;
    case 64: stage_bytes = GemmCfg<64>::kStageBytes; break;
    case 128: stage_bytes = GemmCfg<128>::kStageBytes; break;
    default: stage_bytes = GemmCfg<256>::kStageBytes; break;
  }
  int best = 1;
  for (int s = 2; s <= 8 && bn / s >= 2; s *= 2) {
    const int need = s * 128 * (bn / s + 4) * 4 + (epi == EPI_GLU ? (bn / s) * 256 : 0);
    if (need <= stages * stage_bytes) best = s;
  }
  return best;
}

int launch_gemm_tc(const GemmParams& p_in, const void* w, const void* x, int bn, cudaStream_t stream) {
  GemmParams p = p_in;
  const int elt = p.fp8 ? 1 : 2;
  const int bke = ROW_BYTES / elt;
  if (p.n_out % BM != 0 || p.k % bke != 0 || p.m_tok <= 0) return -2;
  if (p.splitk < 1) p.splitk = 1;
  if (p.splitk > 8) p.splitk = 8;
  {
    const int dflt = gemm_tc_default_stages(bn);
    if (p.stages <= 0 || p.stages > dflt) p.stages = dflt;
    if (p.stages < 2) p.stages = 2;
  }
  {
    // the epilogue reuses the (by then idle) stage ring: GLU exchange buffer bn x 64 floats when there is no split-K
    // landing zone in front of it -- a shallow ring must still hold it
    const int stage_bytes = 128 * 128 + bn * 128;
    const int need = (p.epi == EPI_GLU) ? bn * 256 : 0;
    while (p.stages * stage_bytes < need && p.stages < gemm_tc_default_stages(bn)) ++p.stages;
  }
  const int smax = gemm_tc_max_splitk(bn, p.epi, p.stages);
  if (p.splitk > smax) p.splitk = smax;
  if (p.splitk > p.k / bke) p.splitk = p.k / bke;
  while (p.splitk & (p.splitk - 1)) --p.splitk;      // cluster reduce-scatter: power of two (divides the token tile)
  CUtensorMap tw, tx;
  int r = make_tmap(&tw, w, p.n_out, p.k, p.k, BM, elt);
  if (r) return r;
  r = make_tmap(&tx, x, p.m_tok, p.k, p.k, bn, elt);
  if (r) return r;
  switch (bn) {
    case 16: return launch_bn<16>(p, tw, tx, stream);
    case 32: return launch_bn<32>(p, tw, tx, stream);
    case 64: return launch_bn<64>(p, tw, tx, stream);
    case 128: return launch_bn<128>(p, tw, tx, stream);
    case 256: return launch_bn<256>(p, tw, tx, stream);
    default: return -3;
  }
}

int set_wait_policy_gemm(uint32_t* abort_word, unsigned long long limit_ns) {
  cudaError_t e = cudaMemcpyToSymbol(g_abort_word, &abort_word, sizeof(abort_word));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_wait_limit_ns, &limit_ns, sizeof(limit_ns));
  return static_cast<int>(e);
}

}  // namespace b2b
