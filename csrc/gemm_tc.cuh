// Parameter block shared by the tcgen05 GEMM kernel and its host launcher.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace b2b {

enum GemmEpilogue : int {
  EPI_PLAIN = 0,      // out = s*acc (+bias)                               -> bf16 or fp32
  EPI_RESIDUAL = 1,   // out = s*acc (+bias) + residual                    -> bf16 (O-proj / down-proj / piece tail)
  EPI_GLU = 2,        // rows [0,64) gate, [64,128) up: out = act(g)*u     -> bf16 (SwiGLU / GeGLU)
  EPI_QKV_ROPE = 3,   // q: rope -> q buffer; k: rope -> paged K; v -> paged V
  EPI_GELU = 4,       // out = gelu_tanh(s*acc + bias)                     -> bf16 (GPT-2 MLP up)
};

struct GemmParams {
  // problem: out[t, n] = epi( sum_k X[t,k] * W[n,k] ),  W is [N, K] row-major (K-major)
  int m_tok;          // rows of X
  int n_out;          // rows of W (multiple of 128)
  int k;              // multiple of 64
  int8_t splitk;         // cluster size along grid.z (1..8)
  int8_t epi;
  int8_t out_fp32;       // EPI_PLAIN only: write fp32 (logits)
  int8_t act_gelu;       // EPI_GLU: 0 = SiLU (SwiGLU), 1 = tanh-GELU (GeGLU)
  int8_t fp8;            // operands are e4m3 (W8A8): W [N,K] and X [T,K] one byte per element
  int8_t stages;         // shared-memory ring depth (0 = the token tile's default)
  const float* w_scale;  // fp8: per-output-row dequant scale [n_out] (activation scale rides in `rstd`)
  // MX fp8 (tcgen05 kind::mxf8f6f4.block_scale): UE8M0 scale per 32 K elements, pre-arranged in 512-byte
  // chunks per (128 rows, 128 K): byte (r % 32) * 16 + (r / 32) * 4 + (k / 32) % 4.  sfa: weights
  // [n_out/128][k/128][512]; sfb: activations [token tiles of BN][k/128][512 * ceil(BN/128)].  null = not MX.
  const uint8_t* sfa;
  const uint8_t* sfb;

  void* out;          // [m_tok, ld_out]
  int ld_out;
  void* out2;         // EPI_RESIDUAL: optional second destination with the same layout (e.g. the peer's staging slot), or null
  const __nv_bfloat16* residual;  // [m_tok, ld_res]
  int ld_res;
  const float* bias;              // [n_out] or null

  // fused RMSNorm of the input: gamma is pre-folded into W, so only the per-token
  // 1/rms remains; it is either given (rstd) or computed by the epilogue warps
  // from the raw input rows while the MMA pipeline runs (norm_src).
  const float* rstd;              // [m_tok] or null
  const __nv_bfloat16* norm_src;  // [m_tok, k] raw input (same tensor as X) or null
  float eps;

  // Fused MX quantisation of the OUTPUT for the next GEMM (EPI_RESIDUAL / EPI_GLU): e4m3 values + UE8M0 scale per 32
  // features in the consumer's scale-factor chunk layout (token tile q_bn), optional per-token sum of squares of the
  // output (the consumer's RMSNorm: 1/rms is applied in ITS epilogue from `sumsq`), optional zeroing of the other
  // norm point's accumulator.  A warp of the epilogue owns 32 consecutive output features = one MX block per token.
  uint8_t* q_out8;                // [m_tok, ld_q] e4m3, or null
  uint8_t* q_sf;                  // scale-factor chunks of the consumer GEMM's activation operand
  int ld_q;                       // row stride of q_out8 in elements (= consumer K)
  int16_t q_bn;                   // consumer token tile (chunk layout), >= 32
  float* sumsq_out;               // [m_tok] += sum over this CTA's features of out^2, or null
  float* zero_buf;                // [m_tok] accumulator to clear (read by an earlier GEMM, re-filled by a later one), or null
  const float* sumsq;             // consumer side: per-token sum of squares of X -> rstd = rsqrt(sumsq / k + eps)

  // EPI_QKV_ROPE
  __nv_bfloat16* q_out;           // [m_tok, n_q_heads*head_dim]
  __nv_bfloat16* k_cache;         // [slots, n_kv_heads, head_dim]
  __nv_bfloat16* v_cache;
  const int* positions;           // [m_tok]
  const int* slots;               // [m_tok] physical KV slot of each token
  int16_t n_q_heads, n_kv_heads, head_dim;
  float rope_theta;               // <=0: no rotary
  float q_scale;                  // folded softmax scale applied to q (1.0 = none)

  // NVLink piece handoff ---------------------------------------------------
  // consumer side (head-of-piece GEMM): wait until *wait_flag >= *wait_epoch + 1
  // before touching X / norm_src (weights are prefetched meanwhile).
  const uint32_t* wait_flag;
  const uint32_t* wait_epoch;
  // producer side (tail-of-piece GEMM): `out`/`residual` target may be peer memory.
  // After every CTA has stored its tile: last CTA publishes epoch+1 to *signal_flag
  // (st.release.sys on the peer), bumps *signal_epoch, and optionally bumps the
  // consumer-side epoch of this piece's own input slot + acks the upstream producer.
  uint32_t* signal_flag;          // peer (or local) flag
  uint32_t* signal_epoch;         // local: number of handoffs already published on this slot
  uint32_t* done_counter;         // local, self-resetting
  const uint32_t* free_flag;      // local: consumer's ack (it has released `*free_flag` payloads of this slot)
  uint8_t free_lag;               // payloads that may be outstanding: 0 = single staging buffer, 1 = double-buffered
  uint32_t* bump_epoch;           // local: this piece's input-slot epoch (incremented once)
  uint32_t* ack_flag;             // peer: upstream producer's free_flag for our input slot

  // optional per-CTA timeline (globaltimer ns) for tuning: 8 slots per CTA, null = off
  unsigned long long* dbg;
};

// Host launcher (gemm_tc.cu). Returns cudaError_t as int.
int gemm_tc_max_splitk(int bn, int epi, int stages);
int launch_gemm_tc(const GemmParams& p, const void* w, const void* x, int bn, cudaStream_t stream);

}  // namespace b2b
