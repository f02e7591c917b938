// Python bindings (torch extension `bee2bee_b200._C`).  The only torch-facing translation
// unit: it validates tensors, picks the current CUDA stream and calls the C launchers.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include "gemm_tc.cuh"
#include "kernels.h"
#include "launch.cuh"
#include "peer.h"

using at::Tensor;
using OptT = c10::optional<Tensor>;

namespace {

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

inline void check(int err, const char* what) {
  if (err != 0) {
    const char* msg = err > 0 ? cudaGetErrorString(static_cast<cudaError_t>(err)) : "invalid argument";
    TORCH_CHECK(false, what, " failed: code ", err, " (", msg, ")");
  }
}
template <typename T>
inline T* ptr_or_null(const OptT& t) {
  return (t.has_value() && t->defined()) ? reinterpret_cast<T*>(t->data_ptr()) : nullptr;
}
template <typename T>
inline T* as_ptr(int64_t addr) { return reinterpret_cast<T*>(static_cast<uintptr_t>(addr)); }

void check_bf16(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kBFloat16 && t.is_contiguous(), name,
              " must be a contiguous CUDA bf16 tensor");
}

// ---------------------------------------------------------------------- GEMM
// out[t, n] = epi(X[t,:] . W[n,:]).  Handoff pointers are raw device addresses (0 = unused)
// because they may live in IPC-mapped peer memory.
void gemm(const Tensor& w, const Tensor& x, int64_t out_ptr, int64_t ld_out, int64_t epi, int64_t bn,
          int64_t splitk, int64_t residual_ptr, int64_t ld_res, const OptT& bias, const OptT& rstd,
          bool norm_from_x, double eps, bool act_gelu, bool out_fp32,
          // qkv epilogue
          const OptT& q_out, const OptT& k_cache, const OptT& v_cache, const OptT& positions, const OptT& slots,
          int64_t n_q_heads, int64_t n_kv_heads, int64_t head_dim, double rope_theta, double q_scale,
          // handoff
          int64_t wait_flag, int64_t wait_epoch, int64_t signal_flag, int64_t signal_epoch, int64_t done_counter,
          int64_t free_flag, int64_t bump_epoch, int64_t ack_flag, int64_t dbg, const OptT& w_scale,
          const OptT& sfa, const OptT& sfb, int64_t stages, int64_t free_lag, int64_t out2_ptr,
          // fused MX quantisation of the output / RMSNorm statistics (raw addresses, 0 = off)
          int64_t q_out8, int64_t q_sf, int64_t ld_q, int64_t q_bn, int64_t sumsq_out, int64_t zero_buf, int64_t sumsq) {
  const bool fp8 = w.scalar_type() == at::kFloat8_e4m3fn;
  if (fp8) {
    TORCH_CHECK(x.scalar_type() == at::kFloat8_e4m3fn && w.is_cuda() && x.is_cuda() && w.is_contiguous() &&
                x.is_contiguous(), "fp8 gemm: w and x must be contiguous CUDA float8_e4m3fn");
    const bool mx = sfa.has_value();
    TORCH_CHECK(mx == sfb.has_value(), "MX fp8 gemm needs both sfa and sfb");
    if (mx) {
      const int64_t nkc = w.size(1) / 128, chunk = bn > 128 ? 1024 : 512;
      TORCH_CHECK(w.size(1) % 128 == 0 && bn >= 32, "MX fp8 gemm: K must be a multiple of 128 and bn >= 32");
      TORCH_CHECK(sfa->scalar_type() == at::kByte && sfa->is_contiguous() && sfa->numel() >= (w.size(0) / 128) * nkc * 512,
                  "MX fp8 gemm: sfa too small");
      TORCH_CHECK(sfb->scalar_type() == at::kByte && sfb->is_contiguous() &&
                      sfb->numel() >= ((x.size(0) + bn - 1) / bn) * nkc * chunk, "MX fp8 gemm: sfb too small");
    } else {
      TORCH_CHECK(w_scale.has_value() && w_scale->scalar_type() == at::kFloat, "fp8 gemm needs per-row w_scale (fp32)");
    }
  } else {
    check_bf16(w, "w");
    check_bf16(x, "x");
  }
  TORCH_CHECK(w.dim() == 2 && x.dim() == 2 && w.size(1) == x.size(1), "gemm: shape mismatch");
  c10::cuda::CUDAGuard guard(w.device());
  b2b::GemmParams p{};
  p.m_tok = static_cast<int>(x.size(0));
  p.n_out = static_cast<int>(w.size(0));
  p.k = static_cast<int>(w.size(1));
  p.splitk = static_cast<int8_t>(splitk);
  p.epi = static_cast<int8_t>(epi);
  p.out_fp32 = out_fp32 ? 1 : 0;
  p.act_gelu = act_gelu ? 1 : 0;
  p.fp8 = fp8 ? 1 : 0;
  p.stages = static_cast<int8_t>(stages);
  p.w_scale = ptr_or_null<const float>(w_scale);
  p.sfa = fp8 ? ptr_or_null<const uint8_t>(sfa) : nullptr;
  p.sfb = fp8 ? ptr_or_null<const uint8_t>(sfb) : nullptr;
  p.out = as_ptr<void>(out_ptr);
  p.ld_out = static_cast<int>(ld_out);
  p.out2 = as_ptr<void>(out2_ptr);
  p.q_out8 = as_ptr<uint8_t>(q_out8);
  p.q_sf = as_ptr<uint8_t>(q_sf);
  p.ld_q = static_cast<int>(ld_q);
  p.q_bn = static_cast<int16_t>(q_bn > 0 ? q_bn : 32);
  p.sumsq_out = as_ptr<float>(sumsq_out);
  p.zero_buf = as_ptr<float>(zero_buf);
  p.sumsq = as_ptr<const float>(sumsq);
  TORCH_CHECK(!p.q_out8 || (p.q_sf && p.sfa && p.ld_q % 128 == 0 && (epi == b2b::EPI_RESIDUAL || epi == b2b::EPI_GLU)),
              "fused output quantisation: MX GEMMs with residual / GLU epilogues, scale-factor buffer, row stride multiple of 128");
  p.residual = as_ptr<const __nv_bfloat16>(residual_ptr);
  p.ld_res = static_cast<int>(ld_res);
  p.bias = ptr_or_null<const float>(bias);
  p.rstd = ptr_or_null<const float>(rstd);
  TORCH_CHECK(!(fp8 && norm_from_x), "fp8 gemm: pass the combined activation scale through rstd");
  p.norm_src = norm_from_x ? reinterpret_cast<const __nv_bfloat16*>(x.data_ptr()) : nullptr;
  p.eps = static_cast<float>(eps);
  p.q_out = ptr_or_null<__nv_bfloat16>(q_out);
  p.k_cache = ptr_or_null<__nv_bfloat16>(k_cache);
  p.v_cache = ptr_or_null<__nv_bfloat16>(v_cache);
  p.positions = ptr_or_null<const int>(positions);
  p.slots = ptr_or_null<const int>(slots);
  p.n_q_heads = static_cast<int16_t>(n_q_heads);
  p.n_kv_heads = static_cast<int16_t>(n_kv_heads);
  p.head_dim = static_cast<int16_t>(head_dim);
  p.rope_theta = static_cast<float>(rope_theta);
  p.q_scale = static_cast<float>(q_scale);
  p.wait_flag = as_ptr<const uint32_t>(wait_flag);
  p.wait_epoch = as_ptr<const uint32_t>(wait_epoch);
  p.signal_flag = as_ptr<uint32_t>(signal_flag);
  p.signal_epoch = as_ptr<uint32_t>(signal_epoch);
  p.done_counter = as_ptr<uint32_t>(done_counter);
  p.free_flag = as_ptr<const uint32_t>(free_flag);
  p.bump_epoch = as_ptr<uint32_t>(bump_epoch);
  p.ack_flag = as_ptr<uint32_t>(ack_flag);
  p.free_lag = static_cast<uint8_t>(free_lag);
  p.dbg = as_ptr<unsigned long long>(dbg);
  if (p.epi == b2b::EPI_QKV_ROPE) {
    TORCH_CHECK(p.q_out && p.k_cache && p.v_cache && p.slots, "qkv epilogue needs q_out/k_cache/v_cache/slots");
    TORCH_CHECK(p.rope_theta <= 0.f || p.positions, "rope needs positions");
    TORCH_CHECK((p.n_q_heads * p.head_dim) % 128 == 0 && (p.n_kv_heads * p.head_dim) % 128 == 0,
                "q/kv widths must be multiples of 128");
    TORCH_CHECK(p.n_out == (p.n_q_heads + 2 * p.n_kv_heads) * p.head_dim, "qkv rows mismatch");
  }
  if (p.epi == b2b::EPI_RESIDUAL) TORCH_CHECK(p.residual != nullptr, "residual epilogue needs residual");
  if (p.epi == b2b::EPI_GLU) TORCH_CHECK(p.out != nullptr || (p.q_out8 != nullptr && p.sfa != nullptr), "GLU epilogue needs an output");
  if (p.signal_flag || p.bump_epoch) TORCH_CHECK(p.done_counter != nullptr, "handoff needs done_counter");
  check(b2b::launch_gemm_tc(p, w.data_ptr(), x.data_ptr(), static_cast<int>(bn), cur_stream()), "gemm_tc");
}

// Bounded handoff waits (call once per device after peer_alloc'ing the abort word): limit_ms == 0 restores "trap".
void set_wait_policy(int64_t abort_word, double limit_ms) {
  const auto ns = static_cast<unsigned long long>(limit_ms * 1e6);
  check(b2b::set_wait_policy_gemm(as_ptr<uint32_t>(abort_word), ns), "set_wait_policy(gemm)");
  check(b2b::set_wait_policy_elementwise(as_ptr<uint32_t>(abort_word), ns), "set_wait_policy(elementwise)");
}

void set_pdl(bool on) { b2b::g_pdl_mode = on ? 1 : 0; }
bool get_pdl() { return b2b::pdl_enabled(); }

int64_t gemm_max_splitk(int64_t bn, int64_t epi, int64_t stages) {
  return b2b::gemm_tc_max_splitk(static_cast<int>(bn), static_cast<int>(epi), static_cast<int>(stages));
}

void init_kernels(int64_t device) {
  c10::cuda::CUDAGuard guard(static_cast<c10::DeviceIndex>(device));
  check(b2b::gemm_tc_init(), "gemm_tc_init");
  check(b2b::attention_init(), "attention_init");
}

// ----------------------------------------------------------------- elementwise
void rmsnorm(const Tensor& x, const Tensor& gamma, const OptT& residual, const OptT& out, const OptT& rstd_out,
             double eps, bool gemma_plus_one) {
  check_bf16(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  const int h = static_cast<int>(x.size(-1));
  const int tokens = static_cast<int>(x.numel() / h);
  check(b2b::launch_rmsnorm(x.data_ptr(), gamma.data_ptr(), ptr_or_null<void>(residual), ptr_or_null<void>(out),
                            ptr_or_null<float>(rstd_out), tokens, h, static_cast<float>(eps), gemma_plus_one ? 1 : 0,
                            cur_stream()),
        "rmsnorm");
}

void layernorm(const Tensor& x, const Tensor& gamma, const Tensor& beta, const Tensor& out, double eps) {
  check_bf16(x, "x");
  c10::cuda::CUDAGuard guard(x.device());
  const int h = static_cast<int>(x.size(-1));
  check(b2b::launch_layernorm(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
                              static_cast<int>(x.numel() / h), h, static_cast<float>(eps), cur_stream()),
        "layernorm");
}

void embed(int64_t ids_ptr, const Tensor& table, const OptT& pos_table, const OptT& positions, const Tensor& out,
           double scale, int64_t tok_flag, int64_t tok_epoch, int64_t pf_flag, int64_t pf_need) {
  check_bf16(table, "table");
  c10::cuda::CUDAGuard guard(table.device());
  const int h = static_cast<int>(table.size(1));
  check(b2b::launch_embed(as_ptr<const int>(ids_ptr), table.data_ptr(), ptr_or_null<void>(pos_table),
                          ptr_or_null<const int>(positions), out.data_ptr(), static_cast<int>(out.numel() / h), h,
                          static_cast<int>(table.size(0)), static_cast<float>(scale), as_ptr<const uint32_t>(tok_flag),
                          as_ptr<const uint32_t>(tok_epoch), as_ptr<const uint32_t>(pf_flag), as_ptr<const uint32_t>(pf_need),
                          cur_stream()),
        "embed");
}

void kv_append(const Tensor& qkv, const Tensor& q_out, const Tensor& k_cache, const Tensor& v_cache,
               const Tensor& slots, int64_t q_dim, int64_t kv_dim, double q_scale) {
  check_bf16(qkv, "qkv");
  c10::cuda::CUDAGuard guard(qkv.device());
  check(b2b::launch_kv_append(qkv.data_ptr(), q_out.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(),
                              reinterpret_cast<const int*>(slots.data_ptr()), static_cast<int>(qkv.size(0)),
                              static_cast<int>(q_dim), static_cast<int>(kv_dim), static_cast<float>(q_scale),
                              cur_stream()),
        "kv_append");
}

void add(const Tensor& a, const Tensor& b, const Tensor& out) {
  check_bf16(a, "a");
  c10::cuda::CUDAGuard guard(a.device());
  check(b2b::launch_add(a.data_ptr(), b.data_ptr(), out.data_ptr(), static_cast<size_t>(a.numel()), cur_stream()),
        "add");
}

void quant_fp8_rows(const Tensor& x, const Tensor& q, const Tensor& scale_out, double eps, bool with_rms) {
  check_bf16(x, "x");
  TORCH_CHECK(q.scalar_type() == at::kFloat8_e4m3fn && q.is_contiguous() && scale_out.scalar_type() == at::kFloat,
              "quant_fp8_rows: q must be float8_e4m3fn, scale fp32");
  c10::cuda::CUDAGuard guard(x.device());
  const int h = static_cast<int>(x.size(-1));
  check(b2b::launch_quant_fp8_rows(x.data_ptr(), q.data_ptr(), reinterpret_cast<float*>(scale_out.data_ptr()),
                                   static_cast<int>(x.numel() / h), h, static_cast<float>(eps), with_rms ? 1 : 0,
                                   cur_stream()),
        "quant_fp8_rows");
}

void quant_mxfp8_rows(const Tensor& x, const Tensor& q, const Tensor& sf, int64_t bn, double eps, int64_t with_rms,
                      const OptT& sumsq_out) {
  check_bf16(x, "x");
  TORCH_CHECK(q.scalar_type() == at::kFloat8_e4m3fn && q.is_contiguous() && sf.scalar_type() == at::kByte &&
                  sf.is_contiguous(), "quant_mxfp8_rows: q must be float8_e4m3fn, sf uint8");
  c10::cuda::CUDAGuard guard(x.device());
  const int h = static_cast<int>(x.size(-1));
  const int tokens = static_cast<int>(x.numel() / h);
  TORCH_CHECK(sf.numel() >= ((tokens + bn - 1) / bn) * (h / 128) * (bn > 128 ? 1024 : 512), "quant_mxfp8_rows: sf too small");
  check(b2b::launch_quant_mxfp8_rows(x.data_ptr(), q.data_ptr(), sf.data_ptr(), tokens, h, static_cast<int>(bn),
                                     static_cast<float>(eps), static_cast<int>(with_rms), ptr_or_null<float>(sumsq_out),
                                     cur_stream()),
        "quant_mxfp8_rows");
}

void flag_wait(int64_t flag, int64_t epoch, int64_t delta) {
  check(b2b::launch_flag_wait(as_ptr<const uint32_t>(flag), as_ptr<const uint32_t>(epoch),
                              static_cast<uint32_t>(delta), cur_stream()),
        "flag_wait");
}
void decode_advance(const Tensor& positions, const Tensor& kv_len, const Tensor& slots, const Tensor& q_len,
                    const Tensor& block_table) {
  c10::cuda::CUDAGuard guard(positions.device());
  check(b2b::launch_decode_advance(reinterpret_cast<int*>(positions.data_ptr()), reinterpret_cast<int*>(kv_len.data_ptr()),
                                   reinterpret_cast<int*>(slots.data_ptr()),
                                   reinterpret_cast<const int*>(q_len.data_ptr()),
                                   reinterpret_cast<const int*>(block_table.data_ptr()),
                                   static_cast<int>(block_table.size(1)), static_cast<int>(positions.numel()),
                                   cur_stream()),
        "decode_advance");
}
void flag_signal(int64_t flag, int64_t epoch, int64_t bump_epoch, int64_t ack_flag) {
  check(b2b::launch_flag_signal(as_ptr<uint32_t>(flag), as_ptr<uint32_t>(epoch), as_ptr<uint32_t>(bump_epoch),
                                as_ptr<uint32_t>(ack_flag), cur_stream()),
        "flag_signal");
}

// -------------------------------------------------------------------- attention
// query-chunk length from which the tensor-core prefill kernel is used (0 = never); env B2B_ATTN_TC_MIN_Q
static int64_t g_attn_tc_min_q = [] {
  const char* e = std::getenv("B2B_ATTN_TC_MIN_Q");
  return e ? static_cast<int64_t>(std::atoi(e)) : static_cast<int64_t>(2);
}();
void set_attn_tc_min_q(int64_t v) { g_attn_tc_min_q = v; }
int64_t get_attn_tc_min_q() { return g_attn_tc_min_q; }

void attention(const Tensor& q, const Tensor& k_cache, const Tensor& v_cache, const Tensor& out,
               const Tensor& block_table, const Tensor& q_start, const Tensor& q_len, const Tensor& kv_len,
               const OptT& ws, int64_t max_q, int64_t n_q, int64_t n_kv, int64_t head_dim, int64_t window,
               double softcap, int64_t splits, int64_t use_tc, int64_t fq_out, int64_t fq_sf, int64_t fq_bn) {
  check_bf16(q, "q");
  c10::cuda::CUDAGuard guard(q.device());
  TORCH_CHECK(block_table.scalar_type() == at::kInt && q_len.scalar_type() == at::kInt, "int32 metadata expected");
  const int seqs = static_cast<int>(q_len.size(0));
  // use_tc: -1 = by query-chunk length (prefill chunks), 1 = force the tcgen05 kernel (decode: one-token query blocks,
  // the GQA group stacked into the MMA rows), 0 = force the CUDA-core kernel (split-KV decode of few sequences)
  const bool want_tc = use_tc < 0 ? (max_q >= g_attn_tc_min_q && g_attn_tc_min_q > 0) : (use_tc > 0 && g_attn_tc_min_q > 0);
  if (want_tc && splits > 1 && max_q == 1) {
    TORCH_CHECK(ws.has_value(), "split-KV needs a workspace");
    const int64_t R = b2b::attn_rows(static_cast<int>(n_q / n_kv), 1);
    TORCH_CHECK(ws->numel() >= seqs * n_kv * splits * R * (head_dim + 2), "attention workspace too small");
  }
  if (want_tc &&
      b2b::attention_tc_supported(static_cast<int>(n_q), static_cast<int>(n_kv), static_cast<int>(head_dim))) {
    // prefill chunk: tcgen05 flash attention
    check(b2b::launch_attention_tc(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(),
                                   reinterpret_cast<const int*>(block_table.data_ptr()),
                                   reinterpret_cast<const int*>(q_start.data_ptr()),
                                   reinterpret_cast<const int*>(q_len.data_ptr()),
                                   reinterpret_cast<const int*>(kv_len.data_ptr()), seqs, static_cast<int>(max_q),
                                   static_cast<int>(block_table.size(1)), static_cast<int>(q.size(0)),
                                   static_cast<int>(k_cache.size(0)), static_cast<int>(n_q), static_cast<int>(n_kv),
                                   static_cast<int>(head_dim), static_cast<int>(window), static_cast<float>(softcap),
                                   static_cast<int>(splits), ptr_or_null<float>(ws), as_ptr<void>(fq_out), as_ptr<void>(fq_sf),
                                   static_cast<int>(fq_bn), cur_stream()),
          "attention_tc");
    return;
  }
  TORCH_CHECK(fq_out == 0, "fused output quantisation needs the tcgen05 attention kernel");
  if (splits > 1) {
    TORCH_CHECK(ws.has_value(), "split-KV needs a workspace");
    const int64_t R = b2b::attn_rows(static_cast<int>(n_q / n_kv), 1);
    TORCH_CHECK(ws->numel() >= seqs * n_kv * splits * R * (head_dim + 2), "attention workspace too small");
  }
  check(b2b::launch_attention(q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), out.data_ptr(),
                              reinterpret_cast<const int*>(block_table.data_ptr()),
                              reinterpret_cast<const int*>(q_start.data_ptr()),
                              reinterpret_cast<const int*>(q_len.data_ptr()),
                              reinterpret_cast<const int*>(kv_len.data_ptr()), ptr_or_null<float>(ws), seqs,
                              static_cast<int>(max_q), static_cast<int>(block_table.size(1)), static_cast<int>(n_q),
                              static_cast<int>(n_kv), static_cast<int>(head_dim), static_cast<int>(window),
                              static_cast<float>(softcap), static_cast<int>(splits), cur_stream()),
        "attention");
}

// ---------------------------------------------------------------------- sampler
void sample(const Tensor& logits, const OptT& seen, const Tensor& out_tokens, int64_t peer_tokens,
            int64_t history, const OptT& hist_pos, int64_t hist_stride, int64_t vocab, double softcap,
            const OptT& temperature, const OptT& top_p,
            const OptT& rep_penalty, const OptT& seeds, const OptT& step, int64_t signal_flag, int64_t signal_epoch,
            int64_t done_counter, int64_t row_map) {
  TORCH_CHECK(logits.is_cuda() && logits.scalar_type() == at::kFloat && logits.stride(1) == 1, "logits: fp32");
  c10::cuda::CUDAGuard guard(logits.device());
  int* hp = ptr_or_null<int>(hist_pos);
  check(b2b::launch_sample(reinterpret_cast<const float*>(logits.data_ptr()), ptr_or_null<uint32_t>(seen),
                           reinterpret_cast<int*>(out_tokens.data_ptr()), as_ptr<int>(peer_tokens),
                           as_ptr<int>(history), hp, hp, static_cast<int>(hist_stride),
                           static_cast<int>(logits.size(0)), static_cast<int>(vocab > 0 ? vocab : logits.size(1)),
                           static_cast<int>(logits.stride(0)), static_cast<float>(softcap),
                           ptr_or_null<const float>(temperature), ptr_or_null<const float>(top_p),
                           ptr_or_null<const float>(rep_penalty), ptr_or_null<const uint32_t>(seeds),
                           ptr_or_null<const uint32_t>(step), as_ptr<uint32_t>(signal_flag),
                           as_ptr<uint32_t>(signal_epoch), as_ptr<uint32_t>(done_counter), as_ptr<const int>(row_map),
                           cur_stream()),
        "sample");
}

void set_decode_state(const Tensor& positions, const Tensor& kv_len, const Tensor& q_len, int64_t row_map, int64_t kvlen,
                      int64_t n) {
  c10::cuda::CUDAGuard guard(positions.device());
  check(b2b::launch_set_decode_state(reinterpret_cast<int*>(positions.data_ptr()), reinterpret_cast<int*>(kv_len.data_ptr()),
                                     reinterpret_cast<int*>(q_len.data_ptr()), as_ptr<const int>(row_map),
                                     as_ptr<const int>(kvlen), static_cast<int>(n), cur_stream()),
        "set_decode_state");
}

// history / cursors / out / waits are raw addresses: the ring may be peer memory, the rest mapped pinned host memory
void fetch_window(int64_t history, int64_t hist_stride, int64_t cursors, int64_t rows, int64_t width, int64_t out,
                  int64_t waits, int64_t n_waits, int64_t status) {
  check(b2b::launch_fetch_window(as_ptr<const int>(history), static_cast<int>(hist_stride), as_ptr<const int>(cursors),
                                 static_cast<int>(rows), static_cast<int>(width), as_ptr<int>(out),
                                 as_ptr<const b2b::FlagWait>(waits), static_cast<int>(n_waits), as_ptr<int>(status),
                                 cur_stream()),
        "fetch_window");
}

void mark_seen(const Tensor& ids, const Tensor& seq_of, const Tensor& seen, int64_t vocab) {
  c10::cuda::CUDAGuard guard(ids.device());
  check(b2b::launch_mark_seen(reinterpret_cast<const int*>(ids.data_ptr()),
                              reinterpret_cast<const int*>(seq_of.data_ptr()),
                              reinterpret_cast<uint32_t*>(seen.data_ptr()), static_cast<int>(ids.numel()),
                              static_cast<int>(vocab), cur_stream()),
        "mark_seen");
}

// ------------------------------------------------------------------ peer memory
int64_t peer_alloc(int64_t bytes) {
  void* p = nullptr;
  check(b2b::peer_alloc(static_cast<size_t>(bytes), &p), "peer_alloc");
  return static_cast<int64_t>(reinterpret_cast<uintptr_t>(p));
}
void peer_free(int64_t p) { check(b2b::peer_free(as_ptr<void>(p)), "peer_free"); }
py::bytes ipc_export(int64_t p) {
  char h[64];
  check(b2b::ipc_export(as_ptr<void>(p), h), "cudaIpcGetMemHandle");
  return py::bytes(h, 64);
}
int64_t ipc_import(const std::string& handle) {
  TORCH_CHECK(handle.size() == 64, "IPC handle must be 64 bytes");
  void* p = nullptr;
  check(b2b::ipc_import(handle.data(), &p), "cudaIpcOpenMemHandle");
  return static_cast<int64_t>(reinterpret_cast<uintptr_t>(p));
}
void ipc_close(int64_t p) { check(b2b::ipc_close(as_ptr<void>(p)), "cudaIpcCloseMemHandle"); }
void enable_peer_access(int64_t dev, int64_t peer) {
  check(b2b::enable_peer_access(static_cast<int>(dev), static_cast<int>(peer)), "cudaDeviceEnablePeerAccess");
}
bool can_access_peer(int64_t dev, int64_t peer) {
  return b2b::can_access_peer(static_cast<int>(dev), static_cast<int>(peer)) != 0;
}
void memcpy_peer(int64_t dst, int64_t dst_dev, int64_t src, int64_t src_dev, int64_t bytes) {
  check(b2b::memcpy_peer_async(as_ptr<void>(dst), static_cast<int>(dst_dev), as_ptr<const void>(src),
                               static_cast<int>(src_dev), static_cast<size_t>(bytes), cur_stream()),
        "cudaMemcpyPeerAsync");
}
std::pair<int64_t, int64_t> host_ring_alloc(int64_t bytes) {
  void *h = nullptr, *d = nullptr;
  check(b2b::host_ring_alloc(static_cast<size_t>(bytes), &h, &d), "cudaHostAlloc");
  return {static_cast<int64_t>(reinterpret_cast<uintptr_t>(h)), static_cast<int64_t>(reinterpret_cast<uintptr_t>(d))};
}
void host_ring_free(int64_t h) { check(b2b::host_ring_free(as_ptr<void>(h)), "cudaFreeHost"); }

// View raw (possibly peer-mapped or host-mapped) memory as a tensor; no ownership.
Tensor tensor_from_ptr(int64_t p, std::vector<int64_t> sizes, const std::string& dtype, int64_t device) {
  at::ScalarType st = dtype == "bf16" ? at::kBFloat16 : dtype == "f32" ? at::kFloat : dtype == "i32" ? at::kInt
                      : dtype == "u8" ? at::kByte : at::kLong;
  auto opts = at::TensorOptions().dtype(st);
  opts = device >= 0 ? opts.device(at::kCUDA, static_cast<c10::DeviceIndex>(device)) : opts.device(at::kCPU);
  return at::from_blob(as_ptr<void>(p), sizes, opts);
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "bee2bee_b200 native sm_100a kernels + NVLink peer-memory runtime";
  m.def("gemm", &gemm);
  m.def("gemm_max_splitk", &gemm_max_splitk);
  m.def("init_kernels", &init_kernels);
  m.def("set_pdl", &set_pdl);
  m.def("get_pdl", &get_pdl);
  m.def("rmsnorm", &rmsnorm);
  m.def("layernorm", &layernorm);
  m.def("embed", &embed);
  m.def("kv_append", &kv_append);
  m.def("add", &add);
  m.def("quant_fp8_rows", &quant_fp8_rows);
  m.def("quant_mxfp8_rows", &quant_mxfp8_rows);
  m.def("flag_wait", &flag_wait);
  m.def("flag_signal", &flag_signal);
  m.def("decode_advance", &decode_advance);
  m.def("attention", &attention);
  m.def("set_attn_tc_min_q", &set_attn_tc_min_q);
  m.def("get_attn_tc_min_q", &get_attn_tc_min_q);
  m.def("sample", &sample);
  m.def("mark_seen", &mark_seen);
  m.def("set_decode_state", &set_decode_state);
  m.def("fetch_window", &fetch_window);
  m.def("set_wait_policy", &set_wait_policy);
  m.def("peer_alloc", &peer_alloc);
  m.def("peer_free", &peer_free);
  m.def("ipc_export", &ipc_export);
  m.def("ipc_import", &ipc_import);
  m.def("ipc_close", &ipc_close);
  m.def("enable_peer_access", &enable_peer_access);
  m.def("can_access_peer", &can_access_peer);
  m.def("memcpy_peer", &memcpy_peer);
  m.def("host_ring_alloc", &host_ring_alloc);
  m.def("host_ring_free", &host_ring_free);
  m.def("tensor_from_ptr", &tensor_from_ptr);
}
