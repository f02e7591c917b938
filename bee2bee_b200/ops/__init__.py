"""Python face of the hand-written sm_100a kernels (``csrc/*.cu`` -> ``bee2bee_b200/_C``).

Every function here launches a native kernel on the current CUDA stream.  There is no
silent PyTorch fallback on a GPU box: if the extension is missing, ``native()`` raises.
(The CPU execution backend is ``bee2bee_b200.models.torch_ref`` and is selected explicitly
by device, never by an import failure.)
"""
from __future__ import annotations

import importlib
import importlib.util
from typing import Optional

import torch

EPI_PLAIN, EPI_RESIDUAL, EPI_GLU, EPI_QKV_ROPE, EPI_GELU = 0, 1, 2, 3, 4
PAGE = 64           # tokens per KV page (csrc/attention.cu)
NUM_SMS = 148

_C = None

# Kernel launches issued through the extension (eager calls and calls recorded into a CUDA graph alike): every entry
# point that launches exactly one kernel bumps LAUNCHES[0]; the split-KV attention merge pass is added by
# ``attention``.  The runner reads the delta around a graph capture, so the launch counts it reports are the kernels
# that were actually recorded, not a formula.
LAUNCHES = [0]
_KERNEL_ENTRY_POINTS = ("add", "attention", "decode_advance", "embed", "fetch_window", "flag_signal", "flag_wait", "gemm",
                        "kv_append", "layernorm", "mark_seen", "quant_fp8_rows", "quant_mxfp8_rows", "rmsnorm", "sample",
                        "set_decode_state")


class _CountedModule:
    """The extension module with its kernel entry points wrapped by a launch counter (everything else passes through)."""

    def __init__(self, mod):
        self._mod = mod
        for name in dir(mod):
            if name.startswith("__"):
                continue
            fn = getattr(mod, name)
            setattr(self, name, self._counted(fn) if name in _KERNEL_ENTRY_POINTS and callable(fn) else fn)

    @staticmethod
    def _counted(fn):
        def call(*a, **kw):
            LAUNCHES[0] += 1
            return fn(*a, **kw)
        call.__name__ = getattr(fn, "__name__", "kernel")
        call.__doc__ = getattr(fn, "__doc__", None)
        return call


def native():
    """The compiled extension module; built in-tree by ``__graft_entry__.build()``."""
    global _C
    if _C is None:
        try:
            _C = _CountedModule(importlib.import_module("bee2bee_b200._C"))
        except ImportError as e:  # pragma: no cover - exercised only on broken installs
            raise RuntimeError(
                "bee2bee_b200 native extension is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                f"at the repo root (import error: {e})") from e
    return _C


def has_native() -> bool:
    try:
        native()
        return True
    except RuntimeError:
        return False


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


# ------------------------------------------------------------------ weight prep
def rope_interleave_rows(w: torch.Tensor, n_heads: int, head_dim: int) -> torch.Tensor:
    """Row permutation inside each head: new row 2j <- old j, 2j+1 <- old j + D/2, so a rotary
    pair sits in adjacent TMEM lanes of the QKV GEMM epilogue.  q.k dot products are invariant
    under the (shared) permutation, so attention is unchanged."""
    half = head_dim // 2
    idx = torch.arange(head_dim, device=w.device).view(2, half).t().reshape(-1)   # [0, half, 1, half+1, ...]
    wv = w.view(n_heads, head_dim, *w.shape[1:])
    return wv[:, idx].reshape(w.shape).contiguous()


def glu_interleave_rows(w_gate: torch.Tensor, w_up: torch.Tensor) -> torch.Tensor:
    """[gate 0..63 | up 0..63 | gate 64..127 | up 64..127 | ...]: each 128-row MMA tile carries the
    gate and up rows of the same 64 output features (csrc/gemm_tc.cu EPI_GLU)."""
    f, h = w_gate.shape
    assert f % 64 == 0
    g = w_gate.view(f // 64, 64, h)
    u = w_up.view(f // 64, 64, h)
    return torch.cat([g, u], 1).reshape(2 * f, h).contiguous()


def fold_gamma(w: torch.Tensor, gamma: torch.Tensor, plus_one: bool = False) -> torch.Tensor:
    """W' = W diag(gamma): RMSNorm's scale folded into the consuming projection."""
    g = gamma.float() + 1.0 if plus_one else gamma.float()
    return (w.float() * g[None, :]).to(w.dtype).contiguous()


def pad_rows(w: torch.Tensor, multiple: int = 128) -> torch.Tensor:
    r = w.shape[0]
    pad = (-r) % multiple
    if pad == 0:
        return w.contiguous()
    return torch.cat([w, w.new_zeros((pad, *w.shape[1:]))], 0).contiguous()


# ------------------------------------------------------------------------ GEMM
def pick_bn(m_tok: int) -> int:
    for bn in (16, 32, 64, 128):
        if m_tok <= bn:
            return bn
    return 256 if m_tok > 512 else 128


def pick_prefill_tile(n_out: int, m_tok: int, k: int = 0):
    """(token tile, ring depth, cluster split-K) of a prefill GEMM (m_tok > 64), measured on B200 on the Llama-3-8B shapes
    (profiles/prefill_gemm.md).  0 = the tile's default depth / let ``pick_splitk`` decide.

    * more tiles than SMs: TWO resident CTAs per SM with a shallow ring beat one CTA with a deep ring -- the epilogue of
      one tile (TMEM -> registers -> global) overlaps the main loop of the other (955 vs 787 TFLOP/s over the layer at
      4096 tokens, 570 vs 551 at 512);
    * fewer tiles than SMs (O-proj / down / QKV of a 256-1024 token chunk: 32-48 weight tiles): fill the machine with
      split-K instead of running 2 waves of deep-ring CTAs.  Long K (down, 14336): 256-wide token tiles (the 128x256 MMA
      runs at full rate, 128x128 does not), one CTA per SM, split-K until ~one CTA per SM (512 tokens: 66.9 vs 109.5 us).
      Short K: 128-wide tiles with a 3-deep ring, two CTAs per SM, split-K until ~two CTAs per SM (O-proj, 512 tokens:
      37.1 vs 55.7 us).  At least 32 k-blocks per CTA, split-K <= 4."""
    tn = n_out // 128
    tiles256 = tn * ((m_tok + 255) // 256)
    tiles128 = tn * ((m_tok + 127) // 128)
    if m_tok > 256 and tiles256 > NUM_SMS:
        return 256, 2, 1
    kb = k // 64

    def split(tiles: int, cap: int) -> int:
        s = 1
        while s < 4 and tiles * s * 2 <= cap and kb // (s * 2) >= 32:
            s *= 2
        return s

    if m_tok >= 256 and k >= 8192 and tiles256 <= NUM_SMS:
        return 256, 0, split(tiles256, NUM_SMS)
    if tiles128 > NUM_SMS:
        return 128, 3, 1
    if m_tok >= 256 and k > 0:
        return 128, 3, split(tiles128, 2 * NUM_SMS)
    return (128 if m_tok <= 512 else 256), 0, 0          # small chunks: not measured, the decode heuristic decides


#: tuning hook: {"buf": int64 cuda tensor, "off": 0, "log": []} makes every GEMM record a per-CTA timeline
TIMELINE = None

#: (n_out, k) -> split-K override (tuning / sweeps)
SPLITK_OVERRIDE = {}


def pick_splitk(n_out: int, m_tok: int, k: int, bn: int, epi: int, stages: int = 0) -> int:
    """Cluster size along K.  Powers of two only: odd cluster sizes (6, 7) schedule poorly on the
    GPC grid (ncu: launch__cluster_max_active 22 for size 6 vs 74 for size 4)."""
    if (n_out, k) in SPLITK_OVERRIDE:
        want = SPLITK_OVERRIDE[(n_out, k)]
    else:
        # measured (tools/layer_sweep.py, Llama-3-8B, reduce-scatter split-K epilogue): up to ~2 CTAs per SM pay off
        # (bn=32: qkv 4, o 4, gate/up 1, down 8 -> 100 us/layer; bn=16: 4/4/1/4 -> 92.6 us); >= 16 k-blocks per
        # CTA, and every CTA of the cluster keeps >= 4 token columns (vector DSMEM stores)
        tiles = (n_out // 128) * ((m_tok + bn - 1) // bn)
        limit = 256 if bn >= 32 else 200
        want = 1
        while tiles * want * 2 <= limit and want < 8 and bn // (want * 2) >= 4:
            want *= 2
        while want > 1 and (k // 64) // want < 16:
            want //= 2
    want = min(want, 8, max(1, (k // 64) // 2))
    cap = native().gemm_max_splitk(bn, epi, stages)
    while want > cap:
        want //= 2
    return max(1, want)


def gemm(w: torch.Tensor, x: torch.Tensor, out: Optional[torch.Tensor] = None, *, epi: int = EPI_PLAIN,
         residual: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
         rstd: Optional[torch.Tensor] = None, norm_from_x: bool = False, eps: float = 1e-5, act_gelu: bool = False,
         out_fp32: bool = False, bn: int = 0, splitk: int = 0,
         q_out=None, k_cache=None, v_cache=None, positions=None, slots=None, n_q_heads: int = 0,
         n_kv_heads: int = 0, head_dim: int = 0, rope_theta: float = 0.0, q_scale: float = 1.0,
         out_ptr: int = 0, ld_out: int = 0, residual_ptr: int = 0, ld_res: int = 0,
         wait_flag: int = 0, wait_epoch: int = 0, signal_flag: int = 0, signal_epoch: int = 0,
         done_counter: int = 0, free_flag: int = 0, bump_epoch: int = 0, ack_flag: int = 0,
         dbg: int = 0, w_scale: Optional[torch.Tensor] = None,
         sfa: Optional[torch.Tensor] = None, sfb: Optional[torch.Tensor] = None,
         stages: int = -1, free_lag: int = 0, out2_ptr: int = 0,
         fq_out: Optional[torch.Tensor] = None, fq_sf: Optional[torch.Tensor] = None, fq_bn: int = 0,
         sumsq_out: Optional[torch.Tensor] = None, zero_buf: Optional[torch.Tensor] = None,
         sumsq: Optional[torch.Tensor] = None, no_out: bool = False) -> Optional[torch.Tensor]:
    """out[t, n] = epilogue(sum_k x[t, k] * w[n, k]) on the tcgen05 swap-AB kernel."""
    m_tok, k = x.shape
    n_out = w.shape[0]
    if bn <= 0:
        if sfa is not None:
            bn = pick_bn_mx(m_tok)
        elif m_tok > 64:
            bn, st, sk_hint = pick_prefill_tile(n_out, m_tok, k)
            if stages < 0:
                stages = st
            if splitk <= 0 and sk_hint > 0:
                splitk = sk_hint
                cap = native().gemm_max_splitk(bn, epi, max(stages, 0))      # reduce-scatter landing zone must fit the ring
                while splitk > cap:
                    splitk //= 2
        else:
            bn = pick_bn(m_tok)
    if stages < 0:
        stages = 0
    if splitk <= 0:
        splitk = pick_splitk(n_out, m_tok, k, bn, epi, stages)
    if epi == EPI_QKV_ROPE or (no_out and fq_out is not None):
        o_ptr, ldo = 0, 0          # no bf16 output: QKV writes q / KV cache; a GLU whose only consumer reads the fused e4m3 copy
    elif out_ptr:
        o_ptr, ldo = out_ptr, ld_out
    else:
        if out is None:
            width = n_out // 2 if epi == EPI_GLU else n_out
            out = torch.empty((m_tok, width), device=x.device, dtype=torch.float32 if out_fp32 else torch.bfloat16)
        o_ptr, ldo = out.data_ptr(), out.stride(0)
    if residual is not None:
        residual_ptr, ld_res = residual.data_ptr(), residual.stride(0)
    if TIMELINE is not None and not dbg:
        # per-CTA %globaltimer stamps (tools/layer_timeline.py): every GEMM call gets its own slice of the buffer
        n_cta = (n_out // 128) * ((m_tok + bn - 1) // bn) * splitk
        dbg = TIMELINE["buf"].data_ptr() + TIMELINE["off"] * 8
        TIMELINE["log"].append((epi, n_out, k, splitk, TIMELINE["off"], n_cta))
        TIMELINE["off"] += n_cta * 8
        assert TIMELINE["off"] <= TIMELINE["buf"].numel()
    native().gemm(w, x, o_ptr, ldo, epi, bn, splitk, residual_ptr, ld_res, bias, rstd, norm_from_x, eps, act_gelu,
                  out_fp32, q_out, k_cache, v_cache, positions, slots, n_q_heads, n_kv_heads, head_dim, rope_theta,
                  q_scale, wait_flag, wait_epoch, signal_flag, signal_epoch, done_counter, free_flag, bump_epoch,
                  ack_flag, dbg, w_scale, sfa, sfb, stages, free_lag, out2_ptr,
                  _ptr(fq_out), _ptr(fq_sf), fq_out.shape[1] if fq_out is not None else 0, fq_bn, _ptr(sumsq_out), _ptr(zero_buf),
                  _ptr(sumsq))
    return out


# ------------------------------------------------------------------------- fp8
def quantize_weight_fp8(w: torch.Tensor):
    """[N, K] -> (e4m3 weights, fp32 per-row scale).  W ~= q * scale[:, None]."""
    amax = w.float().abs().amax(dim=1).clamp_min(1e-12)
    scale = (amax / 448.0).float()
    q = (w.float() / scale[:, None]).clamp(-448, 448).to(torch.float8_e4m3fn)
    return q.contiguous(), scale.contiguous()


def quant_fp8_rows(x: torch.Tensor, eps: float = 1e-5, with_rms: bool = False, out=None, scale_out=None):
    """Per-token dynamic e4m3 quantisation of a GEMM input; returns (q, scale) where scale already
    contains 1/rms when ``with_rms`` (RMSNorm fused with gamma folded into the fp8 weights)."""
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.float8_e4m3fn)
    if scale_out is None:
        scale_out = torch.empty(x.shape[0], device=x.device, dtype=torch.float32)
    native().quant_fp8_rows(x, out, scale_out, eps, with_rms)
    return out, scale_out


# ------------------------------------------------------- MX (block-scaled) fp8
MX_BLOCK = 32          # K elements per UE8M0 scale (OCP MX / tcgen05 kind::mxf8f6f4.block_scale)


def pick_bn_mx(m_tok: int) -> int:
    """token tile of an MX GEMM: the scale-factor chunks are laid out per tile of >= 32 rows"""
    return max(32, pick_bn(m_tok))


def mx_chunk_layout(sf: torch.Tensor, rows_per_tile: int = 128) -> torch.Tensor:
    """[R, K/32] scale bytes (R multiple of 128, K multiple of 128) -> the tcgen05.cp chunk layout
    [R/128][K/128][32 (r % 32)][4 (r / 32)][4 (k-block in chunk)] flattened (512 bytes per chunk)."""
    R, nb = sf.shape
    assert R % 128 == 0 and nb % 4 == 0
    v = sf.view(R // 128, 4, 32, nb // 4, 4)              # tile, r/32, r%32, kchunk, j
    return v.permute(0, 3, 2, 1, 4).contiguous().view(-1)


def quantize_weight_mxfp8(w: torch.Tensor):
    """[N, K] -> (e4m3 weights, UE8M0 scale factors in chunk layout).  W ~= q * 2^(sf - 127) per 32-K block."""
    N, K = w.shape
    assert N % 128 == 0 and K % 128 == 0, "MX weights: N and K must be multiples of 128"
    blocks = w.float().view(N, K // MX_BLOCK, MX_BLOCK)
    amax = blocks.abs().amax(dim=2)
    mant, ex = torch.frexp(amax / 448.0)                   # amax/448 = mant * 2^ex, mant in [0.5, 1)
    e = torch.where(mant > 0.5, ex, ex - 1).clamp(-126, 127)
    e = torch.where(amax > 0, e, torch.full_like(e, -126))
    q = (blocks * torch.exp2(-e.float())[:, :, None]).clamp(-448, 448).view(N, K).to(torch.float8_e4m3fn)
    sf = (e + 127).to(torch.uint8)
    return q.contiguous(), mx_chunk_layout(sf)


def mx_dequant(q: torch.Tensor, sf_plain: torch.Tensor) -> torch.Tensor:
    """reference helper: q [R, K] e4m3, sf_plain [R, K/32] uint8 -> fp32"""
    R, K = q.shape
    return (q.float().view(R, K // MX_BLOCK, MX_BLOCK) * torch.exp2(sf_plain.float() - 127.0)[:, :, None]).view(R, K)


def mx_unchunk(sf_chunks: torch.Tensor, rows: int, K: int, bn: int = 128) -> torch.Tensor:
    """inverse of the chunk layout for activations quantised with token tile ``bn``: -> [rows, K/32] uint8"""
    nkc = K // 128
    chunk = 1024 if bn > 128 else 512
    tiles = (rows + bn - 1) // bn
    v = sf_chunks[: tiles * nkc * chunk].view(tiles, nkc, chunk // 512, 32, 4, 4)      # tile, kc, half, r%32, r/32, j
    v = v.permute(0, 2, 4, 3, 1, 5).contiguous().view(tiles, (chunk // 512) * 128, nkc * 4)   # tile, row in padded tile, kblock
    return v[:, :bn].reshape(tiles * bn, nkc * 4)[:rows]


def quant_mxfp8_rows(x: torch.Tensor, bn: int = 0, eps: float = 1e-5, with_rms: bool = False, out=None, sf_out=None,
                     sumsq_out=None):
    """Dynamic MX quantisation of GEMM activations (optionally fused with the RMSNorm 1/rms scale);
    returns (q, sf_chunks) for a GEMM whose token tile is ``bn`` (default: what ``gemm`` would pick)."""
    T, K = x.shape
    if bn <= 0:
        bn = pick_bn_mx(T)
    tiles = (T + bn - 1) // bn
    if out is None:
        out = torch.empty((T, K), device=x.device, dtype=torch.float8_e4m3fn)
    if sf_out is None:
        sf_out = torch.empty(tiles * (K // 128) * (1024 if bn > 128 else 512), device=x.device, dtype=torch.uint8)
    # sumsq_out: quantise the raw values and hand the row's sum of squares to the consuming GEMM (mode 2)
    native().quant_mxfp8_rows(x, out, sf_out, bn, eps, 2 if sumsq_out is not None else int(bool(with_rms)), sumsq_out)
    return out, sf_out


# ----------------------------------------------------------------- elementwise
def rmsnorm(x, gamma, out=None, residual=None, eps=1e-5, plus_one=False, rstd_out=None, want_out=True):
    if out is None and want_out:
        out = torch.empty_like(x)
    native().rmsnorm(x, gamma, residual, out, rstd_out, eps, plus_one)
    return out


def rstd(x, eps=1e-5):
    """per-token 1/rms (fp32) for GEMMs whose RMSNorm is fused but whose token tile is large"""
    r = torch.empty(x.shape[0], device=x.device, dtype=torch.float32)
    native().rmsnorm(x, x, None, None, r, eps, False)
    return r


def layernorm(x, gamma, beta, out=None, eps=1e-5):
    if out is None:
        out = torch.empty_like(x)
    native().layernorm(x, gamma, beta, out, eps)
    return out


def embed(ids, table, out, pos_table=None, positions=None, scale=1.0, tok_flag=0, tok_epoch=0, pf_flag=0, pf_need=0):
    native().embed(ids.data_ptr() if isinstance(ids, torch.Tensor) else int(ids), table, pos_table, positions, out,
                   scale, tok_flag, tok_epoch, pf_flag, pf_need)
    return out


def kv_append(qkv, q_out, k_cache, v_cache, slots, q_dim, kv_dim, q_scale):
    native().kv_append(qkv, q_out, k_cache, v_cache, slots, q_dim, kv_dim, q_scale)


def add(a, b, out=None):
    if out is None:
        out = torch.empty_like(a)
    native().add(a, b, out)
    return out


# -------------------------------------------------------------------- attention
def attention(q, k_cache, v_cache, out, block_table, q_start, q_len, kv_len, *, max_q, n_q, n_kv, head_dim,
              window=0, softcap=0.0, splits=1, ws=None, use_tc=-1, fq_out=None, fq_sf=None, fq_bn=0):
    """Paged-KV attention.  Prefill chunks (max_q >= 2) run on the tcgen05 flash kernel.  Decode (max_q == 1) also does
    when the batch fills the machine (sequences x kv heads >= 128 CTAs) or no split-KV was asked for: measured on B200
    (profiles/decode_attention.md) it streams the KV pages at 0.66 of the HBM peak at 8k context against 0.49 for the
    CUDA-core split-KV kernel, and is faster even at 64 tokens (7.9 vs 10.1 us); few sequences with a long context
    keep the split-KV kernel (more CTAs than (sequence, kv head) pairs)."""
    if use_tc < 0 and max_q == 1:
        # split-KV (few sequences x long context) also runs on the tensor-core kernel: every (sequence, kv head, split) CTA
        # streams its share of the pages, the shared merge pass combines the partials
        use_tc = 1
    native().attention(q, k_cache, v_cache, out, block_table, q_start, q_len, kv_len, ws, max_q, n_q, n_kv, head_dim,
                       window, softcap, splits, use_tc, _ptr(fq_out), _ptr(fq_sf), fq_bn)
    if splits > 1:
        LAUNCHES[0] += 1           # split-KV: the merge pass is a second kernel
    return out


def attention_fuses_quant(max_q: int, n_q: int, n_kv: int, head_dim: int, splits: int) -> bool:
    """True when ``attention`` will run the tcgen05 kernel without split-KV, i.e. can emit the e4m3 copy itself."""
    g = n_q // max(1, n_kv)
    tc_ok = n_kv > 0 and n_q % n_kv == 0 and g in (1, 2, 4, 8, 16) and head_dim in (64, 128, 256) and get_attn_tc_min_q() > 0
    if not tc_ok:
        return False
    return (max_q == 1 and splits <= 1) or (max_q > 1 and max_q >= get_attn_tc_min_q())


def set_attn_tc_min_q(n: int) -> None:
    """Query-chunk length from which prefill attention runs on the tcgen05 kernel (0 = scalar kernel only)."""
    native().set_attn_tc_min_q(int(n))


def get_attn_tc_min_q() -> int:
    return int(native().get_attn_tc_min_q())


# ---------------------------------------------------------------------- sampler
def sample(logits, out_tokens, *, seen=None, temperature=None, top_p=None, rep_penalty=None, seeds=None, step=None,
           peer_tokens=0, history=0, hist_pos=None, hist_stride=0, signal_flag=0, signal_epoch=0, done_counter=0,
           vocab=0, softcap=0.0, row_map=0):
    """``row_map``: device address of int32 [rows of logits] mapping each logits row to its batch row (< 0 = skip)."""
    native().sample(logits, seen, out_tokens, peer_tokens, history, hist_pos, hist_stride, vocab, softcap,
                    temperature, top_p,
                    rep_penalty, seeds, step, signal_flag, signal_epoch, done_counter, row_map)
    return out_tokens


def mark_seen(ids, seq_of, seen, vocab):
    native().mark_seen(ids, seq_of, seen, vocab)
