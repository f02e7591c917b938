"""Numerics of every hand-written sm_100a kernel against a plain PyTorch fp32 reference."""
import math

import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from bee2bee_b200 import ops  # noqa: E402
from bee2bee_b200.models import torch_ref  # noqa: E402


def dev():
    return torch.device("cuda:0")


def bf(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed + sum(shape))
    return (torch.randn(*shape, device="cuda", generator=g) * scale).to(torch.bfloat16)


def close(a, b, rtol=2e-2, atol=2e-2):
    a, b = a.float(), b.float()
    err = (a - b).abs().max().item()
    ref = b.abs().max().item()
    assert torch.isfinite(a).all(), "non-finite output"
    assert err <= atol + rtol * ref, f"max err {err} vs ref scale {ref}"


# ----------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("m,n,k", [(1, 256, 128), (5, 384, 256), (16, 256, 4096), (32, 512, 1024), (33, 256, 512),
                                   (100, 256, 256), (300, 384, 512), (600, 256, 192)])
def test_gemm_plain(m, n, k):
    w, x = bf(n, k, scale=0.05), bf(m, k)
    out = ops.gemm(w, x, splitk=1)
    close(out, x.float() @ w.float().t())


@pytest.mark.parametrize("bn", [16, 32, 64, 128, 256])
def test_gemm_all_token_tiles(bn):
    m = bn - 3
    w, x = bf(256, 512, scale=0.05), bf(m, 512)
    close(ops.gemm(w, x, bn=bn, splitk=1), x.float() @ w.float().t())


@pytest.mark.parametrize("splitk", [2, 3, 4, 8])
@pytest.mark.parametrize("m", [1, 16, 31])
def test_gemm_splitk_cluster(splitk, m):
    w, x = bf(384, 2048, scale=0.05), bf(m, 2048)
    close(ops.gemm(w, x, splitk=splitk), x.float() @ w.float().t())       # cluster / DSMEM kernel


@pytest.mark.parametrize("bn,splitk,stages",
                         [(256, 2, 0), (256, 4, 0), (128, 2, 3), (128, 4, 3), (128, 2, 0), (256, 1, 0), (128, 1, 0)])
@pytest.mark.parametrize("m", [256, 300, 512])
def test_gemm_prefill_splitk_tiles(bn, splitk, stages, m):
    """the (token tile, split-K, ring depth) combinations ops.pick_prefill_tile emits for under-filled prefill GEMMs:
    cluster split-K with the DSMEM reduce-scatter on 128 / 256-wide token tiles, and the same tiles without split-K;
    plain and residual epilogues, ragged last token tile"""
    w, x, r = bf(512, 4096, scale=0.03), bf(m, 4096), bf(m, 512)
    ref = x.float() @ w.float().t()
    close(ops.gemm(w, x, bn=bn, splitk=splitk, stages=stages), ref)
    out = ops.gemm(w, x, bn=bn, splitk=splitk, stages=stages, epi=ops.EPI_RESIDUAL, residual=r)
    close(out, ref + r.float())
    # ... and through the heuristic itself (long K -> 256-wide tiles + split-K)
    w2, x2 = bf(256, 8192, scale=0.02), bf(m, 8192)
    close(ops.gemm(w2, x2), x2.float() @ w2.float().t())


def test_gemm_fp32_out_and_bias():
    w, x = bf(256, 256, scale=0.05), bf(7, 256)
    bias = torch.randn(256, device="cuda")
    out = ops.gemm(w, x, bias=bias, out_fp32=True)
    assert out.dtype == torch.float32
    close(out, x.float() @ w.float().t() + bias, rtol=5e-3, atol=5e-3)


@pytest.mark.parametrize("splitk", [1, 4])
def test_gemm_residual(splitk):
    w, x, r = bf(256, 1024, scale=0.05), bf(9, 1024), bf(9, 256)
    out = ops.gemm(w, x, epi=ops.EPI_RESIDUAL, residual=r, splitk=splitk)
    close(out, x.float() @ w.float().t() + r.float())


def test_gemm_gelu_bias():
    w, x = bf(256, 256, scale=0.05), bf(12, 256)
    bias = torch.randn(256, device="cuda") * 0.1
    out = ops.gemm(w, x, epi=ops.EPI_GELU, bias=bias)
    close(out, torch_ref.gelu_tanh(x.float() @ w.float().t() + bias))


@pytest.mark.parametrize("gelu", [False, True])
@pytest.mark.parametrize("m,splitk", [(1, 1), (20, 2), (70, 1)])
def test_gemm_glu(gelu, m, splitk):
    f, h = 256, 512
    wg, wu, x = bf(f, h, scale=0.05, seed=1), bf(f, h, scale=0.05, seed=2), bf(m, h)
    w = ops.glu_interleave_rows(wg, wu)
    out = ops.gemm(w, x, epi=ops.EPI_GLU, act_gelu=gelu, splitk=splitk)
    g = x.float() @ wg.float().t()
    act = torch_ref.gelu_tanh(g) if gelu else torch.nn.functional.silu(g)
    close(out, act * (x.float() @ wu.float().t()))


@pytest.mark.parametrize("inline", [True, False])
def test_gemm_fused_rmsnorm(inline):
    h, n, m = 512, 256, 10
    w, x, gamma = bf(n, h, scale=0.05), bf(m, h, scale=3.0), (1 + 0.1 * torch.randn(h, device="cuda")).to(torch.bfloat16)
    wf = ops.fold_gamma(w, gamma)
    if inline:
        out = ops.gemm(wf, x, norm_from_x=True, eps=1e-5)
    else:
        out = ops.gemm(wf, x, rstd=ops.rstd(x, 1e-5))
    ref = torch_ref.rms_norm(x.float(), gamma.float(), 1e-5, False) @ w.float().t()
    close(out, ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("hd,nq,nkv", [(128, 4, 2), (256, 2, 1), (64, 4, 4)])
def test_gemm_qkv_rope_append(hd, nq, nkv):
    h, m, theta = 256, 6, 10000.0
    wq, wk, wv = bf(nq * hd, h, scale=0.05, seed=1), bf(nkv * hd, h, scale=0.05, seed=2), bf(nkv * hd, h, scale=0.05, seed=3)
    x = bf(m, h)
    w = torch.cat([ops.rope_interleave_rows(wq, nq, hd), ops.rope_interleave_rows(wk, nkv, hd), wv], 0).contiguous()
    pages = 4
    kc = torch.zeros(pages, ops.PAGE, nkv, hd, device="cuda", dtype=torch.bfloat16)
    vc = torch.zeros_like(kc)
    q_out = torch.zeros(m, nq * hd, device="cuda", dtype=torch.bfloat16)
    pos = torch.tensor([0, 1, 2, 70, 71, 500], device="cuda", dtype=torch.int32)
    slots = torch.tensor([5, 6, 64, 130, -1, 200], device="cuda", dtype=torch.int32)
    scale = 0.25
    ops.gemm(w, x, epi=ops.EPI_QKV_ROPE, q_out=q_out, k_cache=kc, v_cache=vc, positions=pos, slots=slots,
             n_q_heads=nq, n_kv_heads=nkv, head_dim=hd, rope_theta=theta, q_scale=scale)
    torch.cuda.synchronize()
    xf = x.float()
    q = torch_ref.rope((xf @ wq.float().t()).view(1, m, nq, hd), pos.long()[None], theta)[0] * scale
    k = torch_ref.rope((xf @ wk.float().t()).view(1, m, nkv, hd), pos.long()[None], theta)[0]
    v = (xf @ wv.float().t()).view(m, nkv, hd)
    half = hd // 2
    perm = torch.arange(hd, device="cuda").view(2, half).t().reshape(-1)     # kernel layout: interleaved pairs
    close(q_out.view(m, nq, hd), q[:, :, perm])
    kflat, vflat = kc.view(-1, nkv, hd), vc.view(-1, nkv, hd)
    for i, s in enumerate(slots.tolist()):
        if s < 0:
            continue
        close(kflat[s], k[i][:, perm])
        close(vflat[s], v[i])
    assert kflat[131].abs().sum() == 0   # the slot of the masked token stays untouched


# ----------------------------------------------------------------- elementwise
def test_rmsnorm_and_rstd():
    x, g, r = bf(17, 512, scale=2.0), bf(512), bf(17, 512)
    close(ops.rmsnorm(x, g, eps=1e-6), torch_ref.rms_norm(x.float(), g.float(), 1e-6, False))
    close(ops.rmsnorm(x, g, eps=1e-6, plus_one=True, residual=r),
          torch_ref.rms_norm(x.float(), g.float(), 1e-6, True) + r.float())
    ref = torch.rsqrt(x.float().pow(2).mean(-1) + 1e-6)
    close(ops.rstd(x, 1e-6), ref, rtol=1e-4, atol=1e-5)


def test_layernorm():
    x, g, b = bf(9, 768, scale=2.0), bf(768), bf(768)
    close(ops.layernorm(x, g, b, eps=1e-5), torch_ref.layer_norm(x.float(), g.float(), b.float(), 1e-5))


def test_embed_scale_and_positions():
    table, ptab = bf(100, 256), bf(64, 256)
    ids = torch.tensor([3, 99, 0, 7], device="cuda", dtype=torch.int32)
    pos = torch.tensor([0, 5, 63, 1], device="cuda", dtype=torch.int32)
    out = torch.empty(4, 256, device="cuda", dtype=torch.bfloat16)
    ops.embed(ids, table, out)
    assert torch.equal(out, table[ids.long()])
    ops.embed(ids, table, out, pos_table=ptab, positions=pos)
    close(out, table[ids.long()].float() + ptab[pos.long()].float(), rtol=1e-2, atol=1e-2)
    ops.embed(ids, table, out, scale=16.0)
    close(out, table[ids.long()].float() * 16.0, rtol=1e-2, atol=1e-2)


def test_decode_advance():
    n, mp = 5, 4
    bt = torch.arange(n * mp, device="cuda", dtype=torch.int32).view(n, mp)
    pos = torch.tensor([0, 62, 63, 64, 10], device="cuda", dtype=torch.int32)
    kv = pos + 1
    q_len = torch.tensor([1, 1, 1, 1, 0], device="cuda", dtype=torch.int32)
    slots = torch.zeros(n, device="cuda", dtype=torch.int32)
    ops.native().decode_advance(pos, kv, slots, q_len, bt)
    assert pos.tolist() == [1, 63, 64, 65, 10]
    assert kv.tolist() == [2, 64, 65, 66, 11]
    assert slots.tolist() == [0 * 64 + 1, 4 * 64 + 63, 9 * 64 + 0, 13 * 64 + 1, -1]


# ------------------------------------------------------------------- attention
def _paged_setup(seq_lens, nkv, hd, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    max_pages = max((l + ops.PAGE - 1) // ops.PAGE for l in seq_lens) + 1
    total_pages = len(seq_lens) * max_pages + 1
    kc = (torch.randn(total_pages, ops.PAGE, nkv, hd, device="cuda", generator=g)).to(torch.bfloat16)
    vc = (torch.randn(total_pages, ops.PAGE, nkv, hd, device="cuda", generator=g)).to(torch.bfloat16)
    perm = torch.randperm(total_pages - 1, device="cuda", generator=g).int() + 1
    bt = perm[: len(seq_lens) * max_pages].view(len(seq_lens), max_pages).contiguous()
    return kc, vc, bt


def _attn_ref(q, kc, vc, bt, q_lens, kv_lens, nq, nkv, hd, window, softcap):
    outs = []
    off = 0
    for s, (ql, kl) in enumerate(zip(q_lens, kv_lens)):
        if ql == 0:
            continue
        pages = bt[s].long()
        k = kc[pages].reshape(-1, nkv, hd)[:kl].float()
        v = vc[pages].reshape(-1, nkv, hd)[:kl].float()
        qq = q[off:off + ql].float().view(ql, nkv, nq // nkv, hd)
        sc = torch.einsum("tkgd,skd->kgts", qq, k)
        if softcap > 0:
            sc = torch.tanh(sc / softcap) * softcap
        qpos = torch.arange(kl - ql, kl, device=q.device)[:, None]
        kpos = torch.arange(kl, device=q.device)[None, :]
        ok = kpos <= qpos
        if window > 0:
            ok = ok & (kpos > qpos - window)
        sc = sc.masked_fill(~ok[None, None], float("-inf"))
        o = torch.einsum("kgts,skd->tkgd", sc.softmax(-1), v).reshape(ql, nq * hd)
        outs.append(o)
        off += ql
    return torch.cat(outs, 0)


@pytest.mark.parametrize("hd,nq,nkv", [(128, 8, 2), (64, 4, 4), (256, 4, 2), (128, 32, 8)])
@pytest.mark.parametrize("window,softcap", [(0, 0.0), (100, 50.0)])
@pytest.mark.parametrize("use_tc", [1, 0])
def test_attention_decode(hd, nq, nkv, window, softcap, use_tc):
    """decode (one query token per sequence) on the tcgen05 flash kernel (one-token query blocks, the default) and on
    the CUDA-core kernel; an inactive batch row (q_len 0) must be left alone by both"""
    kv_lens = [1, 63, 64, 65, 300, 17, 1000]
    S = len(kv_lens)
    kc, vc, bt = _paged_setup(kv_lens, nkv, hd)
    q = bf(S, nq * hd, scale=0.3)
    out = torch.zeros_like(q)
    ar = torch.arange(S, device="cuda", dtype=torch.int32)
    ones = torch.ones(S, device="cuda", dtype=torch.int32)
    ones[3] = 0                                     # inactive slot
    kvl = torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    ops.attention(q, kc, vc, out, bt, ar, ones, kvl, max_q=1, n_q=nq, n_kv=nkv, head_dim=hd, window=window,
                  softcap=softcap, use_tc=use_tc)
    ref = _attn_ref(q, kc, vc, bt, [1] * S, kv_lens, nq, nkv, hd, window, softcap)
    keep = [i for i in range(S) if i != 3]
    close(out[keep], ref[keep])
    assert float(out[3].abs().max()) == 0.0


@pytest.mark.parametrize("splits", [2, 5, 16])
@pytest.mark.parametrize("use_tc", [1, 0])
@pytest.mark.parametrize("hd,nq,nkv", [(128, 8, 2), (256, 8, 4)])
def test_attention_decode_split_kv(splits, use_tc, hd, nq, nkv):
    """split-KV decode: (sequence, kv head, split) CTAs + merge pass, on the tcgen05 kernel and the CUDA-core kernel;
    splits with no tiles at all (short sequences) publish empty partials"""
    kv_lens = [1000, 130, 64, 5]
    S = len(kv_lens)
    kc, vc, bt = _paged_setup(kv_lens, nkv, hd)
    q = bf(S, nq * hd, scale=0.3)
    out = torch.zeros_like(q)
    ws = torch.zeros(S * nkv * splits * 4 * (hd + 2), device="cuda")
    ar = torch.arange(S, device="cuda", dtype=torch.int32)
    ones = torch.ones(S, device="cuda", dtype=torch.int32)
    kvl = torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    ops.attention(q, kc, vc, out, bt, ar, ones, kvl, max_q=1, n_q=nq, n_kv=nkv, head_dim=hd, splits=splits, ws=ws,
                  use_tc=use_tc)
    close(out, _attn_ref(q, kc, vc, bt, [1] * S, kv_lens, nq, nkv, hd, 0, 0.0))


@pytest.mark.parametrize("hd,nq,nkv", [(128, 8, 2), (64, 2, 2), (256, 2, 1)])
@pytest.mark.parametrize("window", [0, 50])
def test_attention_prefill(hd, nq, nkv, window):
    q_lens = [70, 1, 33, 16]
    kv_lens = [70, 9, 100, 16]          # sequences 1 and 2 have cached context
    kc, vc, bt = _paged_setup(kv_lens, nkv, hd)
    T = sum(q_lens)
    q = bf(T, nq * hd, scale=0.3)
    out = torch.zeros_like(q)
    qs = torch.tensor([0, 70, 71, 104], device="cuda", dtype=torch.int32)
    ql = torch.tensor(q_lens, device="cuda", dtype=torch.int32)
    kvl = torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    ops.attention(q, kc, vc, out, bt, qs, ql, kvl, max_q=max(q_lens), n_q=nq, n_kv=nkv, head_dim=hd, window=window)
    close(out, _attn_ref(q, kc, vc, bt, q_lens, kv_lens, nq, nkv, hd, window, 0.0))


def test_attention_prefill_scalar_fallback_kernel():
    """The CUDA-core kernel (used for short chunks / unsupported head layouts) stays correct."""
    hd, nq, nkv = 128, 8, 2
    q_lens, kv_lens = [70, 1, 33, 16], [70, 9, 100, 16]
    kc, vc, bt = _paged_setup(kv_lens, nkv, hd)
    q = bf(sum(q_lens), nq * hd, scale=0.3)
    out = torch.zeros_like(q)
    qs = torch.tensor([0, 70, 71, 104], device="cuda", dtype=torch.int32)
    ql = torch.tensor(q_lens, device="cuda", dtype=torch.int32)
    kvl = torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    old = ops.get_attn_tc_min_q()
    ops.set_attn_tc_min_q(0)
    try:
        ops.attention(q, kc, vc, out, bt, qs, ql, kvl, max_q=max(q_lens), n_q=nq, n_kv=nkv, head_dim=hd)
    finally:
        ops.set_attn_tc_min_q(old)
    close(out, _attn_ref(q, kc, vc, bt, q_lens, kv_lens, nq, nkv, hd, 0, 0.0))


@pytest.mark.parametrize("hd,nq,nkv,window,softcap", [
    (128, 32, 8, 0, 0.0),        # Llama-3 / Mistral head layout
    (128, 32, 8, 300, 0.0),      # sliding window (Mistral / Gemma-2 local layers)
    (256, 8, 4, 0, 50.0),        # Gemma-2: d=256, soft-capping
    (64, 12, 12, 0, 0.0),        # GPT-2: MHA, d=64
])
def test_attention_prefill_tcgen05_long(hd, nq, nkv, window, softcap):
    """tcgen05 flash-attention prefill: long prompts, chunked prefill on top of cached context, ragged batch."""
    q_lens = [1000, 257, 640]
    kv_lens = [1000, 900, 640]         # sequence 1 is a second chunk on top of 643 cached tokens
    kc, vc, bt = _paged_setup(kv_lens, nkv, hd)
    q = bf(sum(q_lens), nq * hd, scale=0.3)
    out = torch.zeros_like(q)
    qs = torch.tensor([0, 1000, 1257], device="cuda", dtype=torch.int32)
    ql = torch.tensor(q_lens, device="cuda", dtype=torch.int32)
    kvl = torch.tensor(kv_lens, device="cuda", dtype=torch.int32)
    assert ops.get_attn_tc_min_q() > 0
    ops.attention(q, kc, vc, out, bt, qs, ql, kvl, max_q=max(q_lens), n_q=nq, n_kv=nkv, head_dim=hd, window=window,
                  softcap=softcap)
    close(out, _attn_ref(q, kc, vc, bt, q_lens, kv_lens, nq, nkv, hd, window, softcap))


# --------------------------------------------------------------------- sampler
def test_sampler_greedy_and_penalty():
    B, V = 4, 1000
    logits = torch.randn(B, V, device="cuda") * 3
    out = torch.zeros(B, device="cuda", dtype=torch.int32)
    ops.sample(logits, out)
    assert out.tolist() == logits.argmax(-1).tolist()
    # repetition penalty on the arg-max pushes greedy to the runner-up when the margin is small
    seen = torch.zeros(B, (V + 31) // 32, device="cuda", dtype=torch.int32)
    top = logits.argmax(-1)
    ops.mark_seen(top.int(), torch.arange(B, device="cuda", dtype=torch.int32), seen, V)
    pen = torch.full((B,), 100.0, device="cuda")
    temp = torch.zeros(B, device="cuda")
    ops.sample(logits, out, seen=seen, rep_penalty=pen, temperature=temp)
    seen_bool = torch.zeros(B, V, dtype=torch.bool, device="cuda")
    seen_bool[torch.arange(B), top] = True
    ref = torch_ref.sample_reference(logits, seen_bool, 0.0, 1.0, 100.0)
    assert out.tolist() == ref.tolist()
    # sampled ids were recorded in the bitmap
    for b in range(B):
        t = out[b].item()
        assert (seen[b, t // 32].item() >> (t % 32)) & 1


@pytest.mark.parametrize("V", [1000, 50257, 128256])
def test_sampler_top_p_stays_in_nucleus_and_matches_distribution(V):
    B = 8
    torch.manual_seed(0)
    logits = torch.randn(B, V, device="cuda") * 4
    temp, top_p = 0.7, 0.95
    keep = torch_ref.top_p_keep_mask(logits, temp, top_p)
    out = torch.zeros(B, device="cuda", dtype=torch.int32)
    t = torch.full((B,), temp, device="cuda")
    p = torch.full((B,), top_p, device="cuda")
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    counts = torch.zeros(V, device="cuda")
    n_draws = 300
    for i in range(n_draws):
        step.fill_(i)
        seeds = torch.full((B,), 1234 + i, device="cuda", dtype=torch.int32)
        ops.sample(logits, out, temperature=t, top_p=p, seeds=seeds, step=step)
        assert keep[torch.arange(B), out.long()].all(), "sampled outside the nucleus"
        counts[out[0].long()] += 1
    # row 0: empirical frequency of its most likely token ~ renormalised probability
    pr = (logits[0] / temp).softmax(-1) * keep[0]
    pr = pr / pr.sum()
    top = pr.argmax()
    assert abs(counts[top].item() / n_draws - pr[top].item()) < 0.12


def test_sampler_padded_vocab_and_softcap():
    B, V, ld = 3, 500, 512
    buf = torch.full((B, ld), 1e9, device="cuda")     # padding columns hold junk that must be ignored
    buf[:, :V] = torch.randn(B, V, device="cuda") * 40
    out = torch.zeros(B, device="cuda", dtype=torch.int32)
    ops.sample(buf, out, vocab=V, softcap=30.0)
    capped = torch.tanh(buf[:, :V] / 30.0) * 30.0
    assert out.tolist() == capped.argmax(-1).tolist()


# ------------------------------------------------------------------------- fp8
@pytest.mark.parametrize("m,n,k,splitk", [(1, 256, 512, 1), (20, 384, 1024, 2), (64, 256, 256, 1), (200, 256, 384, 1)])
def test_gemm_fp8_w8a8(m, n, k, splitk):
    w, x = bf(n, k, scale=0.05), bf(m, k, scale=2.0)
    wq, ws = ops.quantize_weight_fp8(w)
    xq, xs = ops.quant_fp8_rows(x)
    # quantiser: dequantised values reproduce the input to e4m3 precision, scale = amax / 448
    close(xq.float() * xs[:, None], x, rtol=7e-2, atol=0.0)
    assert torch.allclose(xs, x.float().abs().amax(1) / 448, rtol=1e-3)
    out = ops.gemm(wq, xq, rstd=xs, w_scale=ws, splitk=splitk)
    ref_q = (xq.float() * xs[:, None]) @ (wq.float() * ws[:, None]).t()      # exact math on the quantised operands
    close(out, ref_q, rtol=1e-2, atol=1e-2)
    close(out, x.float() @ w.float().t(), rtol=6e-2, atol=6e-2)              # and close to the bf16 result


@pytest.mark.parametrize("m,n,k,splitk,bn", [(1, 256, 256, 1, 0), (33, 256, 512, 1, 0), (128, 256, 384, 1, 0),
                                              (200, 384, 1024, 2, 0), (300, 256, 512, 1, 256)])
def test_gemm_mxfp8_block_scaled(m, n, k, splitk, bn):
    """tcgen05 kind::mxf8f6f4.block_scale: e4m3 operands with one UE8M0 scale per 32 K elements (scales in TMEM)."""
    w, x = bf(n, k, scale=0.05, seed=1), bf(m, k, scale=2.0, seed=2)
    # block magnitudes spread over 2^-6..2^5 so that a wrong scale-factor address shows up as a large error
    x = (x.float() * torch.exp2(torch.randint(-6, 6, (m, k // 32), device="cuda").float()).repeat_interleave(32, 1)).to(torch.bfloat16)
    w = (w.float() * torch.exp2(torch.randint(-4, 4, (n, k // 32), device="cuda").float()).repeat_interleave(32, 1)).to(torch.bfloat16)
    wq, sfa = ops.quantize_weight_mxfp8(w)
    bn = bn or ops.pick_bn_mx(m)
    xq, sfb = ops.quant_mxfp8_rows(x, bn)
    xd = ops.mx_dequant(xq, ops.mx_unchunk(sfb, m, k, bn))
    wd = ops.mx_dequant(wq, ops.mx_unchunk(sfa, n, k, 128))
    # quantiser: per-block power-of-two scale, e4m3 rounding (3 mantissa bits; subnormals below amax * 2^-15)
    amax = x.float().view(m, k // 32, 32).abs().amax(-1).repeat_interleave(32, 1)
    assert ((xd - x.float()).abs() <= 0.0625 * x.float().abs() + 1e-3 * amax).all()
    out = ops.gemm(wq, xq, sfa=sfa, sfb=sfb, splitk=splitk, bn=bn)
    ref_q = xd @ wd.t()                                     # exact math on the quantised operands
    scale = ref_q.abs().max().item()
    assert (out.float() - ref_q).abs().max().item() <= 6e-3 * scale      # bf16 output rounding
    ref = x.float() @ w.float().t()
    assert ((out.float() - ref).norm() / ref.norm()).item() <= 0.08          # e4m3 noise vs the unquantised product


def test_gemm_mxfp8_fused_rmsnorm_glu():
    h, f, m = 512, 256, 40
    x, gamma = bf(m, h, scale=3.0), (1 + 0.1 * torch.randn(h, device="cuda")).to(torch.bfloat16)
    wg, wu = bf(f, h, scale=0.05, seed=1), bf(f, h, scale=0.05, seed=2)
    wgu = ops.fold_gamma(ops.glu_interleave_rows(wg, wu), gamma)
    q, sfa = ops.quantize_weight_mxfp8(wgu)
    xq, sfb = ops.quant_mxfp8_rows(x, eps=1e-5, with_rms=True)
    hmid = ops.gemm(q, xq, epi=ops.EPI_GLU, sfa=sfa, sfb=sfb)
    xn = x.float() * torch.rsqrt(x.float().pow(2).mean(-1, keepdim=True) + 1e-5) * gamma.float()
    ref = torch.nn.functional.silu(xn @ wg.float().t()) * (xn @ wu.float().t())
    close(hmid, ref, rtol=8e-2, atol=8e-2)


def test_gemm_fp8_fused_rmsnorm_glu_residual():
    h, f, m = 512, 256, 9
    x, gamma, res = bf(m, h, scale=3.0), (1 + 0.1 * torch.randn(h, device="cuda")).to(torch.bfloat16), bf(m, 256)
    wg, wu, wd = bf(f, h, scale=0.05, seed=1), bf(f, h, scale=0.05, seed=2), bf(256, f, scale=0.05, seed=3)
    wgu = ops.fold_gamma(ops.glu_interleave_rows(wg, wu), gamma)
    q, sc = ops.quantize_weight_fp8(wgu)
    xq, xs = ops.quant_fp8_rows(x, 1e-5, with_rms=True)
    hmid = ops.gemm(q, xq, epi=ops.EPI_GLU, rstd=xs, w_scale=sc)
    xn = torch_ref.rms_norm(x.float(), gamma.float(), 1e-5, False)
    ref_h = torch.nn.functional.silu(xn @ wg.float().t()) * (xn @ wu.float().t())
    close(hmid, ref_h, rtol=8e-2, atol=8e-2)
    dq, dsc = ops.quantize_weight_fp8(wd)
    hq, hs = ops.quant_fp8_rows(hmid)
    out = ops.gemm(dq, hq, epi=ops.EPI_RESIDUAL, residual=res, rstd=hs, w_scale=dsc)
    close(out, hmid.float() @ wd.float().t() + res.float(), rtol=8e-2, atol=8e-2)


# ------------------------------------------------------- shapes of the decode step
@pytest.mark.parametrize("m,n,k", [(1, 128, 64), (3, 256, 4096), (32, 6144, 4096), (32, 4096, 14336), (17, 28672, 1024),
                                   (64, 1024, 8192), (40, 384, 640)])
@pytest.mark.parametrize("stages", [0, 3])
def test_gemm_decode_shapes(m, n, k, stages):
    """cluster split-K kernel on the Llama decode shapes, default and shallow shared-memory ring"""
    w, x = bf(n, k, scale=0.03), bf(m, k)
    ref = x.float() @ w.float().t()
    out = ops.gemm(w, x, stages=stages)
    close(out, ref)
    assert torch.equal(out, ops.gemm(w, x, stages=stages))     # handoff counters / barriers self-reset


def test_gemm_fused_epilogues_chain():
    h, f, m = 1024, 512, 24
    x, gamma = bf(m, h, scale=2.0), (1 + 0.1 * torch.randn(h, device="cuda")).to(torch.bfloat16)
    wg, wu = bf(f, h, scale=0.05, seed=1), bf(f, h, scale=0.05, seed=2)
    wgu = ops.fold_gamma(ops.glu_interleave_rows(wg, wu), gamma)
    out = ops.gemm(wgu, x, epi=ops.EPI_GLU, norm_from_x=True, eps=1e-5)
    xn = torch_ref.rms_norm(x.float(), gamma.float(), 1e-5, False)
    close(out, torch.nn.functional.silu(xn @ wg.float().t()) * (xn @ wu.float().t()), rtol=3e-2, atol=3e-2)
    wd, res = bf(256, f, scale=0.05, seed=3), bf(m, 256)
    out2 = ops.gemm(wd, out, epi=ops.EPI_RESIDUAL, residual=res)
    close(out2, out.float() @ wd.float().t() + res.float())
    bias = torch.randn(256, device="cuda") * 0.1
    close(ops.gemm(wd, out, epi=ops.EPI_GELU, bias=bias),
          torch_ref.gelu_tanh(out.float() @ wd.float().t() + bias))


# ---------------------------------------------------------------- K12: dense layer fwd / bwd on the tcgen05 GEMM
def test_dense_layer_forward_backward_on_tensor_cores():
    """legacy split-learning layer tasks (node.py layer_forward_train / layer_backward): tile-aligned shapes run on
    the tcgen05 GEMM (bf16 operands, fp32 accumulation) and agree with the fp32 formulas."""
    from bee2bee_b200 import model as mlp

    torch.manual_seed(0)
    T, din, dout = 128, 256, 384
    W = torch.randn(din, dout, device="cuda") * 0.05
    b = torch.randn(dout, device="cuda") * 0.1
    x = torch.randn(T, din, device="cuda")
    g = torch.randn(T, dout, device="cuda")
    assert mlp._tc_ok("cuda", dout, k=din)
    for act in ("relu", "gelu", "none"):
        y, z = mlp.dense_forward_device(W, b, act, x, device="cuda")
        z_ref = x @ W + b
        close(z, z_ref, rtol=2e-2, atol=2e-2)
        gX, gW, gb = mlp.dense_backward_device(W, act, x, z_ref, g, device="cuda")
        xr, Wr = x.clone().requires_grad_(True), W.clone().requires_grad_(True)
        zr = xr @ Wr + b
        yr = torch.relu(zr) if act == "relu" else (torch.nn.functional.gelu(zr, approximate="tanh") if act == "gelu" else zr)
        yr.backward(g)
        close(gX, xr.grad, rtol=3e-2, atol=3e-2)
        close(gW, Wr.grad, rtol=3e-2, atol=1e-1)
        close(gb, g.mul((zr > 0).float()).sum(0) if act == "relu" else gb, rtol=1e-3, atol=1e-3)


def test_attention_p_in_tmem():
    """P kept in tensor memory (TS-form tcgen05.mma): the numerics script must report every case within bf16 error."""
    import re
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "attn_tc_check.py")], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    errs = [float(x) for x in re.findall(r"max_err ([0-9.]+)", out.stdout)]
    assert len(errs) >= 5 and max(errs) < 0.03, out.stdout
