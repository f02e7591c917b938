#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): decode tokens/s + p50 TTFT for Llama-3-8B (bf16,
random-init weights, synthetic 16-token prompts) split into N pieces on N B200s.

    python bench.py --gpus 1 --steps 64 --warmup 8
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # A: the unmodified reference (baseline/_ref), HFService path
    python bench.py --impl nccl ...          # B: OUR CONSTRUCTED NCCL(+cuBLAS) pipeline (baseline/nccl_pipeline.py)
    python bench.py --config 2|3|4|5 ...     # the other BASELINE.json configs (see CONFIGS below)
    python bench.py --dump-outputs DIR ...   # also save the last timed step's tokens + logits (.npy): compare two builds

ours (C): every GPU hosts one contiguous layer range ("piece"); N micro-batch groups of
`--batch` sequences travel through the pieces as a wavefront; the hop between pieces is the
fused tail-GEMM -> NVLink peer store -> flag -> head-GEMM path, no NCCL on the token path.
One "step" = one decode step of every group = N * batch new tokens (weak scaling: per-GPU
token work is fixed, the model is sliced thinner).  Timing: CUDA events on the launch
stream, barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# no network -> no checkpoints: the benchmark runs the named architecture on random-init weights ("data": "synthetic")
os.environ.setdefault("B2B_ALLOW_RANDOM_WEIGHTS", "1")

# BASELINE.json "configs" (config 1 is the CPU plumbing test: tests/test_pipeline_node.py, tools/cpu_plumbing_bench.py)
CONFIGS = {
    0: dict(),                                                                   # headline: Llama-3-8B bf16, 32 x N
    2: dict(model="llama-3-8b", dtype="bf16", batch=1, groups=1),                # batch-1 decode latency over N pieces
    3: dict(model="llama-3-8b", dtype="mxfp8", batch=32),                        # block-scaled fp8, wavefront throughput
    4: dict(model="gemma-2-2b", dtype="bf16", batch=1, prompt_len=4096, steps=128, warmup=3),   # serve-ollama shape
    5: dict(model="zephyr-7b-beta", dtype="bf16", batch=32),                     # device side of the /generate load test
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"])
    ap.add_argument("--config", type=int, default=0, choices=sorted(CONFIGS))
    ap.add_argument("--model", default=None)
    ap.add_argument("--batch", type=int, default=None, help="sequences per micro-batch group")
    ap.add_argument("--groups", type=int, default=None, help="micro-batch groups in flight (default: N)")
    ap.add_argument("--prompt-len", type=int, default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dtype", default=None, choices=["bf16", "fp8", "mxfp8"],
                    help="fp8 = W8A8 e4m3 GEMMs with per-row/per-token scales; mxfp8 = block-scaled (UE8M0 per 32 K) "
                         "tcgen05 kind::mxf8f6f4 GEMMs (secondary configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save what the last timed decode step computed as DIR/<name>.npy: "
                         "tokens.npy (the id sampled for every sequence, float64) and logits.npy (the sampler's input "
                         "for the sequences of the last micro-batch group, float32; a fixed seeded sample of vocabulary "
                         "columns, listed in logits_columns.npy, when the whole would exceed 64 MB)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs is only supported with --impl ours")
    cfg = CONFIGS[a.config]
    dflt = dict(model="llama-3-8b", dtype="bf16", batch=32, groups=0, prompt_len=16, steps=64, warmup=8)
    for k, v in dflt.items():
        if getattr(a, k) is None:
            setattr(a, k, cfg.get(k, v))
    return a


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def mark(self):
        """index of the next sample: everything from here on belongs to the timed region"""
        self.first = len(self.lines)

    def start(self):
        self.first = 0
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        region = self.lines[getattr(self, "first", 0):] or self.lines[-1:]      # (a region shorter than one period: the sample right before it)
        for ln in region:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "samples": len(sm),
                "reasons": sorted(reasons)}


def baseline_number():
    try:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            pub = json.load(f).get("published") or {}
        for v in pub.values():
            if isinstance(v, (int, float)):
                return float(v)
    except Exception:
        pass
    return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def synthetic_prompts(n, length, vocab):
    return [[(7 + 131 * i + 31 * j) % (vocab - 300) + 256 for j in range(length)] for i in range(n)]


DUMP_BYTES = 64 * 10 ** 6 - 4096        # --dump-outputs budget, with room for the .npy headers


def dump_outputs(out_dir, n_seqs, tokens=None, logits=None):
    """Write the last timed step's sampled ids of the ``n_seqs`` sequences (float64: exact for any vocabulary) and
    logits (float32) as .npy files.  Logits beyond the budget are cut to a seeded sample of vocabulary columns that is
    the same in every run of the same shape, so dumps of two builds compare element for element."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    if tokens is not None:
        np.save(os.path.join(out_dir, "tokens.npy"), np.asarray(tokens, dtype=np.float64))
    if logits is not None:
        rows, vocab = logits.shape
        keep = (DUMP_BYTES - n_seqs * 8) // (rows * 4 + 8)       # the tokens file + an 8-byte index per kept column
        if keep < vocab:
            cols = np.sort(np.random.default_rng(0).choice(vocab, size=keep, replace=False))
            np.save(os.path.join(out_dir, "logits_columns.npy"), cols.astype(np.float64))
            logits = logits[:, cols]
        np.save(os.path.join(out_dir, "logits.npy"), np.ascontiguousarray(logits, dtype=np.float32))


def gather_objects(obj, world):
    if world <= 1:
        return [obj]
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


def common_fields(args, world, total, K, W, P, extra_cfg):
    cfgd = {"model": args.model, "global_batch": total, "seq_len": P + W + K, "prompt_len": P, "pieces": world,
            "baseline_config": args.config, "weights": "random-init", "sampling": "T=0.7 top_p=0.95 rep=1.15",
            "l2": "per-step weight stream (>= 1.7 GB/GPU) exceeds the 126 MB L2; a 256 MB buffer is written before timing"}
    cfgd.update(extra_cfg)
    return cfgd


# ----------------------------------------------------------------------------- ours (C)
def run_ours(args):
    import torch

    from bee2bee_b200.engine.core import Engine, SamplingParams
    from bee2bee_b200.engine.runner import GpuRunner, SeqInit
    from bee2bee_b200.models.config import resolve_config
    from bee2bee_b200.parallel.dist import init_distributed, max_over_ranks, shutdown

    rank, world, local = init_distributed()
    if world != args.gpus and world > 1:
        args.gpus = world
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    cfg = resolve_config(args.model)
    groups = args.groups or world
    B = args.batch
    total = B * groups
    K, W = args.steps, max(3, args.warmup)
    P = args.prompt_len
    need = P + W + K + 8
    max_seq = max(1024, ((need + 63) // 64) * 64)
    pf_tokens = max(512, min(4096, P * min(total, 32)))
    eng = Engine(args.model, cfg=cfg, device=str(dev), max_batch=total, groups=groups, max_seq_len=max_seq,
                 max_prefill_tokens=pf_tokens, decode_burst=K, rank=rank, world=world, quant=args.dtype)
    runner: GpuRunner = eng.runner
    prompts = synthetic_prompts(total, P, cfg.vocab_size)

    def barrier_sync():
        torch.cuda.synchronize(dev)
        runner.mesh.barrier()

    # ---------------- kernel-path measurement: prefill once, then W + K device-side decode steps
    ppseq = (need + 63) // 64
    seqs = [SeqInit(slot=i, prompt=prompts[i], pages=list(range(1 + i * ppseq, 1 + (i + 1) * ppseq)),
                    temperature=0.7, top_p=0.95, repetition_penalty=1.15, seed=1000 + i) for i in range(total)]
    # p50 TTFT: single P-token request, prefill -> first token visible on the host of rank 0, device-timed
    ttfts = []
    for rep in range(5):
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(runner.stream)
        runner.prefill(seqs[:1])
        runner.sync()                       # device-side wait for the last piece's sampler (no collective)
        e1.record(runner.stream)
        barrier_sync()
        ttfts.append(max_over_ranks(e0.elapsed_time(e1), dev))
        runner.release([0])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                    # nvidia-smi needs ~0.2 s to come up: start it before the warm-up steps
    runner.prefill(seqs)
    runner.decode(W)
    runner.sync()
    barrier_sync()
    launches0 = runner.kernel_launches
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    flush.fill_(1)
    barrier_sync()
    sampler.mark()                         # clocks are reported from the samples taken during the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(runner.stream)
    runner.decode(K)
    e1.record(runner.stream)
    barrier_sync()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop() if rank == 0 else {}
    launches = runner.kernel_launches - launches0
    win = runner.fetch_window([0] * total, 1 + W + K)
    uniq = 0
    if rank == 0:
        assert int((win >= 0).all()) and int((win < cfg.vocab_size).all()), "sampler produced out-of-range ids"
        uniq = len(set(win[:, -1].tolist()))
    if args.dump_outputs and (rank == 0 or runner.last):
        # the last step's logits buffer holds the last group's rows; nothing has overwritten it since the timed window
        dump_outputs(args.dump_outputs, total, tokens=win[:, -1].numpy() if rank == 0 else None,
                     logits=runner.piece.logits[:B, :cfg.vocab_size].cpu().numpy() if runner.last else None)
    runner.release(list(range(total)))
    tok_s = total * K / (ms / 1e3)
    # streamed bytes of ONE group step on this rank: every weight that a decode step reads (the embedding table is
    # only gathered: B rows) + the KV pages of the context
    ctx = P + W + K // 2
    kv_bytes = sum(1 for l in runner.layers if runner.piece.has_attn(l)) * B * ctx * cfg.kv_dim * 2 * 2
    per_rank = gather_objects({"rank": rank, "weight_bytes": runner.piece.streamed_weight_bytes(), "kv_bytes": kv_bytes,
                               "units": runner.units}, world)

    # ---------------- end-to-end through the public API (Engine.generate): host prompts in pinned
    # memory -> H2D, scheduler, graph prefill + decode bursts, token read-back every burst.
    e2e = None
    if not args.no_e2e:
        sp = SamplingParams(max_new_tokens=K, temperature=0.7, top_p=0.95, repetition_penalty=1.15, ignore_eos=True,
                            seed=7)
        eng.decode_burst = min(K, 64)      # tokens are read back once per burst
        eng.generate(prompts, SamplingParams(max_new_tokens=4, ignore_eos=True))   # warm: same prefill buckets as the timed run
        eng.h2d_bytes = eng.d2h_bytes = 0
        h0 = runner.h2d_bytes
        barrier_sync()
        t0 = time.perf_counter()
        outs = eng.generate(prompts, sp)
        torch.cuda.synchronize(dev)
        dt = max_over_ranks(time.perf_counter() - t0, dev)
        n_tok = sum(len(o) for o in outs)
        e2e = {"value": n_tok / dt, "unit": "tokens/s", "wall_s": dt,
               "h2d_bytes_per_step": (eng.h2d_bytes + runner.h2d_bytes - h0) / K,
               "d2h_bytes_per_step": eng.d2h_bytes / K, "includes": "prefill+decode, scheduler, token readback",
               "host_ms": dict(eng.host_ms)}
        # rank-count independence (VERDICT r1 #8): greedy continuation of the same prompts through the same public call;
        # the checksum over the first 32 sequences must be identical at every N (the pieces only change the transport:
        # same kernels, same tiles, same split-K -- tests/test_multigpu.py asserts it token for token on 2 / 4 / 8 GPUs)
        try:
            import zlib
            gouts = eng.generate(prompts, SamplingParams(max_new_tokens=8, temperature=0.0, top_p=1.0,
                                                         repetition_penalty=1.0, ignore_eos=True))
            flat = [int(t) for o in gouts[:32] for t in o]
            e2e["greedy_check"] = {"crc32_first_32_seqs_x_8_tokens": zlib.crc32(",".join(map(str, flat)).encode()),
                                   "seq0": [int(t) for t in gouts[0][:8]]}
        except Exception as exc:        # never let the consistency probe take the measurement down
            e2e["greedy_check"] = {"error": repr(exc)[:200]}

    if rank == 0:
        peaks = measured_peaks()
        step_ms = ms / K
        worst = max(per_rank, key=lambda r: r["weight_bytes"] + r["kv_bytes"])
        # every group step streams a rank's weights once: `groups` times per step
        gbps = [(r["weight_bytes"] + r["kv_bytes"]) * groups / (step_ms / 1e3) / 1e9 for r in per_rank]
        base = baseline_number()
        out = {"metric": "decode_tokens_per_sec", "value": tok_s, "unit": "tokens/s", "n_gpus": world, "steps": K,
               "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": (tok_s / base) if base else None,
               "dtype": {"bf16": "bf16", "fp8": "fp8-e4m3 W8A8 per-row/per-token scales (bf16 KV/attention/residual)",
                         "mxfp8": "mxfp8 block-scaled e4m3 W8A8, UE8M0 per 32 K (bf16 KV/attention/residual)"}[args.dtype],
               "data": "synthetic", "impl": "ours",
               "config": common_fields(args, world, total, K, W, P, {
                   "parallelism": f"pp{world}",
                   "piece_units": "/".join(str(b - a) for a, b in eng.runner.unit_ranges) + " thirds of a layer (attention block | gate/up | down)",
                   "micro_batch_groups": groups, "batch_per_group": B}),
               "p50_ttft_ms": statistics.median(ttfts), "gpu_launches": launches, "clocks": clocks, "e2e": e2e,
               "roofline": {"accounting": "bytes a decode step streams per rank (weights without the gathered embedding "
                                          "table + KV pages); max-stage rank reported, all ranks listed",
                            "streamed_bytes_per_group_step": [r["weight_bytes"] + r["kv_bytes"] for r in per_rank],
                            "achieved_stream_GBps_per_rank": gbps,
                            "max_stage_rank": worst["rank"],
                            "hbm_frac_of_measured_max_stage": (max(gbps) / peaks["hbm_gbs"]) if peaks.get("hbm_gbs") else None,
                            "hbm_frac_of_measured_mean": (sum(gbps) / len(gbps) / peaks["hbm_gbs"]) if peaks.get("hbm_gbs") else None},
               "distinct_last_tokens": uniq}
        print(json.dumps(out), flush=True)
    eng.close()
    shutdown()


# ------------------------------------------------------------------- B: constructed NCCL(+cuBLAS) pipeline
def run_nccl(args):
    """OUR CONSTRUCTED comparator (never the reference's build): same pieces / groups / batch as `ours`, library ops
    (cuBLAS, flash-attn / SDPA, ATen) and torch.distributed NCCL send/recv between the stages."""
    import torch
    import torch.distributed as dist

    from baseline.nccl_pipeline import NcclPipeline
    from bee2bee_b200.models.config import resolve_config
    from bee2bee_b200.parallel.dist import init_distributed, max_over_ranks, shutdown

    os.environ.setdefault("TORCH_NCCL_SHOW_EAGER_INIT_P2P_SERIALIZATION_WARNING", "false")
    rank, world, local = init_distributed(eager=False)       # per-pair P2P communicators: hops are not serialised
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    cfg = resolve_config(args.model)
    groups = args.groups or world
    B, K, W, P = args.batch, args.steps, max(3, args.warmup), args.prompt_len
    total = B * groups
    max_len = ((P + 2 * (K + W) + 8 + 63) // 64) * 64
    pipe = NcclPipeline(args.model, rank, world, dev, groups, B, max_len)
    prompts_host = torch.tensor(synthetic_prompts(total, P, cfg.vocab_size), dtype=torch.int64).pin_memory()

    def barrier_sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def reset_and_prefill():
        pipe.prefill(prompts_host.to(dev, non_blocking=True))

    ttfts = []
    one = prompts_host[:B].repeat(groups, 1)
    for rep in range(3):
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.stream)
        pipe.prefill(one.to(dev, non_blocking=True))
        pipe.finish()
        e1.record(pipe.stream)
        barrier_sync()
        ttfts.append(max_over_ranks(e0.elapsed_time(e1), dev))
    reset_and_prefill()
    pipe.capture()
    pipe.decode(W)
    pipe.finish()
    barrier_sync()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush.fill_(1)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    calls0 = pipe.nccl_calls
    barrier_sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(pipe.stream)
    pipe.decode(K)
    pipe.finish()
    e1.record(pipe.stream)
    barrier_sync()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop() if rank == 0 else {}
    tok_s = total * K / (ms / 1e3)
    toks = pipe.tokens().cpu()
    assert int((toks >= 0).all()) and int((toks < cfg.vocab_size).all())
    # end to end: pinned prompts -> H2D -> prefill -> K decode steps -> tokens read back once per burst of <= 64 steps
    e2e = None
    if not args.no_e2e:
        reset_and_prefill()                 # warm pass, like the product arm's
        pipe.decode(2)
        pipe.finish()
        barrier_sync()
        t0 = time.perf_counter()
        reset_and_prefill()
        done, d2h = 0, 0
        while done < K:
            n = min(64, K - done)
            pipe.decode(n)
            pipe.finish()
            pipe.stream.synchronize()
            d2h += pipe.tokens().cpu().numel() * 8
            done += n
        barrier_sync()
        dt = max_over_ranks(time.perf_counter() - t0, dev)
        e2e = {"value": total * K / dt, "unit": "tokens/s", "wall_s": dt, "h2d_bytes_per_step": prompts_host.numel() * 8 / K,
               "d2h_bytes_per_step": d2h / K, "includes": "prefill+decode, token readback once per burst"}
    if rank == 0:
        print(json.dumps({"metric": "decode_tokens_per_sec", "value": tok_s, "unit": "tokens/s", "n_gpus": world, "steps": K,
                          "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "impl": "nccl",
                          "label": "B: OUR CONSTRUCTED NCCL(+cuBLAS) pipeline -- not the reference's build (it has none)",
                          "config": common_fields(args, world, total, K, W, P, {
                              "parallelism": f"pp{world}", "micro_batch_groups": groups, "batch_per_group": B,
                              "layers_per_piece": "whole layers", "attention": "flash_attn_with_kvcache" if pipe.fa else "SDPA + mask",
                              "hop": "torch.distributed NCCL send/recv", "compute": "CUDA graph of library ops per (rank, group)"}),
                          "p50_ttft_ms": statistics.median(ttfts), "nccl_calls_timed": pipe.nccl_calls - calls0,
                          "gpu_launches": 0, "clocks": clocks, "e2e": e2e}), flush=True)
    shutdown()


# ------------------------------------------------------------------------- A: reference
def run_reference(args):
    """Unmodified reference (baseline/_ref): HFService -> transformers.generate on one GPU per rank
    (the reference has no multi-GPU path; N ranks = N independent replica providers, which is its own
    "load balancing" story, /root/reference/bee2bee/p2p_runtime.py:723-757)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "bee2bee")):
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref not installed"}))
        return
    sys.path.insert(0, ref)
    try:
        import torch
        from bee2bee.services import HFService  # noqa
    except Exception as e:
        print(json.dumps({"impl": "reference", "unavailable": f"import failed: {e!r}"[:200]}))
        return
    from baseline.ref_model import build_reference_checkpoint   # builds config/tokenizer/weights with transformers
    from bee2bee_b200.parallel.dist import init_distributed, max_over_ranks, shutdown

    rank, world, local = init_distributed()
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
    K, W, B, P = args.steps, max(3, args.warmup), args.batch, args.prompt_len
    total = B * (args.groups or world)
    per_rank = total // world
    path = build_reference_checkpoint(args.model, rank)
    svc = HFService(path, 0.0)
    svc.load_sync()
    prompts = [" ".join(f"t{(7 + 131 * i + 31 * j) % 100000 + 300}" for j in range(P)) for i in range(total)]
    mine = prompts[rank * per_rank:(rank + 1) * per_rank]
    svc.execute({"prompt": mine[0], "max_new_tokens": W, "temperature": 0.7})
    # TTFT of the reference's path: one request that generates a single token (prefill + first sample), wall clock
    ttfts = []
    for _ in range(3):
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        t = time.perf_counter()
        svc.execute({"prompt": mine[0], "max_new_tokens": 1, "temperature": 0.7})
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        ttfts.append((time.perf_counter() - t) * 1e3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    toks = 0
    for p in mine:
        r = svc.execute({"prompt": p, "max_new_tokens": K, "temperature": 0.7})
        toks += int(r.get("tokens") or K)
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0, "cuda" if torch.cuda.is_available() else None)
    clocks = sampler.stop() if rank == 0 else {}
    if rank == 0:
        val = toks * world / dt
        print(json.dumps({"metric": "decode_tokens_per_sec", "value": val, "unit": "tokens/s", "n_gpus": world,
                          "steps": K, "warmup": W, "ms_per_step": dt * 1e3 / K, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                          "impl": "reference",
                          "config": {"model": args.model, "global_batch": total, "seq_len": P + K, "prompt_len": P,
                                     "parallelism": f"replica x{world} (reference has no model parallelism)",
                                     "path": "HFService.execute -> transformers.generate, one request at a time",
                                     "note": "the timed region contains prefill + decode of every request (the reference "
                                             "has no other path); inputs are tokenised text, copied to the GPU by "
                                             "transformers inside generate()"},
                          "p50_ttft_ms": statistics.median(ttfts),
                          "clocks": clocks, "e2e": {"value": val, "unit": "tokens/s",
                                                    "h2d_bytes_per_step": P * 8 * per_rank / K, "d2h_bytes_per_step": 8 * per_rank},
                          "gpu_launches": 0}), flush=True)
    shutdown()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "nccl":
        run_nccl(a)
    else:
        run_ours(a)
