"""Per-GPU executor of one piece: device-resident batch state, bucketed CUDA-graph prefill,
CUDA-graph decode bursts, wavefront micro-batch groups.  One ``GpuRunner`` per process/GPU;
rank 0 also owns the token buffers the last piece's sampler writes into over NVLink.

Everything between the host's ``prefill`` / ``decode`` calls and its ``fetch_window`` read-back is
device-driven (all ranks enqueue the same plan):

    prefill(new sequences)  : one pinned staging copy + one graph replay per chunk; chunks travel through the
                              pieces as a wavefront on their own double-buffered channel whose slots are
                              flow-controlled by release / ack flags (no host barrier between chunks)
    decode(n steps)         : for step: for group g: replay graph[g]   -- device-side flags only
                              (piece i works on group g+1 while piece i+1 works on group g)
    fetch_window(...)       : ONE kernel that waits for the sampler / prefill-done flags on rank 0 (peer memory
                              for follower ranks) and gathers the new tokens into mapped pinned host memory

All flags are monotonic epochs that are never reset, so no burst needs a host barrier, a flag reset or an
NCCL broadcast (round 1 paid two barriers + a reset per burst and a broadcast per read-back).
Replaces the per-hop JSON transport of /root/reference/bee2bee/node.py:249-277.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import ops
from ..models.config import UNITS_PER_LAYER, ModelConfig, piece_units, unit_layers
from ..models.native import BatchMeta, NativePiece
from ..models.weights import load_or_init
from ..parallel.mesh import F_TOK_DONE, MeshComm
from .kv import PAGE


@dataclass
class SeqInit:
    """Everything a rank needs to start a sequence (part of the replicated plan)."""
    slot: int
    prompt: List[int]
    pages: List[int]
    temperature: float = 0.7
    top_p: float = 0.95
    repetition_penalty: float = 1.15
    seed: int = 0
    cached: int = 0          # leading prompt tokens whose KV is already resident in ``pages`` (prefix cache): not prefilled


def _pow2_at_least(n: int, lo: int = 1) -> int:
    v = lo
    while v < n:
        v *= 2
    return v


class MeshStalled(RuntimeError):
    """A bounded device-side wait on a peer's flag gave up (late / hung / dead rank): the results of the burst are
    garbage and the mesh epochs are no longer aligned.  The process and its CUDA context are intact."""


class _HostRing:
    """Mapped pinned host memory (cudaHostAlloc) visible to kernels by address and to the host as a tensor."""

    def __init__(self, C, n_int32: int):
        self.C, self.n = C, n_int32
        self.host_ptr, self.dev_ptr = C.host_ring_alloc(max(64, n_int32 * 4))
        self.view = C.tensor_from_ptr(self.host_ptr, [n_int32], "i32", -1)

    def free(self) -> None:
        if self.host_ptr:
            try:
                self.C.host_ring_free(self.host_ptr)
            except Exception:
                pass
            self.host_ptr = 0


class GpuRunner:
    def __init__(self, cfg: ModelConfig, model: str = "", rank: int = 0, world: int = 1,
                 device: Optional[torch.device] = None, max_batch: int = 32, groups: int = 1,
                 max_seq_len: int = 4096, max_prefill_tokens: int = 2048, num_pages: int = 0, seed: int = 0,
                 hist_len: int = 0, control_group=None, use_graphs: bool = True, quant: str = "bf16"):
        assert max_batch % groups == 0, "max_batch must be divisible by the number of micro-batch groups"
        self.cfg, self.rank, self.world = cfg, rank, world
        self.device = torch.device(device if device is not None else f"cuda:{rank}")
        torch.cuda.set_device(self.device)
        self.max_batch, self.groups, self.gb = max_batch, groups, max_batch // groups
        self.max_seq_len = max_seq_len
        self.max_pages_per_seq = (max_seq_len + PAGE - 1) // PAGE
        self.max_prefill_tokens = max_prefill_tokens
        # token history ring per slot: the scheduler reads every burst's window before the sampler can lap it
        self.hist_len = hist_len if hist_len > 0 else max(256, min(4096, _pow2_at_least(max_seq_len)))
        self.use_graphs = use_graphs
        # piece boundaries in third-of-a-layer units (attention block | gate/up GEMM | down GEMM), balanced for the
        # wavefront: the last piece also streams the lm_head and runs the sampler.  B2B_UNIT_BOUNDS="0,4,12" overrides the
        # search (tests).
        env_bounds = os.environ.get("B2B_UNIT_BOUNDS", "")
        bounds = [int(v) for v in env_bounds.split(",")] if env_bounds and world > 1 else None
        self.unit_ranges = piece_units(cfg, world, bounds)
        assert len(self.unit_ranges) == world, f"{cfg.name}: cannot split into {world} pieces ({self.unit_ranges})"
        self.units = self.unit_ranges[rank]
        self.layers = list(unit_layers(self.units))
        # a cut between a gate/up and a down GEMM anywhere in the mesh -> every hop slot also stages the MLP hidden
        mlp_cut = any(u1 % UNITS_PER_LAYER == 2 for _, u1 in self.unit_ranges[:-1])
        self.first, self.last = rank == 0, rank == world - 1
        if num_pages <= 0:
            num_pages = 1 + max_batch * self.max_pages_per_seq
        self.num_pages = num_pages
        tensors = load_or_init(model, cfg, self.layers, self.first, self.last, device=self.device,
                               dtype=torch.bfloat16, seed=seed)
        max_tokens = max(max_prefill_tokens, self.gb, 16)
        self.max_tokens = max_tokens
        self.max_chunk_seqs = max(self.gb, 64)
        self.piece = NativePiece(cfg, self.layers, self.first, self.last, tensors, self.device, max_tokens,
                                 self.max_chunk_seqs, num_pages, quant=quant, units=self.units)
        del tensors
        self.mesh = MeshComm(rank, world, self.device, cfg.hidden_size, max_tokens, groups, self.gb, self.hist_len,
                             control_group, ffn=cfg.ffn_size if mlp_cut else 0,
                             mx=bool(getattr(self.piece, "mx_hand", False)))
        self.C = ops.native()
        dev, i32 = self.device, torch.int32
        B = max_batch
        # ---- device-resident batch state (static addresses -> CUDA graphs)
        if world > 1 and self.first:
            self.tokens = self.mesh.local_view("tok", (B,), "i32")
            self.history = self.mesh.local_view("hist", (B, self.hist_len), "i32")
        else:
            self.tokens = torch.zeros(B, device=dev, dtype=i32)
            self.history = torch.zeros((B, self.hist_len), device=dev, dtype=i32)
        self.positions = torch.zeros(B, device=dev, dtype=i32)
        self.kv_len = torch.zeros(B, device=dev, dtype=i32)
        self.q_len = torch.zeros(B, device=dev, dtype=i32)
        self.slots = torch.full((B,), -1, device=dev, dtype=i32)
        self.block_table = torch.zeros((B, self.max_pages_per_seq), device=dev, dtype=i32)
        self.q_start = torch.arange(self.gb, device=dev, dtype=i32)
        self.temperature = torch.zeros(B, device=dev)
        self.top_p = torch.ones(B, device=dev)
        self.rep_pen = torch.ones(B, device=dev)
        self.seeds = torch.zeros(B, device=dev, dtype=i32)
        self.hist_pos = torch.zeros(B, device=dev, dtype=i32)
        self.step_ctr = torch.zeros(1, device=dev, dtype=i32)
        self.seen = torch.zeros((B, (cfg.vocab_size + 31) // 32), device=dev, dtype=i32)
        self.tok_local = torch.zeros(B, device=dev, dtype=i32)     # last rank's own copy of sampled ids
        self.graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self._pf: Dict[tuple, dict] = {}           # prefill state (staging + graph) per bucket
        self.stream = torch.cuda.Stream(device=dev)
        self.kernel_launches = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self.decode_splits = 1
        if max_seq_len > 1024:
            self.decode_splits = max(1, min(self.piece.max_splits, ops.NUM_SMS // max(1, self.gb * cfg.n_kv_heads)))
        # ---- host <-> device rendezvous without collectives
        self.tok_target = [1] * groups              # value rank 0's token flag of group g reaches after the enqueued steps
        self.pf_calls = 0                           # prefill() calls so far
        self.pf_need = [0] * groups                 # chunks the last piece must have completed before group g may decode
        self.pf_chunks = 0                          # chunks sent through the prefill channel (parity of the staging buffer)
        self._cur = _HostRing(self.C, B)            # per-slot read cursors (host writes, kernel reads)
        self._waits = _HostRing(self.C, 4 * (groups + 2))
        self._win: Optional[_HostRing] = None
        self._win_width = 0
        self._fetch_ev = torch.cuda.Event()
        self.C.init_kernels(self.device.index)
        # bounded handoff waits: a peer that does not publish within the limit raises the (device-resident) abort word
        # instead of trapping the GPU; fetch_window reports it through a mapped host word.  B2B_WAIT_TIMEOUT_MS=0 -> trap.
        self.wait_timeout_ms = float(os.environ.get("B2B_WAIT_TIMEOUT_MS", "30000"))
        self.aborted = False
        self._status = _HostRing(self.C, 16)
        self._status.view.zero_()
        self._abort_word = self.C.peer_alloc(256)
        self.C.tensor_from_ptr(self._abort_word, [64], "i32", self.device.index).zero_()
        torch.cuda.synchronize(self.device)
        self.C.set_wait_policy(self._abort_word if self.wait_timeout_ms > 0 else 0, self.wait_timeout_ms)
        if world == 1:
            self.warmup()
        self._ensure_graphs()

    # ------------------------------------------------------------------ helpers
    def _grp(self, t: torch.Tensor, g: int) -> torch.Tensor:
        return t[g * self.gb:(g + 1) * self.gb]

    def launches_per_decode_step(self) -> int:
        """Native kernel launches one rank issues per group decode step: counted while the decode graph was recorded
        (``ops.LAUNCHES``); before the first capture, an estimate from the layer structure."""
        if getattr(self, "_decode_launches", 0):
            return self._decode_launches
        c, n = self.cfg, len(self.layers)
        if c.norm == "ln":
            per = 9
        elif c.post_norms:
            per = 7
        else:
            per = 5
        if self.piece.fp8:
            # activation quantisers (QKV, O, gate/up, down inputs); mxfp8 with fused epilogues keeps one per piece head
            per += 0 if getattr(self.piece, "mx_fuse", False) else 4
        total = 1 + n * per                      # decode_advance + layers
        if per == 5 and not self.piece.fp8:
            total = 1 + self.piece.n_launches()  # sub-layer piece ends: count the GEMMs / attention actually present
        if self.first:
            total += 1                           # embed
        if self.last:
            total += 2 + (0 if c.norm == "rms" else 1)   # lm_head GEMM + sampler (+ final LN)
            if not self.first:
                total += 1                       # input-slot release
        return total

    # ------------------------------------------------------------------ prefill
    def prefill(self, seqs: Sequence[SeqInit]) -> None:
        """Run the prompts of ``seqs`` through this rank's piece (chunked, wavefront), install their decode state,
        and (last rank) sample their first token into rank 0's token buffer.  Nothing here waits on the host: the
        caller's next ``fetch_window(first=True)`` is the synchronisation point."""
        if not seqs:
            return
        with torch.cuda.stream(self.stream):
            self._install(seqs)
            for chunk in self._pack(seqs):
                self._run_chunk(chunk)
                # the last piece publishes "chunk #n done: its sequences' first tokens are in rank 0's ring" (inside the
                # chunk graph); a group may start decoding as soon as the chunks holding ITS sequences are through --
                # piece 0's embed kernel waits for that count, so decode can be enqueued right behind the prefill and
                # the pipeline never drains between the two
                for s, _, c1 in chunk:
                    if c1 == len(s.prompt):
                        g = s.slot // self.gb
                        self.pf_need[g] = max(self.pf_need[g], self.pf_chunks)
            self.pf_calls += 1
            if self.world > 1 and self.first:
                need = torch.tensor(self.pf_need, dtype=torch.int32).pin_memory()
                self.mesh.local_view("pf_need", (self.groups,), "i32").copy_(need, non_blocking=True)

    def _install(self, seqs: Sequence[SeqInit]) -> None:
        """Per-sequence state of all admitted sequences in a handful of batched copies (one tiny launch per field
        and sequence cost ~25 ms for 256 admissions)."""
        dev, i32 = self.device, torch.int32
        S = len(seqs)
        bt_np = np.zeros((S, self.max_pages_per_seq), dtype=np.int32)
        for i, s in enumerate(seqs):
            bt_np[i, :len(s.pages)] = s.pages
        bt_host = torch.from_numpy(bt_np)
        fl_host = torch.tensor([[s.temperature, s.top_p, s.repetition_penalty] for s in seqs], dtype=torch.float32)
        seed_host = torch.tensor([int(s.seed) & 0x7FFFFFFF for s in seqs], dtype=i32)
        rows = torch.tensor([s.slot for s in seqs], dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
        fl = fl_host.pin_memory().to(dev, non_blocking=True)
        self.block_table.index_copy_(0, rows, bt_host.pin_memory().to(dev, non_blocking=True))
        self.temperature.index_copy_(0, rows, fl[:, 0].contiguous())
        self.top_p.index_copy_(0, rows, fl[:, 1].contiguous())
        self.rep_pen.index_copy_(0, rows, fl[:, 2].contiguous())
        self.seeds.index_copy_(0, rows, seed_host.pin_memory().to(dev, non_blocking=True))
        self.hist_pos.index_fill_(0, rows, 0)
        self.seen.index_fill_(0, rows, 0)
        self.h2d_bytes += bt_host.numel() * 4 + fl_host.numel() * 4 + S * (4 + 8)
        if self.last:
            flat = np.concatenate([np.asarray(s.prompt, dtype=np.int32) for s in seqs])
            owner = np.repeat(np.asarray([s.slot for s in seqs], dtype=np.int32), [len(s.prompt) for s in seqs])
            self.h2d_bytes += 8 * len(flat)
            ops.mark_seen(torch.from_numpy(flat).pin_memory().to(dev, non_blocking=True),
                          torch.from_numpy(owner).pin_memory().to(dev, non_blocking=True), self.seen,
                          self.cfg.vocab_size)

    def _pack(self, seqs: Sequence[SeqInit]) -> List[List[Tuple[SeqInit, int, int]]]:
        """prompts -> chunks of <= max_prefill_tokens tokens / max_chunk_seqs sequences; one sequence contributes at
        most one span per chunk (a later span attends to the KV of the earlier one)."""
        work: List[Tuple[SeqInit, int, int]] = []
        for s in seqs:
            L = len(s.prompt)
            for c0 in range(min(s.cached, L - 1), L, self.max_prefill_tokens):     # the cached prefix is attended to, not recomputed
                work.append((s, c0, min(L, c0 + self.max_prefill_tokens)))
        batch: List[Tuple[SeqInit, int, int]] = []
        used = 0
        chunks: List[List[Tuple[SeqInit, int, int]]] = []
        for w in work:
            n = w[2] - w[1]
            same_seq = any(x[0].slot == w[0].slot for x in batch)
            if batch and (used + n > self.max_prefill_tokens or same_seq or len(batch) >= self.max_chunk_seqs):
                chunks.append(batch)
                batch, used = [], 0
            batch.append(w)
            used += n
        if batch:
            chunks.append(batch)
        return chunks

    # ---- bucketed prefill: static staging + (optionally) a captured graph per (tokens, sequences, max_q, parity) ----
    def _pf_bucket(self, T: int, S: int, max_q: int) -> Tuple[int, int, int]:
        tb = min(_pow2_at_least(T, 16), self.max_tokens)
        if tb < T:
            tb = self.max_tokens
        sb = 1 if S == 1 else (8 if S <= 8 else self.max_chunk_seqs)
        sb = min(sb, self.max_chunk_seqs)
        mq = min(_pow2_at_least(max_q, 16), tb)
        return tb, sb, mq

    def _pf_state(self, key: Tuple[int, int, int, int]) -> dict:
        st = self._pf.get(key)
        if st is not None:
            return st
        tb, sb, mq, parity = key
        dev, i32 = self.device, torch.int32
        mp = self.max_pages_per_seq
        n = 3 * tb + 5 * sb + sb * mp
        stage = torch.zeros(n, device=dev, dtype=i32)
        o = 0

        def take(k):
            nonlocal o
            v = stage[o:o + k]
            o += k
            return v

        v = {"ids": take(tb), "pos": take(tb), "slots": take(tb), "q_start": take(sb), "q_len": take(sb),
             "kv_len": take(sb), "last_idx": take(sb), "row_map": take(sb), "bt": take(sb * mp).view(sb, mp)}
        hosts = [torch.zeros(n, dtype=i32).pin_memory() for _ in range(4)]      # staging ring: copies stay in flight
        st = {"stage": stage, "v": v, "hosts": hosts, "hosts_np": [t.numpy() for t in hosts], "events": [None] * 4,
              "turn": 0, "graph": None, "n": n}
        hand = self.mesh.handoff_prefill(parity) if self.world > 1 else None
        x_in = h_in = None
        if not self.first:
            x_in = self.C.tensor_from_ptr(hand.in_x, [tb, self.cfg.hidden_size], "bf16", dev.index)
            if self.piece.head_mode == 2:
                h_in = self.C.tensor_from_ptr(hand.in_h, [tb, self.cfg.ffn_size], "bf16", dev.index)
        meta = BatchMeta(ids=v["ids"], positions=v["pos"], slots=v["slots"], q_start=v["q_start"], q_len=v["q_len"],
                         kv_len=v["kv_len"], block_table=v["bt"], n_tokens=tb, n_seqs=sb, max_q=mq,
                         last_idx=v["last_idx"])
        st["meta"] = meta       # captured kernels address these views by raw pointer: keep them alive

        def body():
            out = self.piece.forward(meta, x_in=x_in, hand=hand, h_in=h_in)
            if self.last:
                multi = self.world > 1
                ops.sample(out, self.tok_local if multi else self.tokens, seen=self.seen, temperature=self.temperature,
                           top_p=self.top_p, rep_penalty=self.rep_pen, seeds=self.seeds, step=self.step_ctr,
                           vocab=self.cfg.vocab_size, softcap=self.cfg.final_softcap,
                           history=self.mesh.hist_base() if multi else self.history.data_ptr(), hist_pos=self.hist_pos,
                           hist_stride=self.hist_len, peer_tokens=self.mesh.tok_base() if multi else 0,
                           row_map=v["row_map"].data_ptr())
                if multi:
                    flag, epoch = self.mesh.pf_done_signal()
                    self.C.flag_signal(flag, epoch, 0, 0)       # chunk counter on rank 0 (release after the peer stores)
            self.C.set_decode_state(self.positions, self.kv_len, self.q_len, v["row_map"].data_ptr(),
                                    v["kv_len"].data_ptr(), sb)

        st["body"] = body
        if self.use_graphs:
            with torch.cuda.stream(self.stream):
                if self.world == 1:
                    # dry run (allocations, descriptor cache): every row inactive -> no KV / state / token is written
                    v["slots"].fill_(-1)
                    v["row_map"].fill_(-1)
                    v["q_len"].zero_()
                    body()
                    self.stream.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = ops.LAUNCHES[0]
                with torch.cuda.graph(g, stream=self.stream, capture_error_mode="thread_local"):
                    body()
                st["launches"] = ops.LAUNCHES[0] - n0        # kernels recorded into this chunk graph
                st["graph"] = g
        self._pf[key] = st
        return st

    def _run_chunk(self, chunk: List[Tuple[SeqInit, int, int]]) -> None:
        T = sum(c1 - c0 for _, c0, c1 in chunk)
        S = len(chunk)
        tb, sb, mq = self._pf_bucket(T, S, max(c1 - c0 for _, c0, c1 in chunk))
        parity = (self.pf_chunks & 1) if self.world > 1 else 0
        st = self._pf_state((tb, sb, mq, parity))
        turn = st["turn"]
        st["turn"] = (turn + 1) % len(st["hosts"])
        if st["events"][turn] is not None:
            st["events"][turn].synchronize()         # the copy that last used this host buffer has been consumed
        h = st["hosts_np"][turn]
        h[:] = 0
        mp = self.max_pages_per_seq
        o_pos, o_slots, o_qs = tb, 2 * tb, 3 * tb
        o_ql, o_kv, o_last, o_row, o_bt = o_qs + sb, o_qs + 2 * sb, o_qs + 3 * sb, o_qs + 4 * sb, o_qs + 5 * sb
        h[o_slots:o_slots + tb] = -1
        h[o_row:o_row + sb] = -1
        lens = [c1 - c0 for _, c0, c1 in chunk]
        starts = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int32)
        pos = np.concatenate([np.arange(c0, c1, dtype=np.int32) for _, c0, c1 in chunk])
        h[0:T] = np.concatenate([np.asarray(s.prompt[c0:c1], dtype=np.int32) for s, c0, c1 in chunk])
        h[o_pos:o_pos + T] = pos
        bt = h[o_bt:o_bt + sb * mp].reshape(sb, mp)
        for i, (s, c0, c1) in enumerate(chunk):
            bt[i, :len(s.pages)] = s.pages
        seq_of = np.repeat(np.arange(S, dtype=np.int32), lens)
        h[o_slots:o_slots + T] = bt[seq_of, pos >> 6] * PAGE + (pos & (PAGE - 1))
        h[o_qs:o_qs + S] = starts
        h[o_ql:o_ql + S] = lens
        h[o_kv:o_kv + S] = [c1 for _, _, c1 in chunk]
        h[o_last:o_last + S] = starts + np.asarray(lens, dtype=np.int32) - 1
        h[o_row:o_row + S] = [s.slot if c1 == len(s.prompt) else -1 for s, _, c1 in chunk]
        h = st["hosts"][turn]
        self.h2d_bytes += st["n"] * 4
        st["stage"].copy_(h, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(self.stream)
        st["events"][turn] = ev
        if st["graph"] is not None:
            st["graph"].replay()
        else:
            st["body"]()
        self.pf_chunks += 1
        self.kernel_launches += st.get("launches") or (self.launches_per_decode_step() + 1)

    # ------------------------------------------------------------------- decode
    def _decode_group(self, g: int) -> None:
        """One decode step of micro-batch group g on this rank (graph-capturable)."""
        gb = self.gb
        pos, kvl, slots, ql = (self._grp(x, g) for x in (self.positions, self.kv_len, self.slots, self.q_len))
        bt = self._grp(self.block_table, g)
        self.C.decode_advance(pos, kvl, slots, ql, bt)
        meta = BatchMeta(ids=self._grp(self.tokens, g), positions=pos, slots=slots, q_start=self.q_start, q_len=ql,
                         kv_len=kvl, block_table=bt, n_tokens=gb, n_seqs=gb, max_q=1, splits=self.decode_splits)
        hand = self.mesh.handoff(g)
        x_in = h_in = None
        if not self.first:
            x_in = self.C.tensor_from_ptr(hand.in_x, [gb, self.cfg.hidden_size], "bf16", self.device.index)
            if self.piece.head_mode == 2:
                h_in = self.C.tensor_from_ptr(hand.in_h, [gb, self.cfg.ffn_size], "bf16", self.device.index)
        out = self.piece.forward(meta, x_in=x_in, hand=hand if self.world > 1 else None, h_in=h_in)
        if self.last:
            multi = self.world > 1
            hist_ptr = (self.mesh.history_ptr(g) if multi else self._grp(self.history, g).data_ptr())
            ops.sample(out, self._grp(self.tok_local, g) if multi else self._grp(self.tokens, g),
                       seen=self._grp(self.seen, g), temperature=self._grp(self.temperature, g),
                       top_p=self._grp(self.top_p, g), rep_penalty=self._grp(self.rep_pen, g),
                       seeds=self._grp(self.seeds, g), step=self.step_ctr, vocab=self.cfg.vocab_size,
                       softcap=self.cfg.final_softcap, history=hist_ptr, hist_pos=self._grp(self.hist_pos, g),
                       hist_stride=self.hist_len, peer_tokens=hand.out_x if multi else 0,
                       signal_flag=hand.out_flag if multi else 0, signal_epoch=hand.out_epoch if multi else 0,
                       done_counter=(self.mesh._flag(self.mesh.local, g, F_TOK_DONE) if multi else 0))
            if g == self.groups - 1:
                self.step_ctr.add_(1)

    def _ensure_graphs(self) -> None:
        if self.graphs or not self.use_graphs:
            return
        # multi-rank: graphs that spin on peer flags cannot be warmed up in isolation; capture without a dry run.
        # ONE graph holds a decode step of every group (in wavefront order): the PDL chain then also spans the group
        # boundaries (the first kernel of group g+1 becomes resident under the tail of group g) and a step costs one
        # graph launch instead of `groups`.  B2B_GRAPH_PER_GROUP=1 restores one graph per group.
        per_group = os.environ.get("B2B_GRAPH_PER_GROUP", "0") == "1"
        n0 = ops.LAUNCHES[0]
        with torch.cuda.stream(self.stream):
            if per_group:
                for g in range(self.groups):
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, stream=self.stream, capture_error_mode="thread_local"):
                        self._decode_group(g)
                    self.graphs[g] = graph
            else:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=self.stream, capture_error_mode="thread_local"):
                    for g in range(self.groups):
                        self._decode_group(g)
                self.graphs[-1] = graph
        self._decode_launches = (ops.LAUNCHES[0] - n0) // self.groups      # kernels recorded per group step
        self.stream.synchronize()

    def warmup(self) -> None:
        """Eagerly run every kernel variant once (sets smem attributes, fills the TMA descriptor
        cache) with all rows inactive, so nothing is written to the KV cache. Single rank only;
        multi-rank warm-up happens through a real burst."""
        if self.world > 1:
            return
        saved = self.q_len.clone()
        self.q_len.zero_()
        pos, kvl = self.positions.clone(), self.kv_len.clone()
        with torch.cuda.stream(self.stream):
            for g in range(self.groups):
                self._decode_group(g)
        self.stream.synchronize()
        self.q_len.copy_(saved)
        self.positions.copy_(pos)
        self.kv_len.copy_(kvl)
        self.hist_pos.zero_()
        self.step_ctr.zero_()
        self.seen.zero_()
        self.tokens.zero_()
        torch.cuda.synchronize(self.device)

    def prepare_burst(self) -> None:
        """Kept for callers of the round-1 API: bursts need no preparation any more (monotonic epochs)."""
        self._ensure_graphs()

    def decode(self, n_steps: int, prepared: bool = False) -> None:
        """Enqueue ``n_steps`` decode steps for every group (no host synchronisation, no collective)."""
        from ..utils.tracing import TRACER
        with TRACER.range(f"decode_burst[{n_steps}]", self.stream):
            self._enqueue_decode(n_steps)

    def _enqueue_decode(self, n_steps: int) -> None:
        with torch.cuda.stream(self.stream):
            step_graph = self.graphs.get(-1) if self.use_graphs else None
            for _ in range(n_steps):
                if step_graph is not None:
                    step_graph.replay()
                    continue
                for g in range(self.groups):
                    if self.use_graphs:
                        self.graphs[g].replay()
                    else:
                        self._decode_group(g)
        for g in range(self.groups):
            self.tok_target[g] += n_steps
        self.kernel_launches += n_steps * self.groups * self.launches_per_decode_step()

    # ------------------------------------------------------------------- results
    def fetch_window(self, cursors: Sequence[int], width: int, first: bool = False) -> torch.Tensor:
        """[max_batch, width] int32 on the host: tokens ``cursors[b] .. cursors[b] + width`` of every slot's ring.

        One kernel: waits until rank 0's flags say that everything enqueued so far has been produced (the sampler
        flag of every group has reached its target; after a prefill, the prefill-done counter), then gathers from
        rank 0's ring (peer memory on follower ranks) into mapped pinned host memory.  This is also the only point
        where the host blocks; every rank blocks on the same global condition, so the ranks' schedulers stay in
        lock-step without a collective."""
        B = self.max_batch
        if self._win is None or self._win_width < width:
            if self._win is not None:
                self._win.free()
            self._win_width = max(width, 64)
            self._win = _HostRing(self.C, B * self._win_width)
        self._cur.view[:B] = torch.as_tensor(list(cursors), dtype=torch.int32)
        n_waits = 0
        if self.world > 1:
            w64 = self._waits.view.view(torch.int64)
            for g in range(self.groups):
                w64[2 * n_waits], w64[2 * n_waits + 1] = self.mesh.tok_flag(g), self.tok_target[g]
                n_waits += 1
            if first or self.pf_chunks:
                w64[2 * n_waits], w64[2 * n_waits + 1] = self.mesh.pf_done_flag(), self.pf_chunks
                n_waits += 1
        hist = self.mesh.hist_base() if self.world > 1 else self.history.data_ptr()
        with torch.cuda.stream(self.stream):
            self.C.fetch_window(hist, self.hist_len, self._cur.dev_ptr, B, width, self._win.dev_ptr, self._waits.dev_ptr,
                                n_waits, self._status.dev_ptr)
            self._fetch_ev.record(self.stream)
        self._fetch_ev.synchronize()
        if int(self._status.view[0]) != 0:
            self.aborted = True
            raise MeshStalled(f"rank {self.rank}: a peer piece did not publish its handoff flag within "
                              f"{self.wait_timeout_ms:.0f} ms; the burst was drained and discarded")
        self.h2d_bytes += B * 4 + n_waits * 16
        self.d2h_bytes += B * width * 4
        return self._win.view[:B * width].view(B, width).clone()

    def sync(self) -> None:
        """Block until everything enqueued so far has completed on EVERY rank (device-side condition, no collective)."""
        self.fetch_window([0] * self.max_batch, 1)

    def read_history(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(history ring [B, hist_len], hist_pos [B]) on the host.  hist_pos lives on the last rank; on a
        multi-rank mesh the caller tracks positions by step count instead."""
        return self.history.cpu(), self.hist_pos.cpu()

    def release(self, slots: Sequence[int]) -> None:
        if not slots:
            return
        with torch.cuda.stream(self.stream):
            rows = torch.tensor(list(slots), dtype=torch.int64).pin_memory().to(self.device, non_blocking=True)
            self.q_len.index_fill_(0, rows, 0)
            self.slots.index_fill_(0, rows, -1)
            self.kv_len.index_fill_(0, rows, 0)

    def close(self) -> None:
        self.graphs.clear()
        self._pf.clear()
        for r in (self._cur, self._waits, self._win, self._status):
            if r is not None:
                r.free()
        try:
            self.C.set_wait_policy(0, 0.0)
            self.C.peer_free(self._abort_word)
        except Exception:
            pass
        self.mesh.close()
