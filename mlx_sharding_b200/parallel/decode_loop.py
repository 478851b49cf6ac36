"""Graph-captured steady-state decode: one CUDA-graph launch per stage per micro-batch step.

The reference's per-token loop is host driven end to end (``mx.async_eval`` one-token look-ahead, N
blocking RPCs per token, shard/utils.py:156-186).  Here a decode step of a micro-batch group is a
*device-resident program*: the step metadata (positions, KV slots, context lengths) lives in static
device buffers and is advanced by a tiny kernel, sampled tokens feed the next step on device, and stage
hand-offs are the fused P2P stores of ``p2p_fused.py`` (or NCCL p2p as the baseline transport).  The
host only replays graphs; with ``num_groups == num_stages`` every stage always has a group to work on
(micro-batched token scheduling, SURVEY §2.4 / BASELINE config 3).

Per-stage graph of group ``g`` (fused transport):

    rank 0   : wait(token flag g) -> embed(token inbox g) -> layers -> [last kernel stores into rank 1's inbox g, flag++]
    rank r   : wait(hidden flag g) -> layers on inbox g        -> [last kernel stores into rank r+1's inbox g, flag++]
    last rank: wait(hidden flag g) -> layers -> norm -> LM head -> sample -> copy tokens to rank 0's token inbox g, flag++
    every rank: advance_meta(g)

All ranks replay the groups in the same global order, so every wait points at work that is earlier in
that order on another GPU — no cyclic waits.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.distributed as dist

from ..ops.meta import BatchMeta


class GroupState:
    """Static device buffers of one micro-batch group on one stage."""

    def __init__(self, B: int, max_blocks: int, page_size: int, device):
        i32 = dict(dtype=torch.int32, device=device)
        self.B = B
        self.positions = torch.zeros(B, **i32)
        self.slot_mapping = torch.zeros(B, **i32)
        self.context_lens = torch.zeros(B, **i32)
        self.block_tables = torch.zeros(B, max_blocks, **i32)
        self.cu_seqlens = torch.arange(B + 1, **i32)
        self.last_idx = torch.arange(B, **i32)
        self.tokens = torch.zeros(B, dtype=torch.int64, device=device)
        self.page_size = page_size
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.meta: Optional[BatchMeta] = None

    def load(self, positions, block_tables, tokens, max_ctx: int):
        """positions = position of the token each sequence decodes *next* (i.e. current length)."""
        self.positions.copy_(positions.to(torch.int32))
        bt = block_tables.to(torch.int32)
        self.block_tables.zero_()
        self.block_tables[:, : bt.shape[1]].copy_(bt)
        pos = self.positions.long()
        self.slot_mapping.copy_((self.block_tables.gather(1, (pos // self.page_size)[:, None]).squeeze(1).long()
                                 * self.page_size + pos % self.page_size).to(torch.int32))
        self.context_lens.copy_(self.positions + 1)
        if tokens is not None:
            self.tokens.copy_(tokens)
        self.meta = BatchMeta(self.positions, self.slot_mapping, self.cu_seqlens, self.context_lens, self.block_tables,
                              self.last_idx, self.B, self.B, 1, int(max_ctx), self.page_size)


class DecodeLoop:
    """Steady-state decode of ``num_groups`` micro-batch groups on this stage."""

    def __init__(self, stage, num_groups: int, batch: int, max_blocks: int, transport: str = "auto",
                 use_graphs: bool = True, standalone: bool = False):
        """``standalone``: this rank runs the *whole* layer stack on its own sequences (data-parallel attention +
        expert-parallel MoE, ``parallel/ep.py``) — there is no stage hand-off even though ``torch.distributed`` is up."""
        self.stage = stage
        self.model = stage.model
        self.dev = self.model.device
        self.rank = dist.get_rank() if dist.is_initialized() and not standalone else 0
        self.world = dist.get_world_size() if dist.is_initialized() and not standalone else 1
        self.G, self.B = num_groups, batch
        self.page_size = stage.kv.page_size
        self.groups = [GroupState(batch, max_blocks, self.page_size, self.dev) for _ in range(num_groups)]
        self.use_graphs = use_graphs and self.dev.type == "cuda"
        if transport == "auto":
            transport = "fused" if (self.world > 1 and self.model.backend_name == "b200") else "nccl"
        self.transport = transport if self.world > 1 else "local"
        self.p2p = None
        self.launches_per_step = 0
        H = self.model.cfg.hidden_size
        if self.transport == "fused":
            from .p2p_fused import FusedP2PBoundary

            self.p2p = FusedP2PBoundary(H, num_groups, batch, batch)
        elif self.transport == "nccl":
            self.hidden_in = [torch.zeros(batch, H, dtype=self.model.dtype, device=self.dev) for _ in range(num_groups)]
        self.temps = torch.zeros(batch, device=self.dev)
        self.top_p = torch.ones(batch, device=self.dev)
        self.first, self.last = self.rank == 0, self.rank == self.world - 1

    # ------------------------------------------------------------------------------------------ one step body
    def _body(self, g: int):
        """Device work of one decode step of group ``g`` on this stage (captured or eager)."""
        st, m, O = self.groups[g], self.model, self.model.ops
        C = self.p2p.C if self.p2p is not None else None
        if self.transport == "fused":
            if self.first:
                self.p2p.wait_tokens(g)
                x = self.p2p.token_inbox(g, self.B)
            else:
                self.p2p.wait_hidden(g)
                x = self.p2p.hidden_inbox(g, self.B)
            if not self.last:
                m.boundary = (self.p2p.next_hidden(g, self.B), self.p2p.next_hidden_flag(g))
        else:
            x = st.tokens if self.first else self.hidden_in[g]
        out = m.forward(x, st.meta, self.stage.kv)
        m.boundary = None
        if self.last:
            toks, _, _, _ = O.sample(out, self.temps, self.top_p, None, 0)
            if self.transport == "fused":
                self.p2p.send_tokens(toks, g)
            else:
                st.tokens.copy_(toks)
        elif self.transport == "fused" and not m.boundary_fused:
            self.p2p.send_hidden(out, g)  # the stage's last kernel has no fused epilogue (Gemma-2 ends in a norm): copy + signal
        if self.dev.type == "cuda" and m.backend_name == "b200":
            O.C().advance_meta(st.positions, st.context_lens, st.slot_mapping, st.block_tables, self.page_size)
        else:
            st.positions += 1
            st.context_lens += 1
            pos = st.positions.long()
            st.slot_mapping.copy_((st.block_tables.gather(1, (pos // self.page_size)[:, None]).squeeze(1).long()
                                   * self.page_size + pos % self.page_size).to(torch.int32))
        return out

    def _nccl_pre(self, g: int):
        if self.transport != "nccl":
            return
        if self.first:
            if self._steps_done[g] > 0:
                dist.recv(self.groups[g].tokens, self.world - 1)
        else:
            dist.recv(self.hidden_in[g], self.rank - 1)

    def _send(self, t: torch.Tensor, dst: int):
        """NCCL sends are stream-ordered and return immediately; gloo's ``send`` blocks until the peer posts the matching
        ``recv``, which would dead-lock the ring (rank r sends group g+1 forward while the last rank sends group g's tokens
        back) — on gloo the send is posted asynchronously and completed in ``drain`` / before the buffer is reused."""
        if dist.get_backend() != "gloo":
            dist.send(t, dst)
            return
        self._sends = [(w, keep) for w, keep in getattr(self, "_sends", []) if not w.is_completed()]
        keep = t.clone()
        self._sends.append((dist.isend(keep, dst), keep))

    def _nccl_post(self, g: int, out):
        if self.transport != "nccl":
            return
        if self.last:
            self._send(self.groups[g].tokens, 0)
        else:
            self._send(out, self.rank + 1)

    # ------------------------------------------------------------------------------------------ setup
    def prime_tokens(self):
        """Fused transport: publish the first decode-step tokens of every group into stage 0's token inbox
        (rank 0 does it locally; counts as hand-off #1 of each group)."""
        if self.transport == "fused" and self.first:
            for g in range(self.G):
                self.p2p.C.copy_signal(self.groups[g].tokens, self.p2p._token_ptr(self.p2p.base, g),
                                       self.p2p._flag_ptr(self.p2p.base, g, 1), 0)

    def capture(self, warmup: int = 0):
        """Capture one graph per group.  NCCL transport keeps send/recv outside the graph."""
        self._steps_done = [0] * self.G
        self._outs = [None] * self.G
        if not self.use_graphs:
            return
        from ..ops import b200 as _b

        for g in range(self.G):
            st = self.groups[g]
            snap = [t.clone() for t in (st.positions, st.context_lens, st.slot_mapping, st.tokens)]
            if self.transport != "fused":
                # eager warm-up (allocates scratch, sets func attributes) on a side stream, then capture
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    self._body(g)
                torch.cuda.current_stream().wait_stream(s)
                for t, v in zip((st.positions, st.context_lens, st.slot_mapping, st.tokens), snap):
                    t.copy_(v)
            graph = torch.cuda.CUDAGraph()
            n0 = _b.C().launch_count()
            with torch.cuda.graph(graph):
                self._outs[g] = self._body(g)
            self.launches_per_step = _b.C().launch_count() - n0
            st.graph = graph
            # capture executes nothing, but the eager warm-up advanced the metadata: it was restored above
        torch.cuda.synchronize()

    def warm_kernels(self):
        """Fused transport cannot run an eager warm-up step (it would consume flags); instead exercise the
        stage once on a scratch group with the boundary disabled so scratch buffers / attributes exist."""
        if self.transport != "fused":
            return
        st = self.groups[0]
        snap = [t.clone() for t in (st.positions, st.context_lens, st.slot_mapping)]
        H = self.model.cfg.hidden_size
        x = st.tokens if self.first else torch.zeros(self.B, H, dtype=self.model.dtype, device=self.dev)
        out = self.model.forward(x, st.meta, self.stage.kv)
        if self.last:
            self.model.ops.sample(out, self.temps, self.top_p, None, 0)
        for t, v in zip((st.positions, st.context_lens, st.slot_mapping), snap):
            t.copy_(v)
        torch.cuda.synchronize()

    # ------------------------------------------------------------------------------------------ run
    def step_all(self):
        """One decode step of every group (each sequence of every group emits one token)."""
        for g in range(self.G):
            self._nccl_pre(g)
            if self.use_graphs:
                self.groups[g].graph.replay()
                out = self._outs[g]
            else:
                out = self._outs[g] = self._body(g)
            self._nccl_post(g, out)
            self._steps_done[g] += 1

    def drain(self):
        """NCCL transport: stage 0 still has one token message per group in flight after the last step."""
        if self.transport == "nccl" and self.first and self.world > 1:
            for g in range(self.G):
                dist.recv(self.groups[g].tokens, self.world - 1)
        for w, _ in getattr(self, "_sends", []):
            w.wait()
        self._sends = []
