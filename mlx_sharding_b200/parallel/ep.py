"""Expert parallelism for DeepSeek MoE blocks with a fused all-to-all over NVSwitch peer memory
(BASELINE config 5; SURVEY §2.4 "EP", K11-EP).

The reference executes all routed experts of a layer on the stage that owns the layer (``mx.gather_qmm``).
``ExpertParallelMoE`` shards the ``E`` routed experts of a layer across the ``world`` ranks of one NVSwitch
domain: rank ``r`` keeps experts ``[r*E/world, (r+1)*E/world)`` (1/world of the MoE weights — the dominant
HBM stream of a decode step) and every rank routes *its own* tokens.  Token exchange is done by the kernels
in ``ops/csrc/ep.cu`` — dispatch rows are written straight into the owner's receive region, expert outputs
are stored straight into the source's return buffer by the down-projection GEMM epilogue, publication words /
flags use release/acquire at system scope; there is no NCCL call and no host involvement on the path.

``forward(x, idx, w, residual)`` == ``ops.moe_experts`` on the un-sharded weights (verified in
``tests/test_multigpu.py``).
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.distributed as dist

from ..ops.weights import LinearWeight


class EPBuffers:
    """IPC-mapped receive / return buffers of one rank (shared by all MoE layers of that rank).

    Receive side: an expert-major buffer of ``[experts_per_rank][world * max_tokens][H]`` bf16 rows, the return address of every
    row (u64), two parity-buffered sets of per-expert row counters and one arrival word per source.  Return side: ``[max_tokens *
    top_k][H]`` fp32 rows (one per routed pair of this rank) and the return flag."""

    def __init__(self, hidden: int, max_tokens: int, top_k: int, experts_per_rank: int, group=None):
        from ..ops import b200

        self.C = b200.load_extension()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.dev = torch.cuda.current_device()
        self.H, self.top_k = hidden, top_k
        self.max_tokens = max_tokens
        self.E_local = experts_per_rank
        self.cap = max_tokens * top_k                      # pairs one rank routes per step (rows of its return buffer)
        W, cap, H = self.world, self.cap, hidden
        rows = experts_per_rank * W * max_tokens
        self.off_recv_x = 0
        self.off_recv_meta = self.off_recv_x + rows * H * 2            # -> row_dst table
        self.off_cnt = self.off_recv_meta + rows * 8
        self.off_recv_count = (self.off_cnt + 2 * experts_per_rank * 4 + 255) // 256 * 256   # arrival words: one u64 per source
        self.off_ret_y = (self.off_recv_count + W * 8 + 255) // 256 * 256
        self.off_flags = self.off_ret_y + cap * H * 4
        total = self.off_flags + 256
        self.base, handle = self.C.ipc_alloc(total)
        handles: List = [None] * W
        dist.all_gather_object(handles, (handle, self.dev), group=group)
        self.peer = []
        for r, (h, pdev) in enumerate(handles):
            if r == self.rank:
                self.peer.append(self.base)
            else:
                if pdev != self.dev:
                    self.C.enable_peer_access(pdev)
                self.peer.append(self.C.ipc_open(h))
        # tables of peer addresses
        self.t_recv_x = [p + self.off_recv_x for p in self.peer]
        self.t_recv_meta = [p + self.off_recv_meta for p in self.peer]
        self.t_cnt = [p + self.off_cnt for p in self.peer]
        self.t_recv_count = [p + self.off_recv_count for p in self.peer]
        self.t_ret_flag = [p + self.off_flags + 128 for p in self.peer]
        # my return buffer as mapped by every destination (the address a destination's down-projection epilogue stores to)
        peers_all: List = [None] * W
        dist.all_gather_object(peers_all, list(self.peer), group=group)
        self.t_my_ret = [peers_all[d][self.rank] + self.off_ret_y for d in range(W)]
        self.cnt = self.C.tensor_from_ptr(self.base + self.off_cnt, [2 * experts_per_rank], "int32", self.dev)
        self._views = {}
        # device-resident local state, one int32 word each: dispatch CTAs done | down-GEMM tiles done | return arrivals the
        # combine waits for | dispatch step sequence | error flag
        self.state = torch.zeros(5, dtype=torch.int32, device="cuda")
        self.done, self.tiles, self.ret_expected, self.seq = (self.state[j:j + 1] for j in range(4))
        self.error_ptr = self.state[4:].data_ptr()
        self.ret_y = self.C.tensor_from_ptr(self.base + self.off_ret_y, [cap, H], "float32", self.dev)
        self.ret_flags_dev = torch.tensor(self.t_ret_flag, dtype=torch.int64, device="cuda")   # every source's return flag
        dist.barrier(group=group)

    def error(self) -> bool:
        return bool(self.state[-1].item())

    def stride(self, Tmax: int) -> int:
        """Receive rows per expert for a step in which no rank routes more than ``Tmax`` tokens: ``world * Tmax`` rounded up to 64
        (every rank computes the same value: ranks step in lock-step with equal batch shapes, or share a ``Tmax`` bound)."""
        return min(self.world * self.max_tokens, (self.world * Tmax + 63) // 64 * 64)

    def recv_views(self, stride: int):
        """(rows [E_local * stride, H] bf16, row_dst [E_local * stride] int64) over the receive buffer for this step's stride."""
        v = self._views.get(stride)
        if v is None:
            R = self.E_local * stride
            v = self._views[stride] = (self.C.tensor_from_ptr(self.base + self.off_recv_x, [R, self.H], "bfloat16", self.dev),
                                       self.C.tensor_from_ptr(self.base + self.off_recv_meta, [R], "int64", self.dev))
        return v


class ExpertParallelMoE:
    """One MoE layer's routed experts, sharded over the ranks of ``bufs``.

    A block is four launches: dispatch (slot reservation at the sender) -> grouped gate/up GEMM (acquires the arrivals itself) ->
    grouped down GEMM (epilogue returns the rows) -> combine.  :meth:`forward` dispatches rows that were routed separately;
    :meth:`route_forward` folds the pre-MoE RMSNorm and the router into the dispatch kernel and the next layer's input norm into
    the combine."""

    def __init__(self, bufs: EPBuffers, Wg: LinearWeight, Wu: LinearWeight, Wd: LinearWeight, num_experts: int,
                 act: str = "silu", weights_are_local: bool = False):
        from ..ops import b200

        self.b = bufs
        self.ops = b200
        self.E = num_experts
        assert num_experts % bufs.world == 0
        self.E_local = num_experts // bufs.world
        lo, hi = bufs.rank * self.E_local, (bufs.rank + 1) * self.E_local
        pick = (lambda W: b200._dense(W)) if weights_are_local else (lambda W: b200._dense(W)[lo:hi].contiguous())
        self.wg, self.wu, self.wd = pick(Wg), pick(Wu), pick(Wd)
        self.act = b200.ACT_IDS[act]
        self.peer_tokens_default = 0   # bound of the tokens any rank routes per step when ranks run different batch sizes

    def forward(self, x: torch.Tensor, idx: torch.Tensor, w: torch.Tensor, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, peer_tokens: Optional[int] = None, join=None) -> torch.Tensor:
        """``peer_tokens``: upper bound of the tokens *any* rank routes in this step (default: this rank's own ``T`` —
        ranks stepping in lockstep with equal batch shapes); sizes the receive stride of the local expert GEMMs."""
        b = self.b
        T, k = idx.shape

        def dispatch(stride):
            b.C.ep_dispatch_scatter(x, idx, self.E_local, b.rank, stride, b.t_recv_x, b.t_recv_meta, b.t_cnt, b.t_recv_count,
                                    b.t_my_ret, b.seq, b.done, b.ret_expected)
            return w, residual, join

        return self._exchange(T, k, max(T, peer_tokens or self.peer_tokens_default), dispatch, out)

    def route_forward(self, h, gate_w, route_kw: dict, pre_norm, residual_fn, out=None, next_norm=None):
        """The whole block for ``1 <= T <= 1024``: the router with the pre-MoE RMSNorm and the dispatch folded in (``moe.cu``: the
        token's CTA reserves its pairs' slots on the owners with remote atomics, stores the normalised row there and takes part in
        the publication), then the experts and the combine with the next layer's input norm folded in.

        ``h``: un-normalised residual stream; ``pre_norm = (weight, eps)``; ``residual_fn(normed)`` -> ``(residual, join)``: called
        right after the router so the shared-expert branch (which consumes ``normed``) forks onto the side stream behind it;
        ``next_norm = (weight, eps)`` or None.  Returns ``out`` or ``(out, normed_next)``."""
        b, O = self.b, self.ops
        T = h.shape[0]
        k = int(route_kw["top_k"])
        assert 1 <= T <= 1024, "the fused router + dispatch kernel takes 1 <= T <= 1024 tokens"
        rk = route_kw
        n_group, topk_group = O.route_groups(rk.get("method", "greedy"), rk.get("n_group", 1), rk.get("topk_group", 1))
        normed = torch.empty_like(h)

        def dispatch(stride):
            idx, w = b.C.ep_route_dispatch(h, O._bf16(gate_w), k, n_group, topk_group, float(rk["scaling"]), bool(rk["norm_topk"]),
                                           self.E_local, b.rank, stride, b.t_recv_x, b.t_recv_meta, b.t_cnt, b.t_recv_count,
                                           b.t_my_ret, b.seq, b.done, b.ret_expected, O._bf16(pre_norm[0]), float(pre_norm[1]),
                                           normed)
            return (w, *residual_fn(normed))

        return self._exchange(T, k, max(T, self.peer_tokens_default), dispatch, out, next_norm)

    def _exchange(self, T, k, Tmax, dispatch, out, next_norm=None):
        """``dispatch(stride)`` -> ``(w, residual, join)``, then the grouped GEMMs on the received rows and the combine."""
        b, C, W = self.b, self.b.C, self.b.world
        assert T * k <= b.cap, "token batch exceeds the EP buffer capacity"
        stride = b.stride(Tmax)
        rows, row_dst = b.recv_views(stride)
        w, residual, join = dispatch(stride)
        max_rows = min(W * Tmax, stride)
        arrive = (stride, b.base + b.off_recv_count, b.seq, b.error_ptr, W)
        hmid = C.grouped_linear(rows, self.wg, self.wu, b.cnt, max_rows, self.act, False, None, None, None, T * k, *arrive, True)
        C.grouped_linear(hmid, self.wd, None, b.cnt, max_rows, 0, True, row_dst, b.ret_flags_dev, b.tiles, T * k, *arrive, False)
        if join is not None:
            join.wait()  # ``residual`` (shared-expert branch) is produced on the side stream
        combine = (b.base + b.off_flags + 128, b.ret_expected, b.error_ptr, b.ret_y, w, residual, out)
        if next_norm is None:
            return C.ep_combine(*combine)
        H = b.H
        if H <= 8192:   # (the fused combine-norm kernel holds a row of up to 8192)
            nxt = torch.empty(T, H, dtype=torch.bfloat16, device=w.device)
            return C.ep_combine(*combine, self.ops._bf16(next_norm[0]), float(next_norm[1]), nxt), nxt
        res = C.ep_combine(*combine)
        return res, self.ops.rmsnorm(res, next_norm[0], next_norm[1])


class ExpertParallelMoERef:
    """Backend-agnostic expert parallelism: the same exchange expressed with ``torch.distributed.all_to_all_single`` (gloo on
    CPU, NCCL on GPU) and the ``ops.reference`` expert math.  It is the CPU path of ``enable_expert_parallel`` (tests, plumbing
    without a GPU) and the NCCL baseline the fused kernels of ``ops/csrc/ep.cu`` are compared against.

    Same contract as :class:`ExpertParallelMoE`: ``forward(x, idx, w, residual)`` == ``ops.moe_experts`` on the un-sharded
    weights; every rank must call it the same number of times (token counts may differ per rank)."""

    def __init__(self, Wg: LinearWeight, Wu: LinearWeight, Wd: LinearWeight, num_experts: int, act: str = "silu",
                 weights_are_local: bool = False, group=None):
        from ..ops import reference as R

        self.R, self.group, self.act = R, group, act
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        assert num_experts % self.world == 0
        self.E, self.E_local = num_experts, num_experts // self.world
        lo, hi = self.rank * self.E_local, (self.rank + 1) * self.E_local
        pick = (lambda W: W) if weights_are_local else (lambda W: W.slice_experts(lo, hi))
        self.wg, self.wu, self.wd = pick(Wg), pick(Wu), pick(Wd)

    def _a2a(self, send: torch.Tensor, send_counts: List[int], recv_counts: List[int]) -> torch.Tensor:
        recv = send.new_empty((sum(recv_counts),) + tuple(send.shape[1:]))
        dist.all_to_all_single(recv, send.contiguous(), recv_counts, send_counts, group=self.group)
        return recv

    def forward(self, x: torch.Tensor, idx: torch.Tensor, w: torch.Tensor, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, peer_tokens: Optional[int] = None, join=None) -> torch.Tensor:
        T, k = idx.shape
        W, R = self.world, self.R
        flat = idx.reshape(-1).long()
        dst = flat // self.E_local
        order = torch.argsort(dst, stable=True)                       # pairs grouped by destination rank
        send_counts = torch.bincount(dst, minlength=W)
        recv_counts = torch.empty_like(send_counts)
        dist.all_to_all_single(recv_counts, send_counts, group=self.group)
        sc, rc = send_counts.tolist(), recv_counts.tolist()
        rows = self._a2a(x[order // k], sc, rc)                       # token rows, one per (token, expert) pair
        local_e = self._a2a((flat[order] % self.E_local).to(torch.int64), sc, rc)
        # my experts on what I received (fp32 output rows, weight 1: the routing weight is applied by the source)
        y = torch.zeros(rows.shape[0], x.shape[1], dtype=torch.float32, device=x.device)
        for e in range(self.E_local):
            sel = torch.where(local_e == e)[0]
            if sel.numel():
                h = R.gated_up(rows[sel], self.wg.select_expert(e), self.wu.select_expert(e), self.act)
                y[sel] = R.linear(h, self.wd.select_expert(e), out_dtype=torch.float32)
        back = self._a2a(y, rc, sc)                                    # rows return in the order they were sent
        pair_y = torch.empty_like(back)
        pair_y[order] = back
        res = (pair_y.view(T, k, -1) * w.float().unsqueeze(-1)).sum(1)
        if residual is not None:
            res = res + residual.float()
        res = res.to(x.dtype)
        if out is not None:
            out.copy_(res)
            return out
        return res


def enable_expert_parallel(model, max_tokens: int = 256, group=None):
    """Switch a DeepSeek-V2 stage model (every rank holding the *same* layers, data-parallel over tokens) to
    expert-parallel execution: each MoE layer keeps only its ``E / world`` local experts and routes tokens through the
    expert all-to-all — the fused NVLink kernels (:class:`ExpertParallelMoE`) on the ``b200`` backend, ``all_to_all`` collectives
    (:class:`ExpertParallelMoERef`) on the reference backend.  Models loaded with ``expert_shard=(rank, world)``
    (``utils/loader.py``) already hold just their slice; otherwise the full banks are sliced here and dropped from this rank
    afterwards (1/world of the MoE memory).  Returns the :class:`EPBuffers` (``None`` on the reference backend)."""
    cfg = model.cfg
    local = getattr(model, "expert_shard", None) is not None
    if local:
        assert tuple(model.expert_shard) == (dist.get_rank(group), dist.get_world_size(group)), \
            "model was loaded for a different expert shard"
    if hasattr(model, "unfuse_shared_experts"):
        model.unfuse_shared_experts()     # shared experts were appended to the (un-sharded) routed bank: split them off again
    fused = model.backend_name == "b200"
    world = dist.get_world_size(group)
    bufs = EPBuffers(cfg.hidden_size, max_tokens, cfg.num_experts_per_tok, group=group,
                     experts_per_rank=cfg.n_routed_experts // world) if fused else None
    model.ep_layers = {}
    for i, w in model.layer_weights.items():
        if "router" not in w:
            continue
        if fused:
            model.ep_layers[i] = ExpertParallelMoE(bufs, w["e_gate"], w["e_up"], w["e_down"], cfg.n_routed_experts,
                                                   weights_are_local=local)
        else:
            model.ep_layers[i] = ExpertParallelMoERef(w["e_gate"], w["e_up"], w["e_down"], cfg.n_routed_experts,
                                                      weights_are_local=local, group=group)
        for k in ("e_gate", "e_up", "e_down"):
            w[k] = None  # the (sliced) bank lives on in the expert-parallel layer object
    if fused:
        torch.cuda.empty_cache()
    return bufs
