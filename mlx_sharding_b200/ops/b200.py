"""``b200`` op backend: the hand-written sm_100a kernels behind the same API as ``ops.reference``.

Loading is strict: if the extension is missing (or is not loadable) on a box with a GPU this raises —
there is no silent PyTorch fallback on the hot path.  The only non-kernel code here is argument
plumbing (views, dtype checks) and the token->sequence map derived from the step metadata.
"""
from __future__ import annotations

import importlib.util
import os
from typing import Optional, Tuple

import torch

from .meta import BatchMeta
from .weights import LinearWeight, RopeSpec

NAME = "b200"
_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_b200_C.so")
_C = None

ACT_IDS = {"none": 0, "silu": 1, "gelu_tanh": 2, "gelu_pytorch_tanh": 2, "gelu_approx": 2}


def load_extension(build_if_missing: bool = False):
    """Import the in-tree ``_b200_C.so`` (optionally building it first with ``ops/build.py``)."""
    global _C
    if _C is not None:
        return _C
    if not os.path.exists(_SO):
        if build_if_missing:
            from .build import build

            build()
        else:
            raise ImportError(
                f"{_SO} not found: build the sm_100a extension with `python -m mlx_sharding_b200.ops.build` "
                "(or __graft_entry__.build())")
    spec = importlib.util.spec_from_file_location("_b200_C", _SO)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _C = mod
    if torch.cuda.is_available():
        # persistent scratch (split-K / attention-split workspace, tile tickets) must exist before any
        # CUDA-graph capture
        mod.init_scratch(torch.cuda.current_device(), 32 << 20)
    return _C


def C():
    return load_extension()


def is_available() -> bool:
    return os.path.exists(_SO) and torch.cuda.is_available()


def _bf16(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.bfloat16:
        raise TypeError(f"b200 backend runs bf16 activations/weights, got {t.dtype}")
    return t


def _dense(W: LinearWeight) -> torch.Tensor:
    """bf16 ``[.., N, K]`` view of a weight.  Only used for bf16 checkpoints and for quantised layouts the in-kernel
    dequant GEMM does not cover (2-bit, odd group sizes; expert-parallel banks): those are expanded once at
    first use.  int4 / int8 group-64/128 weights take :func:`_qpack` and stay packed in HBM."""
    if W.is_quantized:
        if W.weight is None:
            W.weight = W.dense(torch.bfloat16).contiguous()
        return W.weight
    return _bf16(W.weight)


_qpack_warned = []


def _qpack(W: LinearWeight):
    """(packed int32 codes [rows, words], scales_t, biases_t [K/g, rows]) for the in-kernel dequant GEMM, or None
    when the layout is not supported by the kernel (then the weight is expanded to bf16 once)."""
    if not W.is_quantized:
        return None
    qt = getattr(W, "_qt", None)
    if qt is None:
        K = W.in_features
        if not C().gemm_q_supported(W.bits, W.group_size, K) or W.scales.dtype != torch.bfloat16:
            if W.scales.dtype != torch.bfloat16 and not _qpack_warned:
                import logging

                logging.getLogger(__name__).warning(
                    "quantised weights with %s scale tables: the in-kernel dequant GEMM takes bf16 tables, so these weights are "
                    "dequantised exactly (stored-precision scales) to bf16 once at first use instead", W.scales.dtype)
                _qpack_warned.append(True)
            W._qt = False
            return None
        rows = W.wq.numel() // W.wq.shape[-1]
        ng = K // W.group_size
        wq = W.wq.reshape(rows, W.wq.shape[-1]).contiguous()
        if W.bits == 4:
            # load-time re-pack (same bits, kernel-friendly order): nibble j <- code 2j, nibble 4+j <- code 2j+1, so the
            # kernel's (w >> 4i) & 0x000F000F yields the adjacent pair (v_2i, v_2i+1) directly
            from ..utils import quant as _q

            wq = _q.repack_int4_pairs(wq).contiguous()
        st = W.scales.reshape(rows, ng).t().contiguous()
        bt = W.biases.reshape(rows, ng).t().contiguous()
        qt = (wq, st, bt)
        W._qt = qt
    return qt or None


# ------------------------------------------------------------------------------------------------ ops
def embed(ids: torch.Tensor, emb: LinearWeight, scale: float = 1.0, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    ids = ids.to(torch.int64).contiguous()
    if emb.is_quantized:
        return C().embed(ids, emb.wq, emb.scales, emb.biases, emb.bits, emb.group_size, float(scale))
    return C().embed(ids, _bf16(emb.weight), None, None, 0, 64, float(scale))


def rmsnorm(x, w, eps: float, gemma: bool = False, residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
            signal: Optional[Tuple[int, int]] = None):
    """``out`` / ``signal``: fused stage boundary — the norm stores straight into the next stage's inbox (peer memory) and the
    last CTA raises its flag (Gemma-2 stages end in a norm, not in a GEMM)."""
    flag, val = signal if signal is not None else (0, 0)
    return C().rmsnorm(x, w, float(eps), bool(gemma), residual, out, int(flag), int(val))


def add_rmsnorm(x, residual, w, eps, gemma=False):
    h = x + residual
    return rmsnorm(h, w, eps, gemma), h


def linear(x: torch.Tensor, W: LinearWeight, residual: Optional[torch.Tensor] = None,
           out_dtype: Optional[torch.dtype] = None, out: Optional[torch.Tensor] = None,
           signal: Optional[Tuple[int, int]] = None, softcap: float = 0.0) -> torch.Tensor:
    fp32 = out_dtype == torch.float32
    flag, val = signal if signal is not None else (0, 0)
    q = _qpack(W)
    if q is not None:
        return C().linear_q(x, q[0], q[1], q[2], None, None, None, W.bits, W.group_size, W.out_features, residual, W.bias, 0,
                            float(softcap), fp32, out, 0, int(flag), int(val))
    return C().linear(x, _dense(W), None, residual, W.bias, 0, float(softcap), fp32, out, 0, int(flag), int(val))


def gated_up(x: torch.Tensor, Wg: LinearWeight, Wu: LinearWeight, act: str = "silu") -> torch.Tensor:
    if Wg.bias is not None or Wu.bias is not None:
        raise NotImplementedError("gated MLP with bias")
    qg, qu = _qpack(Wg), _qpack(Wu)
    if qg is not None and qu is not None:
        return C().linear_q(x, qg[0], qg[1], qg[2], qu[0], qu[1], qu[2], Wg.bits, Wg.group_size, Wg.out_features, None, None,
                            ACT_IDS[act], 0.0, False, None, 0, 0, 0)
    return C().linear(x, _dense(Wg), _dense(Wu), None, None, ACT_IDS[act], 0.0, False, None, 0, 0, 0)


def rope_(x: torch.Tensor, positions: torch.Tensor, spec: RopeSpec, rot_offset: int = 0) -> torch.Tensor:
    C().rope_(x, positions, spec.inv_freq, int(rot_offset), int(spec.rot_dim), bool(spec.interleaved), float(spec.mscale))
    return x


def kv_write(k, v, kpool, vpool, slot_mapping):
    C().kv_write(k, v, kpool, vpool, slot_mapping)


def kv_write_mla(kv, k_pe, kpool, vpool, slot_mapping, nope: int, vdim: int):
    C().kv_write_mla(kv, k_pe, kpool, vpool, slot_mapping, int(nope), int(vdim))


def _token_seq(meta: BatchMeta) -> torch.Tensor:
    ts = getattr(meta, "_token_seq", None)
    if ts is None:
        if meta.num_tokens == meta.num_seqs:
            ts = torch.arange(meta.num_seqs, dtype=torch.int32, device=meta.positions.device)
        else:
            lens = (meta.cu_seqlens[1:] - meta.cu_seqlens[:-1]).long()
            ts = torch.repeat_interleave(torch.arange(meta.num_seqs, device=lens.device), lens).to(torch.int32)
        meta._token_seq = ts
    return ts


def paged_attention(q, kpool, vpool, meta: BatchMeta, scale: float, softcap: float = 0.0):
    c = C()
    if meta.max_q_len > 1 and not softcap and c.flash_prefill_supported(kpool.shape[3], vpool.shape[3]):
        # prefill chunk / mixed batch: tensor-core causal flash attention over the paged cache
        return c.flash_prefill(q, kpool, vpool, meta.block_tables, meta.cu_seqlens, meta.context_lens, float(scale),
                               int(meta.num_tokens))
    return C().paged_attention(q, kpool, vpool, meta.block_tables, meta.positions, _token_seq(meta), float(scale),
                               float(softcap or 0.0), int(meta.max_ctx_len))


def route_groups(method: str, n_group: int, topk_group: int) -> Tuple[int, int]:
    """``(n_group, topk_group)`` the router kernels run with: group-limited top-k only for ``method == "group_limited_greedy"``,
    one group of all experts for every other method."""
    return (int(n_group), int(topk_group)) if method == "group_limited_greedy" else (1, 1)


def moe_route(x, gate_w, top_k: int, method: str = "greedy", n_group: int = 1, topk_group: int = 1,
              scaling: float = 1.0, norm_topk: bool = False, extra: int = 0):
    """``extra``: always-on experts appended to the routed bank (ids E .. E+extra-1, weight 1.0) — see ``fuse_shared_experts``."""
    n_group, topk_group = route_groups(method, n_group, topk_group)
    idx, w = C().moe_route(x, _bf16(gate_w), int(top_k), int(n_group), int(topk_group), float(scaling), bool(norm_topk), int(extra))
    return idx, w


class _Join:
    """Handle of work forked onto the side stream by :func:`run_aside`; ``wait()`` joins it into the current stream."""

    def __init__(self, event):
        self.event = event

    def wait(self):
        torch.cuda.current_stream().wait_event(self.event)
        C().pdl_skip_next()  # the joining kernel depends on two streams: plain dependencies, no programmatic edge


_side_streams = {}


def run_aside(fn) -> _Join:
    """Run ``fn()`` on this device's side stream, forked from the current stream (event record / wait, so it is also legal
    inside CUDA-graph capture and becomes a parallel branch of the graph).  Used to run the shared-expert GEMMs of a
    DeepSeek MoE block concurrently with the router / permutation / expert all-to-all, which do not depend on them.
    ``fn`` must write its result into a tensor allocated *before* the fork."""
    cur = torch.cuda.current_stream()
    side = _side_streams.get(cur.device.index)
    if side is None:
        side = _side_streams[cur.device.index] = torch.cuda.Stream(device=cur.device)
    fork = torch.cuda.Event()
    fork.record(cur)
    side.wait_event(fork)
    with torch.cuda.stream(side):
        C().pdl_skip_next()  # first side kernel depends on the other stream
        fn()
        done = torch.cuda.Event()
        done.record(side)
    return _Join(done)


def moe_experts(x, idx, w, Wg: LinearWeight, Wu: LinearWeight, Wd: LinearWeight, act: str = "silu",
                extra: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, signal: Optional[Tuple[int, int]] = None, join: Optional[_Join] = None):
    """router output -> permute -> grouped dual GEMM (act(gate)*up) -> grouped down GEMM (fp32) ->
    weighted combine (+ residual [+ P2P store & flag])."""
    c = C()
    T, k = idx.shape
    fp8 = fp8_experts_enabled(Wg) and x.shape[1] % 128 == 0
    qg, qu, qd = (None, None, None) if fp8 else (_qpack(Wg), _qpack(Wu), _qpack(Wd))
    if fp8:
        (gq, gs), (uq, us), (dq, ds) = _fp8pack(Wg), _fp8pack(Wu), _fp8pack(Wd)
        E = gq.shape[0]
        offs, pair_row, xp = c.moe_permute(idx, x, E)
        xq, xsf = c.quant_mxfp8(xp)
        h = c.linear_fp8(xq, xsf, gq, gs, uq, us, offs, T, None, ACT_IDS[act], False, 0, 0)
        hq, hsf = c.quant_mxfp8(h)
        y = c.linear_fp8(hq, hsf, dq, ds, None, None, offs, T, None, 0, True, 0, 0)
    elif qg is not None and qu is not None and qd is not None:
        E = Wg.wq.shape[0]
        offs, pair_row, xp = c.moe_permute(idx, x, E)
        h = c.grouped_linear_q(xp, qg[0], qg[1], qg[2], qu[0], qu[1], qu[2], Wg.bits, Wg.group_size, E, Wg.out_features,
                               offs, T, ACT_IDS[act], False)
        y = c.grouped_linear_q(h, qd[0], qd[1], qd[2], None, None, None, Wd.bits, Wd.group_size, E, Wd.out_features, offs, T,
                               0, True)
    else:
        wg, wu, wd = _dense(Wg), _dense(Wu), _dense(Wd)
        E = wg.shape[0]
        offs, pair_row, xp = c.moe_permute(idx, x, E)
        h = c.grouped_linear(xp, wg, wu, offs, T, ACT_IDS[act], False)
        y = c.grouped_linear(h, wd, None, offs, T, 0, True)
    if extra is not None:
        residual = extra if residual is None else residual + extra
    flag, val = signal if signal is not None else (0, 0)
    if join is not None:
        join.wait()  # ``residual`` is produced on the side stream (shared experts)
    return c.moe_combine(y, pair_row, w, residual, out, int(k), int(flag), int(val))


def quant_mxfp8(x: torch.Tensor):
    """bf16 activations ``[R, K]`` -> (e4m3 bytes, ue8m0 scales per 32 K-values): the B operand of the block-scaled FP8 GEMMs."""
    return C().quant_mxfp8(x)


def _fp8pack(W: LinearWeight):
    """MXFP8 form of a weight (``utils/quant.py::to_mxfp8``), built once on first use from the dense / dequantised values; the
    source tensors (bf16 bank or packed MLX codes) are released — afterwards the weight lives in HBM as 1.03 bytes per parameter."""
    f = getattr(W, "_fp8", None)
    if f is None:
        from ..utils.quant import to_mxfp8

        src = W.dense(torch.bfloat16) if W.is_quantized else W.weight
        qs, sfs = [], []
        for chunk in (src.split(8) if src.dim() == 3 else [src]):     # bound the fp32 temporaries of the conversion
            q, sf = to_mxfp8(chunk)
            qs.append(q); sfs.append(sf)
        f = W._fp8 = (torch.cat(qs).contiguous(), torch.cat(sfs).contiguous())
        W.fp8_shape = tuple(src.shape)
        W.weight = W.wq = W.scales = W.biases = None
    return f


def fp8_experts_enabled(W: LinearWeight) -> bool:
    """Block-scaled FP8 expert banks.  The stage model converts at load (MLX 4/8-bit checkpoints by default, bf16 checkpoints with
    MLXB200_FP8_EXPERTS=1; ``models/deepseek_v2.py::_convert_quantized_for_b200``); packed MLX weights handed to the ops directly
    always take the exact in-kernel dequant GEMMs."""
    if getattr(W, "_fp8", None) is not None:
        return True                      # converted at load (models/deepseek_v2.py::_convert_quantized_for_b200)
    return os.environ.get("MLXB200_FP8_EXPERTS", "") == "1" and not W.is_quantized   # explicit opt-in for bf16 banks used directly


_scatter_bufs = {}
SCATTER_MAX_TOKENS = 128


def moe_block(x, gate_w, route_kw: dict, Wg: LinearWeight, Wu: LinearWeight, Wd: LinearWeight, act: str = "silu",
              residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, signal: Optional[Tuple[int, int]] = None,
              extra: int = 0, pre_norm: Optional[Tuple[torch.Tensor, float]] = None,
              next_norm: Optional[Tuple[torch.Tensor, float]] = None):
    """Router + routed (and appended shared) experts of one MoE block.

    ``pre_norm = (weight, eps)``: ``x`` is the un-normalised residual stream and the block starts with ``rmsnorm(x) * weight`` — on
    the scatter path the router kernel normalises the row in shared memory (no norm kernel).  ``next_norm = (weight, eps)``: the
    block also returns ``rmsnorm(result) * weight`` (the next layer's input norm), fused into the combine kernel on the scatter
    path; the return value is then ``(result, normed)``.

    Decode-sized batches (``T <= SCATTER_MAX_TOKENS``) with bf16 or FP8 banks take the *scatter* path: the router kernel claims a
    slot per (token, expert) pair in the expert's fixed-stride segment and copies the token row there itself, the grouped GEMMs
    read per-expert row counts — route / counting sort / gather are ONE launch, the block is router -> grouped gate-up -> grouped
    down -> combine.  Larger batches (prefill) and packed-integer banks keep the compact counting-sort permutation, with the
    norms as separate kernels."""
    c = C()
    T = x.shape[0]
    fp8 = fp8_experts_enabled(Wg) and x.shape[1] % 128 == 0
    quant = (Wg.is_quantized or Wu.is_quantized or Wd.is_quantized) and not fp8
    if quant or T > SCATTER_MAX_TOKENS:
        if pre_norm is not None:
            x = rmsnorm(x, pre_norm[0], pre_norm[1])
        idx, wts = moe_route(x, gate_w, extra=extra, **route_kw)
        res = moe_experts(x, idx, wts, Wg, Wu, Wd, act, residual=residual, out=out, signal=signal)
        return res if next_norm is None else (res, rmsnorm(res, next_norm[0], next_norm[1]))
    if fp8:
        (gq, gs), (uq, us), (dq, ds) = _fp8pack(Wg), _fp8pack(Wu), _fp8pack(Wd)
        E, H = gq.shape[0], x.shape[1]
    else:
        wg, wu, wd = _dense(Wg), _dense(Wu), _dense(Wd)
        E, H = wg.shape[0], x.shape[1]
    stride = 64 if T <= 64 else SCATTER_MAX_TOKENS
    key = (x.device.index, E, H, stride)
    bufs = _scatter_bufs.get(key)
    if bufs is None:
        # persistent (graph-safe) per-device buffers: row counters (zero between blocks: the combine resets them) + scattered rows
        bufs = _scatter_bufs[key] = (torch.zeros(E, dtype=torch.int32, device=x.device),
                                     torch.empty(E * stride, H, dtype=torch.bfloat16, device=x.device))
    counts, xs = bufs
    rk = route_kw
    n_group, topk_group = route_groups(rk.get("method", "greedy"), rk.get("n_group", 1), rk.get("topk_group", 1))
    nw, ne = (_bf16(pre_norm[0]), float(pre_norm[1])) if pre_norm is not None else (None, 1e-6)
    idx, wts, pair_row = c.moe_route(x, _bf16(gate_w), int(rk["top_k"]), n_group, topk_group, float(rk["scaling"]),
                                     bool(rk["norm_topk"]), int(extra), counts, stride, xs, nw, ne)
    k = idx.shape[1]
    if fp8:
        # block-scaled FP8 experts: activations are quantised per 32-wide K block right before each GEMM (garbage rows beyond an
        # expert's count are quantised too and never read); tcgen05 kind::mxf8f6f4.block_scale applies both operands' scales
        xq, xsf = c.quant_mxfp8(xs)
        h = c.linear_fp8(xq, xsf, gq, gs, uq, us, counts, stride, None, ACT_IDS[act], False, T * k, stride)
        hq, hsf = c.quant_mxfp8(h)
        y = c.linear_fp8(hq, hsf, dq, ds, None, None, counts, stride, None, 0, True, T * k, stride)
    else:
        h = c.grouped_linear(xs, wg, wu, counts, stride, ACT_IDS[act], False, None, None, None, T * k, stride)
        y = c.grouped_linear(h, wd, None, counts, stride, 0, True, None, None, None, T * k, stride)
    flag, val = signal if signal is not None else (0, 0)
    if next_norm is not None and signal is None and H <= 8192:   # (the fused combine-norm kernel holds a row of up to 8192)
        normed = torch.empty(T, H, dtype=torch.bfloat16, device=x.device)
        res = c.moe_combine(y, pair_row, wts, residual, out, int(k), 0, 0, counts, _bf16(next_norm[0]), float(next_norm[1]), normed)
        return res, normed
    res = c.moe_combine(y, pair_row, wts, residual, out, int(k), int(flag), int(val), counts)
    return res if next_norm is None else (res, rmsnorm(res, next_norm[0], next_norm[1]))


def softcap_(logits, cap: float):
    return torch.tanh(logits / cap) * cap


def apply_penalties_(logits, rep_ctx, penalty, bias_idx, bias_val):
    C().apply_penalties_(logits, rep_ctx.contiguous(), penalty, bias_idx.contiguous(), bias_val.contiguous())
    return logits


_step = [0]


def sample(logits, temperature, top_p, generator: Optional[torch.Generator] = None, top_logprobs: int = 0):
    seed = generator.initial_seed() if generator is not None else 0
    _step[0] += 1
    toks, lp, ti, tl = C().sample(logits.contiguous(), temperature, top_p, int(seed) & 0x7FFFFFFFFFFFFFFF, _step[0],
                                  int(top_logprobs))
    if top_logprobs > 0:
        return toks, lp, ti, tl
    return toks, lp, None, None


def mla_absorbed_supported(num_heads: int, kv_lora_rank: int, rope_dim: int, page_size: int = 64) -> bool:
    """Shapes the tcgen05 absorbed-latent MLA decode kernel is built for (DeepSeek-V2 / V2-Lite / Coder-V2-Lite)."""
    return num_heads == 16 and kv_lora_rank == 512 and rope_dim == 64 and page_size == 64


def mla_absorbed_prologue(q, ckv, k_pe, norm_w, eps: float, pool, meta: BatchMeta, spec: RopeSpec):
    """latent = RMSNorm(c_kv) -> pool[slot][:512], rope(k_pe) -> pool[slot][512:], rope(q_pe) in place: one launch."""
    C().mla_absorbed_prologue(q, ckv, k_pe, norm_w, float(eps), pool, meta.slot_mapping, meta.positions, spec.inv_freq, float(spec.mscale))


def mla_decode(q, pool, meta: BatchMeta, scale: float, nsplit: int = 0):
    """Multi-query attention over the cached latent (d_qk 576 / d_v 512) on tcgen05: ``[B, 16, 576] -> [B, 16, 512]``."""
    return C().mla_decode(q, pool, meta.block_tables, meta.context_lens, float(scale), int(meta.max_ctx_len), int(nsplit))


def sample_block(logits, sv, tag_out, toks_out, lp_out, top_ids_out, top_lp_out):
    """Sampling driven by a step block in device memory (``parallel/graph_decode.py``): every per-step input — temperatures,
    nucleus thresholds, per-request (seed, step) RNG state, penalty contexts, bias tables, the step tag — is read by the kernels
    from the block, so the same captured CUDA graph serves greedy and sampled requests."""
    logits = logits.contiguous()
    if sv.has_pen:
        C().apply_penalties_(logits, sv.rep, sv.penalty, sv.bidx, sv.bval)
    k = 0 if top_ids_out is None else int(top_ids_out.shape[1])
    C().sample_into(logits, sv.temps, sv.top_p, sv.rng, k, toks_out, lp_out, top_ids_out, top_lp_out, sv.tag, tag_out)


def mla_rope_kv_write(q, k_pe, kv, kpool, vpool, meta: BatchMeta, spec: RopeSpec, nope: int, vdim: int):
    if not spec.interleaved:
        raise NotImplementedError("fused MLA prologue expects interleaved (traditional) rope pairs")
    C().mla_rope_kv_write(q, k_pe, kv, kpool, vpool, meta.slot_mapping, meta.positions, spec.inv_freq, float(spec.mscale),
                          int(nope), int(vdim))
