"""Stage-model base: a contiguous layer range of a decoder-only transformer.

Reference mapping: ``IdentityBlock`` (shard/server/model/base.py:6-8) keeps ``layers`` full-length so
layer / cache indices line up; here ``layers`` is also full-length (``None`` marks layers owned by
another stage) but KV storage is only allocated for the local layers.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

from ..config import ModelConfig, ShardSpec, yarn_get_mscale
from ..ops import BatchMeta, LinearWeight, RopeSpec, default_backend_name, get_backend


class IdentityBlock:
    """Placeholder for a layer that lives on another stage (reference base.py:6-8)."""

    def __call__(self, x, *args, **kwargs):
        return x


# --------------------------------------------------------------------------------------------- rope
def default_inv_freq(dim: int, base: float) -> torch.Tensor:
    return 1.0 / (base ** (torch.arange(0, dim, 2, dtype=torch.float32) / dim))


def llama_rope_spec(cfg: ModelConfig) -> RopeSpec:
    """Llama / Mistral / Gemma-2 rotary: half-split pairs, optional ``linear`` / ``llama3`` scaling (U1)."""
    dim = cfg.head_dim
    inv = default_inv_freq(dim, cfg.rope_theta)
    rs = cfg.rope_scaling
    if rs:
        typ = rs.get("type", rs.get("rope_type", "default"))
        if typ == "linear":
            inv = inv / float(rs["factor"])
        elif typ == "llama3":
            factor = float(rs["factor"])
            lo, hi = float(rs.get("low_freq_factor", 1.0)), float(rs.get("high_freq_factor", 4.0))
            old = float(rs.get("original_max_position_embeddings", 8192))
            wavelen = 2 * math.pi / inv
            smooth = ((old / wavelen) - lo) / (hi - lo)
            scaled = torch.where(wavelen > old / lo, inv / factor, inv)
            mid = (wavelen <= old / lo) & (wavelen >= old / hi)
            inv = torch.where(mid, (1 - smooth) * inv / factor + smooth * inv, scaled)
        elif typ in ("default", None):
            pass
        else:
            raise ValueError(f"unsupported rope_scaling type '{typ}' for {cfg.model_type}")
    return RopeSpec(inv_freq=inv, rot_dim=dim, interleaved=bool(cfg.rope_traditional) and cfg.model_type != "deepseek_v2")


def _yarn_find_correction_dim(num_rot, dim, base, max_pos):
    return (dim * math.log(max_pos / (num_rot * 2 * math.pi))) / (2 * math.log(base))


def deepseek_rope_spec(cfg: ModelConfig) -> RopeSpec:
    """DeepSeek-V2 rotary on the 64-dim ``*_pe`` slice: interleaved pairs + YaRN frequencies (U3)."""
    dim, base = cfg.qk_rope_head_dim, cfg.rope_theta
    rs = cfg.rope_scaling
    if not rs or rs.get("type", rs.get("rope_type")) not in ("yarn",):
        return RopeSpec(default_inv_freq(dim, base), dim, interleaved=True)
    factor = float(rs["factor"])
    orig = float(rs.get("original_max_position_embeddings", 4096))
    beta_fast, beta_slow = float(rs.get("beta_fast", 32)), float(rs.get("beta_slow", 1))
    freq_extra = base ** (torch.arange(0, dim, 2, dtype=torch.float32) / dim)
    freq_inter = factor * freq_extra
    low = max(math.floor(_yarn_find_correction_dim(beta_fast, dim, base, orig)), 0)
    high = min(math.ceil(_yarn_find_correction_dim(beta_slow, dim, base, orig)), dim - 1)
    if low == high:
        high += 0.001
    ramp = ((torch.arange(dim // 2, dtype=torch.float32) - low) / (high - low)).clamp(0, 1)
    mask = 1.0 - ramp
    freqs = (freq_inter * freq_extra) / (freq_inter * mask + freq_extra * (1 - mask))
    mscale = yarn_get_mscale(factor, rs.get("mscale", 1)) / yarn_get_mscale(factor, rs.get("mscale_all_dim", 0))
    return RopeSpec(inv_freq=1.0 / freqs, rot_dim=dim, interleaved=True, mscale=float(mscale))


# --------------------------------------------------------------------------------------------- base
class StageModel:
    """Common machinery: weight ingestion, embedding / head placement, KV geometry."""

    arch = "base"

    def __init__(self, cfg: ModelConfig, spec: Optional[ShardSpec] = None, dtype=torch.bfloat16,
                 device="cpu", backend: Optional[str] = None):
        self.cfg = cfg
        self.spec = spec or cfg.shard()
        self.dtype = dtype
        self.device = torch.device(device)
        self.backend_name = backend or default_backend_name(self.device)
        self.ops = get_backend(self.backend_name)
        self.qcfg = cfg.quantization
        self.embed_tokens: Optional[LinearWeight] = None
        self.norm_w: Optional[torch.Tensor] = None
        self.lm_head: Optional[LinearWeight] = None
        self.layer_weights: Dict[int, dict] = {}
        self.rope: Optional[RopeSpec] = None
        # fused stage boundary (parallel/p2p_fused.py): when set to (out_rows_tensor, flag_ptr) the last
        # kernel of the last local layer stores straight into that (peer-mapped) buffer and bumps the flag
        self.boundary = None
        self.boundary_fused = False
        # (rank, world) when only this rank's slice of every routed-expert bank was loaded (expert parallelism)
        self.expert_shard = None

    # reference-compatible surface ------------------------------------------------------------
    @property
    def layers(self) -> List:
        return [self.layer_weights.get(i) if self.spec.owns_layer(i) else IdentityBlock()
                for i in range(self.cfg.num_hidden_layers)]

    @property
    def head_dim(self):
        return self.cfg.head_dim

    @property
    def n_kv_heads(self) -> int:
        return self.cfg.kv_heads

    @property
    def needs_embed(self) -> bool:
        return self.spec.is_first or (self.spec.is_last and self.cfg.tie_word_embeddings)

    def kv_geometry(self):
        """(local_layers, kv_heads, d_k, d_v) for the paged cache."""
        return self.spec.num_kv_layers, self.cfg.kv_heads, self.cfg.qk_head_dim, self.cfg.v_dim

    # weights ---------------------------------------------------------------------------------
    def _lin(self, sd, prefix) -> LinearWeight:
        return LinearWeight.from_state(sd, prefix, self.qcfg, dtype=self.dtype, device=self.device)

    def _vec(self, sd, key) -> torch.Tensor:
        return sd.pop(key).to(device=self.device, dtype=self.dtype)

    def sanitize(self, sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Filter a full checkpoint to this stage (reference ``Model.sanitize``)."""
        from ..utils.checkpoint import key_in_shard

        return {k: v for k, v in sd.items() if key_in_shard(k, self.spec, self.cfg.tie_word_embeddings, self.cfg.model_type)}

    def load_state(self, sd: Dict[str, torch.Tensor], strict: bool = True):
        sd = self.sanitize(dict(sd))
        if self.needs_embed:
            self.embed_tokens = self._lin(sd, "model.embed_tokens")
        else:
            for k in [k for k in sd if k.startswith("model.embed_tokens")]:
                sd.pop(k)
        for i in self.spec.layers():
            # half-layer stage boundary: the other block's tensors belong to the neighbouring stage (sanitize dropped them)
            self.layer_weights[i] = self._load_layer(sd, i, self.spec.runs_attn(i), self.spec.runs_mlp(i))
        if self.spec.is_last:
            self.norm_w = self._vec(sd, "model.norm.weight")
            if self.cfg.tie_word_embeddings:
                self.lm_head = self.embed_tokens
                for k in [k for k in sd if k.startswith("lm_head")]:
                    sd.pop(k)
            else:
                self.lm_head = self._lin(sd, "lm_head")
        if strict and sd:
            raise ValueError(f"unexpected checkpoint tensors for stage {self.spec}: {sorted(sd)[:8]} ...")
        self.rope = self._make_rope()
        self.rope.inv_freq = self.rope.inv_freq.to(self.device)
        self._post_load()
        return self

    def _post_load(self):
        pass

    def _load_layer(self, sd, i, attn: bool = True, mlp: bool = True) -> dict:
        raise NotImplementedError

    def _make_rope(self) -> RopeSpec:
        raise NotImplementedError

    def weight_bytes(self) -> int:
        total = 0
        seen = set()

        def visit(o):
            nonlocal total
            if isinstance(o, LinearWeight):
                for t in (o.weight, o.wq, o.scales, o.biases, o.bias) + tuple(getattr(o, "_fp8", None) or ()):
                    if t is not None and t.data_ptr() not in seen:
                        seen.add(t.data_ptr())
                        total += t.numel() * t.element_size()
            elif isinstance(o, torch.Tensor):
                if o.data_ptr() not in seen:
                    seen.add(o.data_ptr())
                    total += o.numel() * o.element_size()
            elif isinstance(o, dict):
                for v in o.values():
                    visit(v)

        visit(self.layer_weights)
        for o in (self.embed_tokens, self.lm_head, self.norm_w):
            visit(o)
        return total

    # forward ---------------------------------------------------------------------------------
    def embed(self, ids: torch.Tensor) -> torch.Tensor:
        return self.ops.embed(ids, self.embed_tokens, 1.0, self.dtype)

    def attn_block(self, i: int, h: torch.Tensor, meta: BatchMeta, kpool, vpool) -> torch.Tensor:
        """``h + attention(norm(h))`` of layer ``i`` (appends this step's K/V to the paged pool)."""
        raise NotImplementedError

    def mlp_block(self, i: int, h: torch.Tensor, meta: BatchMeta) -> torch.Tensor:
        """``h + mlp(norm(h))`` of layer ``i``."""
        raise NotImplementedError

    def layer_forward(self, i: int, h: torch.Tensor, meta: BatchMeta, kpool, vpool) -> torch.Tensor:
        return self.mlp_block(i, self.attn_block(i, h, meta, kpool, vpool), meta)

    def _final_kwargs(self, i: int, T: int, block: str = "mlp") -> dict:
        """Extra kwargs for the last op of ``block`` of layer ``i``: when that op is the last kernel of this stage and a
        fused boundary is armed, it stores straight into the next stage's inbox and bumps its flag."""
        sp = self.spec
        if self.boundary is None or sp.is_last or i != sp.end_layer - 1 or (block == "attn") != sp.defer_last_mlp:
            return {}
        out, flag_ptr = self.boundary
        self.boundary_fused = True
        return dict(out=out[:T], signal=(flag_ptr, 0))

    def head(self, h: torch.Tensor, meta: BatchMeta, all_logits: bool = False) -> torch.Tensor:
        """Final norm + LM head -> fp32 logits for the last position of each sequence (the reference
        computes and ships all ``T`` rows, server.py:36-48; pass ``all_logits=True`` for that)."""
        O = self.ops
        if not all_logits:
            h = h.index_select(0, meta.last_idx.long()) if meta.num_tokens != meta.num_seqs else h
        hn = O.rmsnorm(h, self.norm_w, self.cfg.rms_norm_eps, self.cfg.model_type == "gemma2")
        cap = float(self.cfg.final_logit_softcapping) if (self.cfg.model_type == "gemma2" and self.cfg.final_logit_softcapping) else 0.0
        if cap and self.backend_name == "b200":
            # final-logit soft-capping (reference gemma2.py:82-83) runs in the LM-head GEMM epilogue: cap * tanh(y / cap)
            return O.linear(hn, self.lm_head, out_dtype=torch.float32, softcap=cap)
        logits = O.linear(hn, self.lm_head, out_dtype=torch.float32)
        if cap:
            logits = O.softcap_(logits, cap)
        return logits

    @torch.inference_mode()
    def forward(self, x: torch.Tensor, meta: BatchMeta, kv, all_logits: bool = False) -> torch.Tensor:
        """``x``: token ids ``[T]`` on the first stage, hidden states ``[T, H]`` otherwise.
        Returns hidden ``[T, H]`` (non-last stage) or fp32 logits ``[B, V]`` (last stage)."""
        if self.spec.is_first and not x.is_floating_point():
            h = self.embed(x)
        else:
            h = x.to(self.dtype)
        sp, li = self.spec, 0
        self.boundary_fused = False  # set by _final_kwargs when the stage's last kernel took the fused hand-off
        for i in sp.layers():
            if sp.runs_attn(i):
                h = self.attn_block(i, h, meta, kv.k[li], kv.v[li])
                li += 1
            if sp.runs_mlp(i):
                h = self.mlp_block(i, h, meta)
        if self.spec.is_last:
            return self.head(h, meta, all_logits)
        return h

    __call__ = forward
