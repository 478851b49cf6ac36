"""Sharded DeepSeek-V2 (MLA attention + MoE).

Reference: ``shard/server/model/deepseek_v2.py`` (layer-range wrapper, expert stacking at :101-111,
tuple ``head_dim`` = (192, 128) at :120-125) + upstream ``DeepseekV2DecoderLayer`` (SURVEY U3, §3.6).

B200 design notes:
* ``q_proj`` and ``kv_a_proj_with_mqa`` are concatenated at load into one GEMM (SURVEY K3/K4) when the
  model has no q-LoRA (DeepSeek-V2-Lite);
* the KV cache keeps the reference's *decompressed* layout (K 192 / V 128 per head) so results are
  bit-comparable with the reference pipeline; the MLA append kernel assembles ``[k_nope | k_pe]``
  straight into the paged pool;
* MoE = router kernel (fp32 softmax + top-k) -> token permutation -> grouped swap-AB tcgen05 GEMMs over
  the stacked ``switch_mlp`` weights -> weighted combine fused with shared-expert output + residual.
"""
from __future__ import annotations

import os
import re
from typing import Dict

import torch

from ..ops import BatchMeta, LinearWeight
from ..parallel.ep import ExpertParallelMoE
from .base import StageModel, deepseek_rope_spec

_EXPERT_RE = re.compile(r"^(model\.layers\.\d+\.mlp)\.experts\.(\d+)\.(gate_proj|up_proj|down_proj)\.(weight|scales|biases)$")


class DeepseekV2Stage(StageModel):
    arch = "deepseek_v2"
    overlap_shared_experts = os.environ.get("MLXB200_OVERLAP_SHARED", "1") != "0"
    # KV layout: cache the 512-dim latent + the 64-dim roped key (one shared "head", 576 values per token) instead of the
    # reference's decompressed per-head K/V (16 x (192 + 128) = 5120 values, shard/server/model/deepseek_v2.py:120-125) and absorb
    # kv_b into the query / output side.  Mathematically identical attention (see ``_attn_absorbed``).
    #   None (default): automatic — on when the sm_100a latent-attention kernel supports the shapes (16 heads, kv_lora_rank 512,
    #                   rope 64, no q-LoRA, unquantised attention weights, 64-token pages: DeepSeek-V2-Lite / Coder-V2-Lite);
    #   MLXB200_ABSORBED_MLA=0 / 1 forces it off / on (``1`` on the reference backend selects the einsum formulation).
    absorbed_mla = {"0": False, "1": True}.get(os.environ.get("MLXB200_ABSORBED_MLA", ""), None)

    def __init__(self, cfg, spec=None, dtype=torch.bfloat16, device="cpu", backend=None):
        super().__init__(cfg, spec, dtype, device, backend)
        if self.absorbed_mla is None:
            c = cfg
            # (quantised attention weights: promoted to bf16 at load when the FP8 conversion policy is on, else absorbed goes off —
            #  see ``_post_load``)
            self.absorbed_mla = bool(
                self.backend_name == "b200" and c.q_lora_rank is None and dtype == torch.bfloat16
                and self.ops.mla_absorbed_supported(c.num_attention_heads, c.kv_lora_rank, c.qk_rope_head_dim))

    @property
    def head_dim(self):
        # reference deepseek_v2.py:120-125 returns the (qk, v) tuple
        return (self.cfg.qk_nope_head_dim + self.cfg.qk_rope_head_dim, self.cfg.v_head_dim)

    def _make_rope(self):
        return deepseek_rope_spec(self.cfg)

    def kv_geometry(self):
        if self.absorbed_mla:
            c = self.cfg
            # the sm_100a kernel reads the values as the first 512 dims of the cached key row (no second pool)
            dv = 0 if self.backend_name == "b200" else c.kv_lora_rank
            return self.spec.num_kv_layers, 1, c.kv_lora_rank + c.qk_rope_head_dim, dv
        return super().kv_geometry()

    def _post_load(self):
        """Absorbed-latent MLA on the CUDA backend: fold ``W_UK`` into the query projection and ``W_UV`` into the output
        projection once at load (fp32 products, one bf16 rounding):

            q_abs[h] = W_UK[h]^T (W_q_nope[h] x)            -> rows [h*576, h*576+512) of ``qkv_abs`` (q_pe rows follow, then kv_a)
            out     = sum_h (W_o[:, h] W_UV[h]) o_lat[h]     -> ``o_abs`` [H, 16*512]

        so a decode step needs no kv_b GEMM and attention runs on the cached 576-dim latent (``ops/csrc/mla_decode.cu``).  The
        original q / kv_b / o weights stay for prefill chunks, which decompress the context they attend to."""
        c = self.cfg
        self._convert_quantized_for_b200()
        self._fuse_shared_experts()
        if not (self.absorbed_mla and self.backend_name == "b200"):
            return
        if c.q_lora_rank is not None or not self.ops.mla_absorbed_supported(c.num_attention_heads, c.kv_lora_rank, c.qk_rope_head_dim):
            raise NotImplementedError("absorbed-latent MLA kernel: 16 heads, kv_lora_rank 512, rope 64, no q-LoRA (DeepSeek-V2-Lite shapes)")
        if any(w[k].is_quantized for w in self.layer_weights.values() for k in ("qkv_a", "kv_b", "o") if k in w):
            # quantised attention weights keep their packed form (and the reference's cache layout): folding would expand them
            if os.environ.get("MLXB200_ABSORBED_MLA") == "1":
                raise NotImplementedError("absorbed-latent MLA with quantised attention weights")
            self.absorbed_mla = False
            return
        nh, nope, rd, vd, lr, H = c.num_attention_heads, c.qk_nope_head_dim, c.qk_rope_head_dim, c.v_head_dim, c.kv_lora_rank, c.hidden_size
        for w in self.layer_weights.values():
            if "qkv_a" not in w:
                continue
            qkv = w["qkv_a"].dense(torch.float32)                               # [nh*(nope+rd) + lr + rd, H]
            wq = qkv[: nh * (nope + rd)].view(nh, nope + rd, H)
            wkv = w["kv_b"].dense(torch.float32).view(nh, nope + vd, lr)
            q_abs = torch.einsum("hnl,hnk->hlk", wkv[:, :nope], wq[:, :nope])    # [nh, lr, H]
            rows = torch.cat([torch.cat([q_abs, wq[:, nope:]], 1).reshape(nh * (lr + rd), H), qkv[nh * (nope + rd):]], 0)
            w["qkv_abs"] = LinearWeight(weight=rows.to(self.dtype).contiguous())
            wo = w["o"].dense(torch.float32).view(H, nh, vd)
            o_abs = torch.einsum("ohv,hvl->ohl", wo, wkv[:, nope:]).reshape(H, nh * lr)
            w["o_abs"] = LinearWeight(weight=o_abs.to(self.dtype).contiguous(), bias=w["o"].bias)

    def sanitize(self, sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        sd = super().sanitize(sd)
        # stack per-expert HF weights into switch_mlp.* (reference deepseek_v2.py:101-111)
        groups: Dict[tuple, Dict[int, torch.Tensor]] = {}
        for k in list(sd):
            m = _EXPERT_RE.match(k)
            if m:
                groups.setdefault((m.group(1), m.group(3), m.group(4)), {})[int(m.group(2))] = sd.pop(k)
        n = self.cfg.n_routed_experts
        want = list(range(n))
        if self.expert_shard is not None:  # expert parallelism: only this rank's experts were read (utils/checkpoint.py)
            r, world = self.expert_shard
            want = list(range(r * n // world, (r + 1) * n // world))
        for (prefix, proj, kind), d in groups.items():
            if sorted(d) != want:
                raise ValueError(f"{prefix}.experts.*.{proj}.{kind}: expected experts {want[0]}..{want[-1]}, found {len(d)}")
            sd[f"{prefix}.switch_mlp.{proj}.{kind}"] = torch.stack([d[e] for e in want])
        return sd

    def _load_layer(self, sd, i, attn=True, mlp=True) -> dict:
        c = self.cfg
        p = f"model.layers.{i}"
        a = p + ".self_attn"
        w = {}
        if attn:
            w.update(in_ln=self._vec(sd, p + ".input_layernorm.weight"),
                     kv_a_ln=self._vec(sd, a + ".kv_a_layernorm.weight"),
                     kv_b=self._lin(sd, a + ".kv_b_proj"), o=self._lin(sd, a + ".o_proj"))
            kv_a = self._lin(sd, a + ".kv_a_proj_with_mqa")
            if c.q_lora_rank is None:
                w["qkv_a"] = LinearWeight.concat([self._lin(sd, a + ".q_proj"), kv_a])
            else:
                w["q_a_kv_a"] = LinearWeight.concat([self._lin(sd, a + ".q_a_proj"), kv_a])
                w["q_a_ln"] = self._vec(sd, a + ".q_a_layernorm.weight")
                w["q_b"] = self._lin(sd, a + ".q_b_proj")
        if not mlp:
            return w
        w["post_ln"] = self._vec(sd, p + ".post_attention_layernorm.weight")
        m = p + ".mlp"
        if c.is_moe_layer(i):
            w["router"] = sd.pop(m + ".gate.weight").to(device=self.device, dtype=self.dtype)
            for n in ("gate", "up", "down"):
                w["e_" + n] = self._lin(sd, f"{m}.switch_mlp.{n}_proj")
            if c.n_shared_experts:
                for n in ("gate", "up", "down"):
                    w["s_" + n] = self._lin(sd, f"{m}.shared_experts.{n}_proj")
        else:
            for n in ("gate", "up", "down"):
                w[n] = self._lin(sd, f"{m}.{n}_proj")
        return w

    def attn_block(self, i, h, meta: BatchMeta, kpool, vpool):
        O, c, w = self.ops, self.cfg, self.layer_weights[i]
        T = h.shape[0]
        nh, nope, rd, vd, lr = (c.num_attention_heads, c.qk_nope_head_dim, c.qk_rope_head_dim,
                                c.v_head_dim, c.kv_lora_rank)
        qd = nope + rd
        pn, self._prenormed = getattr(self, "_prenormed", None), None
        # the previous layer's MoE combine may already have produced this layer's input norm (ops/b200.py::moe_block, next_norm)
        normed = pn[1] if (pn is not None and pn[0] is h) else O.rmsnorm(h, w["in_ln"], c.rms_norm_eps)
        if "qkv_abs" in w and meta.max_q_len == 1 and meta.num_tokens == meta.num_seqs and kpool.shape[2] == 64:
            # decode step on the absorbed weights: one GEMM -> [q_abs | q_pe] x 16 heads, c_kv, k_pe; fused prologue (latent norm,
            # both ropes, cache append); tcgen05 multi-query attention over the cached latent; folded output projection
            qkv = O.linear(normed, w["qkv_abs"])
            qa = qkv[:, : nh * (lr + rd)].unflatten(1, (nh, lr + rd))
            O.mla_absorbed_prologue(qa, qkv[:, nh * (lr + rd): nh * (lr + rd) + lr], qkv[:, nh * (lr + rd) + lr:], w["kv_a_ln"],
                                    c.rms_norm_eps, kpool, meta, self.rope)
            o_lat = O.mla_decode(qa, kpool, meta, c.attn_scale)
            return O.linear(o_lat.view(T, nh * lr), w["o_abs"], residual=h, **self._final_kwargs(i, T, "attn"))
        if "qkv_a" in w:
            qkv = O.linear(normed, w["qkv_a"])
            q = qkv[:, : nh * qd]
            ckv = qkv[:, nh * qd: nh * qd + lr]
            k_pe = qkv[:, nh * qd + lr:]
        else:
            qa = O.linear(normed, w["q_a_kv_a"])
            ql = c.q_lora_rank
            q = O.linear(O.rmsnorm(qa[:, :ql], w["q_a_ln"], c.rms_norm_eps), w["q_b"])
            ckv, k_pe = qa[:, ql: ql + lr], qa[:, ql + lr:]
        q = q.view(T, nh, qd) if q.is_contiguous() else q.unflatten(1, (nh, qd))
        if self.absorbed_mla and self.backend_name == "b200":
            return self._attn_absorbed_b200(i, w, h, q, ckv, k_pe, meta, kpool)
        if self.absorbed_mla:
            return O.linear(self._attn_absorbed(w, q, ckv, k_pe, meta, kpool, vpool), w["o"], residual=h,
                            **self._final_kwargs(i, T, "attn"))
        kv = O.linear(O.rmsnorm(ckv, w["kv_a_ln"], c.rms_norm_eps), w["kv_b"]).view(T, nh, nope + vd)
        # rope(q_pe), rope(k_pe) and the cache append K=[k_nope|k_pe], V: one fused launch
        O.mla_rope_kv_write(q, k_pe, kv, kpool, vpool, meta, self.rope, nope, vd)
        attn = O.paged_attention(q, kpool, vpool, meta, c.attn_scale, 0.0)
        return O.linear(attn.reshape(T, nh * vd), w["o"], residual=h, **self._final_kwargs(i, T, "attn"))

    def _attn_absorbed(self, w, q, ckv, k_pe, meta: BatchMeta, kpool, vpool):
        """Weight-absorbed MLA.  With ``kv_b = [W_UK | W_UV]`` per head (``k_nope = W_UK c``, ``v = W_UV c``, ``c`` = normed latent):

            q_nope . k_nope = (W_UK^T q_nope) . c        -> query side absorbs W_UK   (q_abs, 512-dim)
            sum_t p_t v_t   = W_UV (sum_t p_t c_t)       -> output side absorbs W_UV

        so attention runs as multi-query attention over the cached ``[c | rope(k_pe)]`` (576) with values ``c`` (512)."""
        O, c = self.ops, self.cfg
        T = q.shape[0]
        nh, nope, rd, vd, lr = c.num_attention_heads, c.qk_nope_head_dim, c.qk_rope_head_dim, c.v_head_dim, c.kv_lora_rank
        lat = O.rmsnorm(ckv, w["kv_a_ln"], c.rms_norm_eps)                                   # [T, lr]
        q = q.clone()
        O.rope_(q, meta.positions, self.rope, nope)                                           # q_pe in place
        kpe = k_pe.reshape(T, 1, rd).clone()
        O.rope_(kpe, meta.positions, self.rope, 0)
        wkv = w["kv_b"].dense(torch.float32).view(nh, nope + vd, lr)
        q_abs = torch.einsum("thn,hnl->thl", q[..., :nope].float(), wkv[:, :nope]).to(q.dtype)
        O.kv_write(torch.cat([lat.unsqueeze(1), kpe.to(lat.dtype)], -1), lat.unsqueeze(1), kpool, vpool, meta.slot_mapping)
        o_lat = O.paged_attention(torch.cat([q_abs, q[..., nope:]], -1), kpool, vpool, meta, c.attn_scale, 0.0)   # [T, nh, lr]
        return torch.einsum("thl,hvl->thv", o_lat.float(), wkv[:, nope:]).to(q.dtype).reshape(T, nh * vd)

    fuse_shared = os.environ.get("MLXB200_FUSE_SHARED", "1") != "0"

    def _convert_quantized_for_b200(self):
        """Load-time policy for MLX 4/8-bit checkpoints on the CUDA backend (BASELINE config 2; off with MLXB200_FP8_EXPERTS=0, which
        keeps every weight packed and dequantised in-kernel with exact MLX-affine semantics):

        * routed + shared expert banks (93 % of the parameters) -> block-scaled MXFP8 (``utils/quant.py::to_mxfp8``), executed by
          ``tcgen05.mma kind::mxf8f6f4.block_scale`` (``ops/csrc/gemm_fp8.cu``); the shared experts are appended to the bank first;
        * attention projections (7 %) -> bf16, so the absorbed-latent MLA path (folded weights, tcgen05 latent attention) applies;
        * embeddings, LM head, dense layer-0 MLP stay packed (in-kernel dequant GEMMs / gather).

        With MLXB200_FP8_EXPERTS=1 the expert banks of a bf16 checkpoint are converted the same way."""
        env = os.environ.get("MLXB200_FP8_EXPERTS", "")
        if self.backend_name != "b200" or env == "0" or self.expert_shard is not None:
            return
        from ..utils.quant import to_mxfp8

        c = self.cfg
        ns, I, H = c.n_shared_experts or 0, c.moe_intermediate_size, c.hidden_size
        for w in self.layer_weights.values():
            quantized = any(isinstance(v, LinearWeight) and v.is_quantized for v in w.values())
            if not (quantized or env == "1"):
                continue
            for k in ("qkv_a", "q_a_kv_a", "q_b", "kv_b", "o"):
                if k in w and w[k].is_quantized:
                    w[k] = LinearWeight(weight=w[k].dense(self.dtype).contiguous(), bias=w[k].bias)
            if "router" not in w or w.get("e_gate") is None or H % 128 or I % 128:
                continue
            fuse = bool(ns and self.fuse_shared and "s_gate" in w and w["s_gate"].out_features == ns * I)

            def bank(ek, sk, down=False):
                parts = [w[ek].dense(torch.bfloat16)]
                if fuse:
                    sd = w[sk].dense(torch.bfloat16)
                    parts.append(sd.view(H, ns, I).permute(1, 0, 2) if down else sd.view(ns, I, H))
                qs, sfs = zip(*(to_mxfp8(ch) for p_ in parts for ch in p_.split(8)))
                out = LinearWeight()
                out._fp8 = (torch.cat(qs).contiguous(), torch.cat(sfs).contiguous())
                return out

            w["e_gate"], w["e_up"], w["e_down"] = bank("e_gate", "s_gate"), bank("e_up", "s_up"), bank("e_down", "s_down", True)
            if fuse:
                for k in ("s_gate", "s_up", "s_down"):
                    del w[k]
                w["n_fused_shared"] = ns

    def _fuse_shared_experts(self):
        """CUDA backend, bf16 banks, whole banks on this rank: append DeepSeek's shared experts to the routed bank as ``n_shared``
        always-on experts (ids ``E .. E+n_shared-1``, routing weight 1).  A SwiGLU MLP is separable along its intermediate dimension,
        so ``shared(x) = sum_j down_j(silu(gate_j x) * up_j x)`` with ``j`` over ``n_shared`` slices of width ``moe_intermediate_size``
        — exactly the shape of a routed expert.  The two small dense GEMMs of the shared branch (latency-bound: ~37 us per layer for
        35 MB of weights) disappear into the persistent grouped GEMMs that already stream the bank at the HBM roofline; the router
        kernel emits the extra (id, 1.0) columns itself."""
        c = self.cfg
        if not (self.fuse_shared and self.backend_name == "b200" and self.expert_shard is None and c.n_shared_experts):
            return
        ns, I, H = c.n_shared_experts, c.moe_intermediate_size, c.hidden_size
        for w in self.layer_weights.values():
            if "router" not in w or "s_gate" not in w or w.get("e_gate") is None:
                continue
            ws = [w[k] for k in ("e_gate", "e_up", "e_down", "s_gate", "s_up", "s_down")]
            if any(x.is_quantized or x.bias is not None or x.weight is None for x in ws) or w["s_gate"].weight.shape[0] != ns * I:
                continue
            w["e_gate"] = LinearWeight(weight=torch.cat([w["e_gate"].weight, w["s_gate"].weight.view(ns, I, H)], 0))
            w["e_up"] = LinearWeight(weight=torch.cat([w["e_up"].weight, w["s_up"].weight.view(ns, I, H)], 0))
            w["e_down"] = LinearWeight(weight=torch.cat([w["e_down"].weight, w["s_down"].weight.view(H, ns, I).permute(1, 0, 2)], 0))
            for k in ("s_gate", "s_up", "s_down"):
                del w[k]
            w["n_fused_shared"] = ns

    def unfuse_shared_experts(self):
        """Undo ``_fuse_shared_experts`` (expert parallelism shards the routed bank; the shared experts stay replicated)."""
        c = self.cfg
        ns, I, H, E = c.n_shared_experts, c.moe_intermediate_size, c.hidden_size, c.n_routed_experts
        for w in self.layer_weights.values():
            if w.pop("n_fused_shared", None) is None:
                continue
            g, u, d = w["e_gate"].weight, w["e_up"].weight, w["e_down"].weight
            w["s_gate"] = LinearWeight(weight=g[E:].reshape(ns * I, H).contiguous())
            w["s_up"] = LinearWeight(weight=u[E:].reshape(ns * I, H).contiguous())
            w["s_down"] = LinearWeight(weight=d[E:].permute(1, 0, 2).reshape(H, ns * I).contiguous())
            w["e_gate"], w["e_up"], w["e_down"] = (LinearWeight(weight=t[:E].contiguous()) for t in (g, u, d))

    def _attn_absorbed_b200(self, i, w, h, q, ckv, k_pe, meta: BatchMeta, kpool):
        """Prefill chunk / mixed batch with the latent cache (CUDA backend): append this chunk's latents, then *decompress the
        context the batch attends to* (``kv_b`` GEMM over the cached latents of its sequences) into a temporary per-head K/V pool
        and run the tensor-core flash-prefill kernel on it.  Costs O(context) extra GEMM work per chunk, prefill only; decode steps
        never come here (``attn_block`` routes them to the tcgen05 latent kernel)."""
        O, c = self.ops, self.cfg
        T = h.shape[0]
        nh, nope, rd, vd, lr = c.num_attention_heads, c.qk_nope_head_dim, c.qk_rope_head_dim, c.v_head_dim, c.kv_lora_rank
        page = kpool.shape[2]
        lat = O.rmsnorm(ckv, w["kv_a_ln"], c.rms_norm_eps)                                      # [T, lr]
        if getattr(meta, "fresh", False) and self.rope.interleaved and os.environ.get("MLXB200_PREFILL_FAST", "1") != "0":
            # Fresh prompts (no cached context; the TTFT case): everything the batch attends to is this chunk itself, so the
            # per-head K / V come straight from the chunk's own latents — no gather of cached pages, no concatenate / transpose
            # passes.  kv_b on the T rows, then ONE fused launch ropes q_pe in place and writes K = [k_nope | rope(k_pe)] and V
            # into temporary paged pools addressed by an identity block table; flash prefill runs on those.
            B = meta.num_seqs
            mb = max(1, (meta.max_ctx_len + page - 1) // page)
            tmp = getattr(meta, "_fresh_tmp", None)
            if tmp is None or tmp[0] != (page, mb):
                seq = torch.bucketize(torch.arange(T, device=h.device), meta.cu_seqlens[1:].long().contiguous(), right=True)
                pos = meta.positions.long()
                tslots = ((seq * mb + pos // page) * page + pos % page).to(torch.int32)
                tbt = torch.arange(B * mb, dtype=torch.int32, device=h.device).view(B, mb)
                tmp = meta._fresh_tmp = ((page, mb), BatchMeta(meta.positions, tslots, meta.cu_seqlens, meta.context_lens, tbt, meta.last_idx,
                                                               meta.num_tokens, B, meta.max_q_len, meta.max_ctx_len, page))
            tmp_meta = tmp[1]
            kv = O.linear(lat, w["kv_b"]).view(T, nh, nope + vd)
            kpe = k_pe.reshape(T, 1, rd).clone()
            O.rope_(kpe, meta.positions, self.rope, 0)
            kpool.view(-1, lr + rd).index_copy_(0, meta.slot_mapping.long(), torch.cat([lat, kpe.view(T, rd)], 1))   # latent cache
            ktmp = torch.empty(B * mb, nh, page, nope + rd, dtype=lat.dtype, device=h.device)
            vtmp = torch.empty(B * mb, nh, page, vd, dtype=lat.dtype, device=h.device)
            O.mla_rope_kv_write(q, k_pe, kv, ktmp, vtmp, tmp_meta, self.rope, nope, vd)
            attn = O.paged_attention(q, ktmp, vtmp, tmp_meta, c.attn_scale, 0.0)
            return O.linear(attn.reshape(T, nh * vd), w["o"], residual=h, **self._final_kwargs(i, T, "attn"))
        O.rope_(q, meta.positions, self.rope, nope)                                              # q_pe in place
        kpe = k_pe.reshape(T, 1, rd).clone()
        O.rope_(kpe, meta.positions, self.rope, 0)
        kpool.view(-1, lr + rd).index_copy_(0, meta.slot_mapping.long(), torch.cat([lat, kpe.view(T, rd)], 1))
        B = meta.num_seqs
        mb = min(meta.block_tables.shape[1], (meta.max_ctx_len + page - 1) // page)
        ctx = kpool.view(kpool.shape[0], page, lr + rd)[meta.block_tables[:, :mb].reshape(-1).long()]   # [B*mb, page, 576]
        rows = ctx.reshape(-1, lr + rd)
        kvd = O.linear(rows[:, :lr], w["kv_b"]).view(B * mb, page, nh, nope + vd)
        ktmp = torch.cat([kvd[..., :nope], rows[:, lr:].view(B * mb, page, 1, rd).expand(-1, -1, nh, -1)], -1).permute(0, 2, 1, 3).contiguous()
        vtmp = kvd[..., nope:].permute(0, 2, 1, 3).contiguous()
        tmp_meta = BatchMeta(meta.positions, meta.slot_mapping, meta.cu_seqlens, meta.context_lens,
                             torch.arange(B * mb, dtype=torch.int32, device=h.device).view(B, mb), meta.last_idx, meta.num_tokens,
                             B, meta.max_q_len, meta.max_ctx_len, page)
        attn = O.paged_attention(q, ktmp, vtmp, tmp_meta, c.attn_scale, 0.0)
        return O.linear(attn.reshape(T, nh * vd), w["o"], residual=h, **self._final_kwargs(i, T, "attn"))

    def mlp_block(self, i, h, meta: BatchMeta):
        O, c, w = self.ops, self.cfg, self.layer_weights[i]
        T = h.shape[0]
        if "router" not in w:
            normed = O.rmsnorm(h, w["post_ln"], c.rms_norm_eps)
            return O.linear(O.gated_up(normed, w["gate"], w["up"], "silu"), w["down"], residual=h,
                            **self._final_kwargs(i, T, "mlp"))
        route_kw = dict(top_k=c.num_experts_per_tok, method=c.topk_method, n_group=c.n_group or 1, topk_group=c.topk_group or 1,
                        scaling=c.routed_scaling_factor, norm_topk=c.norm_topk_prob)
        ep = (getattr(self, "ep_layers", None) or {}).get(i)
        cuda = self.backend_name == "b200"
        nxt = self.layer_weights.get(i + 1)
        next_norm = (nxt["in_ln"], c.rms_norm_eps) if (nxt is not None and "in_ln" in nxt and self.spec.runs_attn(i + 1)) else None
        if isinstance(ep, ExpertParallelMoE) and 1 <= T <= 1024:
            # expert-parallel block as four kernels (parallel/ep.py::route_forward): [pre-MoE norm + router + dispatch] -> grouped
            # gate/up -> grouped down (+ return) -> [combine + next layer's input norm]; the shared experts fork onto the side
            # stream right behind the router (they consume the normalised rows it stores)
            def shared_branch(normed):
                if "s_gate" not in w:
                    return h, None
                if self.overlap_shared_experts:
                    hs = torch.empty_like(h)
                    return hs, O.run_aside(lambda: O.linear(O.gated_up(normed, w["s_gate"], w["s_up"], "silu"), w["s_down"], residual=h, out=hs))
                return O.linear(O.gated_up(normed, w["s_gate"], w["s_up"], "silu"), w["s_down"], residual=h), None

            res = ep.route_forward(h, w["router"], route_kw, (w["post_ln"], c.rms_norm_eps), shared_branch, next_norm=next_norm)
            if next_norm is not None:
                self._prenormed = res
                return res[0]
            return res
        extra = dict(extra=w["n_fused_shared"]) if "n_fused_shared" in w else {}
        if ep is None and cuda and "s_gate" not in w:
            # CUDA backend, whole bank local, shared experts riding in the bank: the block is router -> grouped gate-up -> grouped
            # down -> combine, with BOTH RMSNorms around it folded in — the pre-MoE norm into the router kernel and the next layer's
            # input norm into the combine (decode batches; ops/b200.py::moe_block runs separate norm kernels for larger ones)
            fk = self._final_kwargs(i, T, "mlp")
            nn = dict(next_norm=next_norm) if (next_norm is not None and not fk) else {}
            res = O.moe_block(h, w["router"], route_kw, w["e_gate"], w["e_up"], w["e_down"], "silu", residual=h,
                              pre_norm=(w["post_ln"], c.rms_norm_eps), **extra, **nn, **fk)
            if nn:
                self._prenormed = res
                return res[0]
            return res
        normed = O.rmsnorm(h, w["post_ln"], c.rms_norm_eps)
        join = None
        if "s_gate" in w:
            # shared experts: h += down(silu(gate x) * up x).  Independent of the routed path until the final combine, so the
            # CUDA backend runs the two GEMMs on a side stream (a parallel branch of the decode graph) while the main
            # stream does router -> permutation / expert all-to-all -> expert GEMMs; the combine joins them.
            if self.overlap_shared_experts and cuda:
                hs, h_in = torch.empty_like(h), h   # result buffer allocated before the fork
                join = O.run_aside(lambda: O.linear(O.gated_up(normed, w["s_gate"], w["s_up"], "silu"), w["s_down"],
                                                    residual=h_in, out=hs))
                h = hs
            else:
                h = O.linear(O.gated_up(normed, w["s_gate"], w["s_up"], "silu"), w["s_down"], residual=h)
        if ep is None and cuda and join is None:
            # CUDA backend, whole bank local: router + experts as one op (scatter path for decode batches, ops/b200.py)
            return O.moe_block(normed, w["router"], route_kw, w["e_gate"], w["e_up"], w["e_down"], "silu", residual=h, **extra,
                               **self._final_kwargs(i, T, "mlp"))
        idx, wts = O.moe_route(normed, w["router"], **route_kw, **extra)
        if ep is not None:
            # expert-parallel mode (parallel/ep.py): routed experts are sharded over the ranks of the NVSwitch domain, tokens
            # travel through the fused dispatch / return kernels (all-to-all collectives on the reference backend)
            return ep.forward(normed, idx, wts, residual=h, join=join)
        kw = dict(join=join) if join is not None else {}
        return O.moe_experts(normed, idx, wts, w["e_gate"], w["e_up"], w["e_down"], "silu", residual=h, **kw,
                             **self._final_kwargs(i, T, "mlp"))


Model = DeepseekV2Stage
