"""GPU numerics: every sm_100a kernel vs the plain-PyTorch fp32 reference of the same op (SURVEY §4)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from mlx_sharding_b200.ops import reference as R
from mlx_sharding_b200.ops.meta import BatchMeta
from mlx_sharding_b200.ops.weights import LinearWeight, RopeSpec
from mlx_sharding_b200.utils import quant

DEV = "cuda"


@pytest.fixture(scope="module")
def B():
    from mlx_sharding_b200.ops import b200

    b200.load_extension()
    return b200


def rnd(*shape, scale=1.0, dtype=torch.bfloat16, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed + sum(shape))
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(dtype)


def close(a, b, atol, rtol):
    a, b = a.float(), b.float()
    err = (a - b).abs()
    ok = (err <= atol + rtol * b.abs()).all()
    assert ok, f"max err {err.max().item():.4g} (ref max {b.abs().max().item():.3g})"


@pytest.mark.parametrize("T,K,N", [(1, 2048, 3648), (7, 512, 4096), (64, 2048, 2048), (200, 2048, 576), (1024, 1024, 1408)])
def test_linear(B, T, K, N):
    x, w = rnd(T, K), rnd(N, K, scale=0.05)
    W = LinearWeight(weight=w)
    close(B.linear(x, W), R.linear(x, W), 2e-2, 2e-2)
    res = rnd(T, N)
    close(B.linear(x, W, residual=res), R.linear(x, W, residual=res), 3e-2, 2e-2)
    close(B.linear(x, W, out_dtype=torch.float32), R.linear(x, W, out_dtype=torch.float32), 1e-2, 1e-3)


def test_linear_strided_input_and_bias(B):
    big = rnd(33, 1024)
    x = big[:, 256:768]
    W = LinearWeight(weight=rnd(384, 512, scale=0.05), bias=rnd(384))
    close(B.linear(x, W), R.linear(x, W), 2e-2, 2e-2)


@pytest.mark.parametrize("act", ["silu", "gelu_tanh"])
@pytest.mark.parametrize("T", [3, 64, 300])
def test_gated_up(B, act, T):
    x = rnd(T, 2048)
    Wg, Wu = LinearWeight(weight=rnd(1408, 2048, scale=0.03, seed=1)), LinearWeight(weight=rnd(1408, 2048, scale=0.03, seed=2))
    close(B.gated_up(x, Wg, Wu, act), R.gated_up(x, Wg, Wu, act), 2e-2, 2e-2)


@pytest.mark.parametrize("H", [512, 2048, 4096])
@pytest.mark.parametrize("gemma", [False, True])
def test_rmsnorm(B, H, gemma):
    x, w, res = rnd(37, H), rnd(H, scale=0.3), rnd(37, H)
    close(B.rmsnorm(x, w, 1e-6, gemma), R.rmsnorm(x, w, 1e-6, gemma), 1e-2, 1e-2)
    close(B.rmsnorm(x, w, 1e-6, gemma, residual=res), R.rmsnorm(x, w, 1e-6, gemma, residual=res), 2e-2, 1e-2)
    xs = rnd(37, 2 * H)[:, H // 2: H // 2 + H]  # strided rows
    close(B.rmsnorm(xs, w, 1e-5, gemma), R.rmsnorm(xs, w, 1e-5, gemma), 1e-2, 1e-2)


@pytest.mark.parametrize("interleaved,rot_off,D", [(False, 0, 128), (True, 128, 192), (True, 0, 64)])
def test_rope(B, interleaved, rot_off, D):
    T, nh = 19, 4
    rd = D - rot_off
    inv = (1.0 / (10000.0 ** (torch.arange(0, rd, 2, dtype=torch.float32) / rd))).to(DEV)
    spec = RopeSpec(inv, rd, interleaved, mscale=1.0 if not interleaved else 1.25)
    pos = torch.randint(0, 5000, (T,), device=DEV, dtype=torch.int32)
    x = rnd(T, nh, D)
    a, b = x.clone(), x.clone()
    B.rope_(a, pos, spec, rot_off)
    R.rope_(b, pos, spec, rot_off)
    close(a, b, 2e-2, 1e-2)


@pytest.mark.parametrize("bits", [0, 4, 8])
def test_embed(B, bits):
    V, H = 1000, 512
    ids = torch.randint(0, V, (23,), device=DEV)
    w = rnd(V, H, scale=0.05)
    if bits:
        wq, s, b = quant.quantize(w.float(), 64, bits, out_dtype=torch.bfloat16)
        emb = LinearWeight(wq=wq, scales=s, biases=b, group_size=64, bits=bits)
    else:
        emb = LinearWeight(weight=w)
    close(B.embed(ids, emb), R.embed(ids, emb), 1e-3, 1e-2)
    close(B.embed(ids, emb, math.sqrt(H)), R.embed(ids, emb, math.sqrt(H)), 1e-2, 1e-2)


def _paged_setup(q_lens, ctx0, Hk, dk, dv, page=16, seed=0):
    Bn = len(q_lens)
    total_pages = sum((c + q + page - 1) // page for c, q in zip(ctx0, q_lens)) + 1
    perm = torch.randperm(total_pages - 1, generator=torch.Generator().manual_seed(seed)) + 1
    bts, o = [], 0
    for c, q in zip(ctx0, q_lens):
        n = (c + q + page - 1) // page
        bts.append(perm[o:o + n].tolist())
        o += n
    meta = BatchMeta.build(q_lens, ctx0, bts, page, device=DEV)
    kpool = rnd(total_pages, Hk, page, dk, seed=seed + 1)
    vpool = rnd(total_pages, Hk, page, dv, seed=seed + 2)
    return meta, kpool, vpool


@pytest.mark.parametrize("Hq,Hk,dk,dv,softcap", [(16, 16, 192, 128, 0.0), (32, 8, 128, 128, 0.0), (4, 2, 256, 256, 50.0),
                                                 (4, 4, 64, 64, 0.0)])
def test_paged_attention_decode_and_prefill(B, Hq, Hk, dk, dv, softcap):
    # mixed ragged batch: decode tokens (q_len 1) with long contexts + prefill chunks
    q_lens, ctx0 = [1, 1, 9, 1, 33], [700, 15, 0, 2047, 40]
    meta, kpool, vpool = _paged_setup(q_lens, ctx0, Hk, dk, dv)
    T = meta.num_tokens
    q = rnd(T, Hq, dk)
    k, v = rnd(T, Hk, dk, seed=5), rnd(T, Hk, dv, seed=6)
    kp2, vp2 = kpool.clone(), vpool.clone()
    B.kv_write(k, v, kpool, vpool, meta.slot_mapping)
    R.kv_write(k, v, kp2, vp2, meta.slot_mapping)
    assert torch.equal(kpool, kp2) and torch.equal(vpool, vp2)
    scale = dk ** -0.5
    close(B.paged_attention(q, kpool, vpool, meta, scale, softcap), R.paged_attention(q, kp2, vp2, meta, scale, softcap),
          2e-2, 2e-2)


def test_kv_write_mla(B):
    T, nh, nope, rd, vd, page = 21, 4, 128, 64, 128, 16
    meta, kpool, vpool = _paged_setup([T], [5], nh, nope + rd, vd, page)
    kv = rnd(T, nh, nope + vd)
    big = rnd(T, 512)
    kpe = big[:, 448:]  # strided [T, 64]
    kp2, vp2 = kpool.clone(), vpool.clone()
    B.kv_write_mla(kv, kpe, kpool, vpool, meta.slot_mapping, nope, vd)
    R.kv_write_mla(kv, kpe, kp2, vp2, meta.slot_mapping, nope, vd)
    assert torch.equal(kpool, kp2) and torch.equal(vpool, vp2)


@pytest.mark.parametrize("method,n_group,topk_group", [("greedy", 1, 1), ("group_limited_greedy", 8, 3)])
@pytest.mark.parametrize("T", [1, 64, 1000])
def test_moe_route(B, method, n_group, topk_group, T):
    H, E, k = 2048, 64, 6
    x, gw = rnd(T, H, seed=11), rnd(E, H, scale=0.05, seed=12)
    i1, w1 = B.moe_route(x, gw, k, method, n_group, topk_group, 1.5, False)
    i2, w2 = R.moe_route(x, gw, k, method, n_group, topk_group, 1.5, False)
    # compare as sets with weights (near-ties may reorder)
    s1, o1 = torch.sort(i1.long(), dim=1)
    s2, o2 = torch.sort(i2.long(), dim=1)
    same = (s1 == s2).all(dim=1)
    assert same.float().mean() > 0.98, same.float().mean()
    close(torch.gather(w1, 1, o1)[same], torch.gather(w2, 1, o2)[same], 1e-3, 2e-2)


@pytest.mark.parametrize("T", [1, 64, 700])
def test_moe_experts(B, T):
    H, I, E, k = 2048, 1408, 64, 6
    x = rnd(T, H)
    gw = rnd(E, H, scale=0.05)
    Wg = LinearWeight(weight=rnd(E, I, H, scale=0.03, seed=1))
    Wu = LinearWeight(weight=rnd(E, I, H, scale=0.03, seed=2))
    Wd = LinearWeight(weight=rnd(E, H, I, scale=0.03, seed=3))
    idx, w = R.moe_route(x, gw, k)
    res = rnd(T, H)
    got = B.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=res)
    dq = lambda w_: LinearWeight(weight=w_.dense(torch.bfloat16))
    ref = R.moe_experts(x, idx, w, dq(Wg), dq(Wu), dq(Wd), "silu", residual=res)
    close(got, ref, 5e-2, 2e-2)


@pytest.mark.parametrize("T,extra", [(1, 0), (64, 2), (100, 2), (64, 0)])
def test_moe_block_scatter_matches_permutation_path(B, T, extra):
    """Scatter path (router claims slots + copies rows, grouped GEMMs on per-expert counts, combine resets the counters) ==
    counting-sort permutation path, incl. the appended always-on (shared) experts; run twice: the counters must come back to 0."""
    H, I, E, k = 2048, 1408, 64, 6
    Et = E + extra
    x = rnd(T, H)
    gw = rnd(E, H, scale=0.05)
    Wg = LinearWeight(weight=rnd(Et, I, H, scale=0.03, seed=1))
    Wu = LinearWeight(weight=rnd(Et, I, H, scale=0.03, seed=2))
    Wd = LinearWeight(weight=rnd(Et, H, I, scale=0.03, seed=3))
    res = rnd(T, H)
    rk = dict(top_k=k, method="greedy", n_group=1, topk_group=1, scaling=1.0, norm_topk=False)
    idx, w = B.moe_route(x, gw, extra=extra, **rk)
    assert idx.shape == (T, k + extra)
    if extra:
        assert (idx[:, k:] == torch.arange(E, Et, device=DEV, dtype=torch.int32)).all() and (w[:, k:] == 1).all()
    ref = B.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=res)
    for _ in range(2):
        got = B.moe_block(x, gw, rk, Wg, Wu, Wd, "silu", residual=res, extra=extra)
        close(got, ref, 2e-2, 1e-2)
    torch.cuda.synchronize()
    assert all(int(c.sum()) == 0 for c, _ in B._scatter_bufs.values())


@pytest.mark.parametrize("T,extra", [(1, 0), (64, 2), (37, 2), (200, 2)])
def test_moe_block_fused_norms(B, T, extra):
    """RMSNorm folded into the router kernel (pre-MoE norm) and into the combine kernel (next layer's input norm) == separate norm
    kernels around the same block; T = 200 takes the permutation fallback (norms run as kernels there)."""
    H, I, E, k = 2048, 1408, 64, 6
    Et = E + extra
    h = rnd(T, H, scale=2.0)
    gw = rnd(E, H, scale=0.05)
    Wg = LinearWeight(weight=rnd(Et, I, H, scale=0.03, seed=1))
    Wu = LinearWeight(weight=rnd(Et, I, H, scale=0.03, seed=2))
    Wd = LinearWeight(weight=rnd(Et, H, I, scale=0.03, seed=3))
    n1, n2 = (1.0 + rnd(H, scale=0.1, seed=7)), (1.0 + rnd(H, scale=0.1, seed=8))
    rk = dict(top_k=k, method="greedy", n_group=1, topk_group=1, scaling=1.0, norm_topk=False)
    ref = B.moe_block(B.rmsnorm(h, n1, 1e-6), gw, rk, Wg, Wu, Wd, "silu", residual=h, extra=extra)
    ref_n = B.rmsnorm(ref, n2, 1e-6)
    for _ in range(2):
        got, got_n = B.moe_block(h, gw, rk, Wg, Wu, Wd, "silu", residual=h, extra=extra, pre_norm=(n1, 1e-6), next_norm=(n2, 1e-6))
        # the statistics are summed in a different order than rmsnorm_kernel's: a normalised value may land on the neighbouring bf16
        close(got, ref, 2e-2, 1e-2)
        close(got_n, ref_n, 2e-2, 2e-2)
    only_pre = B.moe_block(h, gw, rk, Wg, Wu, Wd, "silu", residual=h, extra=extra, pre_norm=(n1, 1e-6))
    close(only_pre, ref, 2e-2, 1e-2)
    torch.cuda.synchronize()
    assert all(int(c.sum()) == 0 for c, _ in B._scatter_bufs.values())


def test_sampler_greedy_logprobs_topk(B):
    Bn, V = 5, 102400
    logits = rnd(Bn, V, scale=3.0, dtype=torch.float32)
    temps, tps = torch.zeros(Bn, device=DEV), torch.ones(Bn, device=DEV)
    t1, l1, ti1, tl1 = B.sample(logits, temps, tps, top_logprobs=5)
    t2, l2, ti2, tl2 = R.sample(logits, temps, tps, top_logprobs=5)
    assert torch.equal(t1, t2) and torch.equal(ti1, ti2)
    close(l1, l2, 1e-3, 1e-4)
    close(tl1, tl2, 1e-3, 1e-4)


def test_sampler_distribution_and_top_p(B):
    V = 64
    base = torch.tensor([4.0, 3.0, 2.0, 1.0] + [-4.0] * (V - 4), device=DEV)
    n = 4000
    logits = base.repeat(n, 1).contiguous()
    g = torch.Generator(device=DEV).manual_seed(1234)
    temps = torch.full((n,), 1.0, device=DEV)
    toks, _, _, _ = B.sample(logits, temps, torch.ones(n, device=DEV), generator=g)
    freq = torch.bincount(toks, minlength=V).float() / n
    p = torch.softmax(base, 0)
    assert (freq[:4] - p[:4]).abs().max() < 0.03, (freq[:4], p[:4])
    # nucleus 0.8: tokens {0,1} have mass 0.64+0.24=0.88 >= 0.8 -> only they may appear
    toks, _, _, _ = B.sample(logits, temps, torch.full((n,), 0.8, device=DEV), generator=g)
    assert set(toks.unique().tolist()) <= {0, 1}
    f0 = (toks == 0).float().mean().item()
    assert abs(f0 - (p[0] / (p[0] + p[1])).item()) < 0.04
    # high temperature flattens
    toks, _, _, _ = B.sample(logits, torch.full((n,), 50.0, device=DEV), torch.ones(n, device=DEV), generator=g)
    assert toks.unique().numel() > 40


def test_apply_penalties(B):
    Bn, V = 3, 1000
    logits = rnd(Bn, V, dtype=torch.float32)
    ctx = torch.tensor([[5, 7, 5, -1], [-1, -1, -1, -1], [999, 0, 1, 2]], dtype=torch.int32, device=DEV)
    pen = torch.tensor([1.3, 1.0, 2.0], device=DEV)
    bidx = torch.tensor([[3, -1], [-1, -1], [999, 4]], dtype=torch.int32, device=DEV)
    bval = torch.tensor([[2.5, 0], [0, 0], [-1.0, 7.0]], device=DEV)
    a, b = logits.clone(), logits.clone()
    B.apply_penalties_(a, ctx, pen, bidx, bval)
    R.apply_penalties_(b, ctx, pen, bidx, bval)
    close(a, b, 1e-6, 1e-6)


def test_mla_rope_kv_write_fused(B):
    """Fused DeepSeek prologue (rope q_pe in place + assemble K=[k_nope|rope(k_pe)], V into the cache)."""
    T, nh, nope, rd, vd, page = 37, 16, 128, 64, 128, 16
    meta, kpool, vpool = _paged_setup([5, 32], [3, 100], nh, nope + rd, vd, page)
    assert meta.num_tokens == T
    inv = (1.0 / (10000.0 ** (torch.arange(0, rd, 2, dtype=torch.float32) / rd))).to(DEV)
    spec = RopeSpec(inv, rd, True, mscale=1.1)
    big = rnd(T, nh * (nope + rd) + 512 + rd)          # strided q / k_pe slices of one projection output
    q = big[:, : nh * (nope + rd)].unflatten(1, (nh, nope + rd))
    kpe = big[:, nh * (nope + rd) + 512:]
    kv = rnd(T, nh, nope + vd, seed=3)
    q2, kp2, vp2 = q.clone(), kpool.clone(), vpool.clone()
    B.mla_rope_kv_write(q, kpe, kv, kpool, vpool, meta, spec, nope, vd)
    R.mla_rope_kv_write(q2, kpe.clone(), kv, kp2, vp2, meta, spec, nope, vd)
    close(q, q2, 2e-2, 1e-2)
    close(kpool, kp2, 2e-2, 1e-2)
    assert torch.equal(vpool, vp2)


@pytest.mark.parametrize("Hq,Hk,dk,dv", [(16, 16, 192, 128), (32, 8, 128, 128), (4, 2, 64, 64)])
def test_flash_prefill_chunks(B, Hq, Hk, dk, dv):
    """Tensor-core prefill kernel: long prompts, chunk continuation at a context offset, ragged tails."""
    q_lens, ctx0 = [300, 64, 1, 129, 17], [0, 500, 77, 64, 1000]
    meta, kpool, vpool = _paged_setup(q_lens, ctx0, Hk, dk, dv, page=64 if dk == 192 else 16, seed=3)
    T = meta.num_tokens
    q = rnd(T, Hq, dk, seed=9)
    scale = dk ** -0.5
    got = B.paged_attention(q, kpool, vpool, meta, scale, 0.0)
    ref = R.paged_attention(q, kpool, vpool, meta, scale, 0.0)
    close(got, ref, 2e-2, 2e-2)
    # strided q (slice of a fused projection output)
    big = rnd(T, Hq * dk + 64, seed=10)
    qs = big[:, : Hq * dk].unflatten(1, (Hq, dk))
    close(B.paged_attention(qs, kpool, vpool, meta, scale, 0.0), R.paged_attention(qs.contiguous(), kpool, vpool, meta, scale, 0.0),
          2e-2, 2e-2)


def _qweight(*shape, bits=4, group=64, seed=0):
    w = rnd(*shape, scale=0.05, seed=seed).float()
    wq, s, b = quant.quantize(w, group, bits, out_dtype=torch.bfloat16)
    return LinearWeight(wq=wq, scales=s, biases=b, group_size=group, bits=bits)


@pytest.mark.parametrize("bits,group", [(4, 64), (8, 64), (4, 128)])
@pytest.mark.parametrize("T", [1, 64, 300])
def test_quantized_linear_in_kernel_dequant(B, bits, group, T):
    """int4/int8 MLX-affine weights dequantised inside the tcgen05 GEMM == dequantise-then-matmul oracle."""
    K, N = 2048, 1408
    x = rnd(T, K)
    W = _qweight(N, K, bits=bits, group=group, seed=1)
    assert B._qpack(W) is not None
    # oracle: dequantise (fp32 affine), round to bf16 like the kernel's producer warps, then fp32-accumulate matmul
    dq = lambda w: LinearWeight(weight=w.dense(torch.bfloat16))
    close(B.linear(x, W), R.linear(x, dq(W)), 3e-2, 2e-2)
    res = rnd(T, N)
    close(B.linear(x, W, residual=res, out_dtype=torch.float32), R.linear(x, dq(W), residual=res, out_dtype=torch.float32), 2e-2, 5e-3)
    Wu = _qweight(N, K, bits=bits, group=group, seed=2)
    close(B.gated_up(x, W, Wu, "silu"), R.gated_up(x, dq(W), dq(Wu), "silu"), 3e-2, 2e-2)


def test_quantized_moe_experts(B):
    H, I, E, k, T = 2048, 1408, 64, 6, 70
    x = rnd(T, H)
    Wg, Wu, Wd = _qweight(E, I, H, seed=1), _qweight(E, I, H, seed=2), _qweight(E, H, I, seed=3)
    idx, w = R.moe_route(x, rnd(E, H, scale=0.05, seed=12), k)
    res = rnd(T, H)
    got = B.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=res)
    dq = lambda w_: LinearWeight(weight=w_.dense(torch.bfloat16))
    ref = R.moe_experts(x, idx, w, dq(Wg), dq(Wu), dq(Wd), "silu", residual=res)
    close(got, ref, 5e-2, 2e-2)
