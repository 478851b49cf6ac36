"""Every launch path of the bf16 and packed-int GEMMs against a float64 reference, one test id per path.

The launchers choose the kernel, the token tile BN and the split-K reduction from the shape and the explicit ``splits``:

* ``splits == 1``: the persistent kernels (``gemm_persistent.cu``, ``gemm_q_persistent.cu``);
* ``1 < splits <= 8`` with ``BN * (2 if dual else 1) <= 128``: the cluster reduction through DSMEM (``gemm_cluster.cuh``);
* any other ``splits > 1``, and every quantised split: the fp32 workspace reduction with self-resetting tile tickets
  (``gemm_common.cuh::run_epilogue``).  ``splits`` above the number of k-blocks is clamped first.

Ids start with that path and BN.  Each output element is compared with a float64 reference built from the exact bf16 inputs and
rounded where the kernel rounds, under the bound derived at ``ACC`` below.  The same comparator must also *reject* two perturbed
references: one without the last k-block of ``x``, and one without the epilogue operand (bias or residual; for cases without
one: gate and up swapped, the neighbouring expert's weights, or the token rows rotated).  That shows the bound is tight enough
to see those bugs.  Outputs go into views of NaN-filled buffers, so a store outside ``out[:T, :N]`` or a skipped epilogue fails.
"""
import itertools

import pytest
import torch

from mlx_sharding_b200.ops.weights import LinearWeight
from mlx_sharding_b200.utils import quant

pytestmark = pytest.mark.gpu

DEV = "cuda"
KB = 64                              # k-block of every GEMM kernel (one 128-byte swizzle row of bf16)
ACT = {"silu": 1, "gelu_tanh": 2}
NAN = float("nan")

# Error bound of one output element.  bf16 products are exact and the kernels accumulate in fp32: the rounding error of a
# K-term sum is below K * 2^-24 * sum_k |x_k w_k| in the worst case and near sqrt(K) * 2^-24 * sum_k |x_k w_k| in practice,
# so ACC * (|x| @ |w|^T) with ACC = 2^-16 covers every K used here.  The epilogue adds a few fp32 operations (bias, residual,
# fast-math exp / tanh / divide): EPI relative.  Each rounding to bf16 may land one bf16 ulp away from the rounding of the exact
# value, so every rounding point adds one ulp of the value rounded there: one for a bf16 output, two with a residual
# (bf16(bf16(y) + r)), none for an fp32 output.  Through the gated activation an error in the gate grows by at most
# max |act'|, which is 1.10 for SiLU and 1.13 for tanh-GELU (ACT_SLOPE).
ACC = 2.0 ** -16
EPI = 2.0 ** -18
ACT_SLOPE = 1.2


@pytest.fixture(scope="module")
def B():
    from mlx_sharding_b200.ops import b200

    b200.load_extension()
    return b200


@pytest.fixture(scope="module")
def C(B):
    return B.C()


def rnd(*shape, scale=1.0, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(torch.bfloat16)


def weight(N, K, seed):
    return rnd(N, K, scale=K ** -0.5, seed=seed)   # outputs of unit scale for unit-scale x


# ------------------------------------------------------------------------------------------------ path selection (id names)
def pick_bn(rows):
    """Token tile of a dense launch (gemm_tcgen05.cu::gemm_pick_bn)."""
    for bn in (16, 32, 64, 128):
        if rows <= bn:
            return bn
    return 256


def dense_path(T, splits, K, dual=False):
    s = min(splits, -(-K // KB))
    if s == 1:
        return "persistent"
    return "cluster" if s <= 8 and pick_bn(T) * (2 if dual else 1) <= 128 else "workspace"


def split_note(splits, kb, group_kb=1):
    """Id suffix for the k-range edge cases: a trailing split with no k-blocks, a clamped split count, a split boundary inside a
    quantisation group."""
    s = min(splits, kb)
    per = -(-kb // s)
    notes = []
    if splits > kb:
        notes.append("clamped")
    if s > 1 and (s - 1) * per >= kb:
        notes.append("empty-split")
    if s > 1 and per % group_kb:
        notes.append("split-in-group")
    return "".join("-" + n for n in notes)


# ------------------------------------------------------------------------------------------------ float64 reference
def ulp_bf16(v):
    """One bf16 ulp (8 significant bits) at |v|, in float64."""
    _, e = torch.frexp(v.abs().clamp_min(2.0 ** -126))
    return torch.exp2((e - 8).to(torch.float64))


def gemm64(x, w):
    """x @ w^T in float64, its accumulation allowance, and the part contributed by the last (possibly partial) k-block."""
    xd, wd = x.double(), w.double()
    k0 = (x.shape[1] - 1) // KB * KB
    return xd @ wd.T, ACC * (xd.abs() @ wd.abs().T), xd[:, k0:] @ wd[:, k0:].T


def act64(act, g):
    if act == ACT["silu"]:
        return g * torch.sigmoid(g)
    k0, k1 = 0.7978845608028654, 0.044715
    return 0.5 * g * (1.0 + torch.tanh(k0 * (g + k1 * g ** 3)))


def rounded(y, err, out_fp32, residual=None):
    """(value, bound): the float64 result y (carrying error allowance err) stored the way the kernel epilogue stores it."""
    err = err + EPI * y.abs()
    if out_fp32:
        return (y if residual is None else y + residual.double()), err
    yb = y.to(torch.bfloat16).double()
    if residual is None:
        return yb, err + ulp_bf16(yb)
    val = (yb + residual.double()).to(torch.bfloat16).double()
    return val, err + ulp_bf16(yb) + ulp_bf16(val)


def reference(x, w, w2=None, act=0, bias=None, residual=None, softcap=0.0, out_fp32=False):
    """{name: (value, bound)}: "exact" and the perturbed references the bound must reject."""
    G, Ag, Lg = gemm64(x, w)
    U, Au, Lu = gemm64(x, w2) if w2 is not None else (None, None, None)

    def build(last_kb=True, epilogue=True, swap=False):
        g, u = (G, U) if last_kb else (G - Lg, None if U is None else U - Lu)
        ag, au = Ag, Au
        if swap:
            g, u, ag, au = u, g, au, ag
        if bias is not None and epilogue:
            g = g + bias.double()
        if u is None:
            y, err = g, ag
        else:
            a = act64(act, g)
            y, err = a * u, ACT_SLOPE * u.abs() * ag + a.abs() * au
        if softcap:
            y = softcap * torch.tanh(y / softcap)
        return rounded(y, err, out_fp32, residual if epilogue else None)

    refs = {"exact": build(), "no-last-k-block": build(last_kb=False)}
    if bias is not None or residual is not None:
        refs["no-bias-or-residual"] = build(epilogue=False)
    elif w2 is not None:
        refs["gate-up-swapped"] = build(swap=True)
    elif x.shape[0] > 1:
        v, b = refs["exact"]
        refs["rows-rotated"] = (v.roll(1, 0), b.roll(1, 0))
    return refs


def grouped_reference(x, w, w2, act, out_fp32, segments):
    """Row indices and {name: (value, bound)} of a grouped GEMM; segments = [(expert, first row, rows)].  Besides the
    k-block perturbation, every expert's rows are also checked against the neighbouring expert's weights."""
    E = w.shape[0]
    rows, parts = [], []
    for e, r0, n in segments:
        if n == 0:
            continue
        xe = x[r0:r0 + n]
        refs = reference(xe, w[e], None if w2 is None else w2[e], act=act, out_fp32=out_fp32)
        e2 = (e + 1) % E
        refs = {"exact": refs["exact"], "no-last-k-block": refs["no-last-k-block"],
                "wrong-expert": reference(xe, w[e2], None if w2 is None else w2[e2], act=act, out_fp32=out_fp32)["exact"]}
        rows.append(torch.arange(r0, r0 + n, device=DEV))
        parts.append(refs)
    merged = {k: tuple(torch.cat([p[k][i] for p in parts]) for i in range(2)) for k in parts[0]}
    return torch.cat(rows), merged


def check(got, refs):
    """Every element of got within the bound of the exact reference; and the bound rejects each perturbed reference."""
    g = got.double()
    val, bound = refs["exact"]
    ok = (g - val).abs() <= bound                      # NaN compares False
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{bad.shape[0]} of {ok.numel()} elements out of bound; first at {i}: got {g[i].item():.6g}, "
                             f"ref {val[i].item():.6g}, bound {bound[i].item():.3g}")
    for name, (v, b) in refs.items():
        if name != "exact":
            assert not bool(((g - v).abs() <= b).all()), f"the bound is too loose to see a {name} bug"


def guarded(T, N, dtype):
    """(buffer, out): out is a [T + 3, N] view into a NaN-filled buffer with 8 guard columns on the left and 24 on the right;
    the kernels get T < out.size(0) rows, so rows T.. are guard rows too.  The row stride stays a multiple of 16 bytes."""
    buf = torch.full((T + 3, N + 32), NAN, dtype=dtype, device=DEV)
    return buf, buf[:, 8:8 + N]


def check_guard(buf, T, N):
    inside = torch.zeros_like(buf, dtype=torch.bool)
    inside[:T, 8:8 + N] = True
    assert not bool(buf[inside].isnan().any()), "part of out[:T, :N] was never stored"
    assert bool(buf[~inside].isnan().all()), "the kernel stored outside out[:T, :N]"


def run_linear(C, x, w, splits, w2=None, act=0, bias=None, residual=None, softcap=0.0, out_fp32=False, flag=0, value=0):
    T, N = x.shape[0], w.shape[0]
    buf, out = guarded(T, N, torch.float32 if out_fp32 else torch.bfloat16)
    got = C.linear(x, w, w2=w2, residual=residual, bias=bias, act=act, softcap=softcap, out_fp32=out_fp32, out=out,
                   splits=splits, signal_flag_ptr=flag, signal_value=value)
    assert got.data_ptr() == out.data_ptr()
    check_guard(buf, T, N)
    return out[:T]


def qweight(B, N, K, bits, group, seed):
    """(kernel operands (codes, scales_t, biases_t), bf16 weights the kernel multiplies with).  The int4 path dequantises with
    one bf16 FMA (a single rounding of s*q + b), the int8 path with an fp32 FMA and then a rounding to bf16; the reference does
    the same, exactly (s*q is exact in fp32 for 8-bit codes and bf16 scales)."""
    wq, s, b = quant.quantize(weight(N, K, seed).float(), group, bits, out_dtype=torch.bfloat16)
    packed = B._qpack(LinearWeight(wq=wq, scales=s, biases=b, group_size=group, bits=bits))
    assert packed is not None
    dt = torch.float64 if bits == 4 else torch.float32
    codes = quant.unpack_codes(wq, bits).to(dt).view(N, K // group, group)
    dq = codes * s.to(dt)[..., None] + b.to(dt)[..., None]
    return packed, dq.view(N, K).to(torch.bfloat16)


def run_linear_q(C, x, q, bits, group, N, splits, q2=None, act=0, bias=None, residual=None, softcap=0.0, out_fp32=False, flag=0,
                 value=0):
    T = x.shape[0]
    buf, out = guarded(T, N, torch.float32 if out_fp32 else torch.bfloat16)
    got = C.linear_q(x, *q, *(q2 if q2 is not None else (None, None, None)), bits, group, N, residual, bias, act, softcap,
                     out_fp32, out, splits, flag, value)
    assert got.data_ptr() == out.data_ptr()
    check_guard(buf, T, N)
    return out[:T]


# ------------------------------------------------------------------------------------------------ dense bf16
def _dense_cases():
    Ts = (1, 15, 17, 33, 64, 65, 127, 129, 255, 257, 300)
    splits = (1, 2, 3, 4, 8, 12)
    nk = [(N, K) for K in (512, 1408, 2048, 2056) for N in (576, 1408, 3648)]
    cases = [(T, s, *nk[(i + 5 * j) % len(nk)]) for (i, T), (j, s) in itertools.product(enumerate(Ts), enumerate(splits))]
    # 9 k-blocks in splits of 3, 3, 3 and 0 (cluster and workspace), and more splits than k-blocks
    cases += [(17, 4, 576, 576), (300, 4, 576, 576), (17, 12, 1408, 512), (200, 12, 576, 512)]
    return [pytest.param(T, s, N, K, id=f"{dense_path(T, s, K)}-bn{pick_bn(T)}-T{T}-s{s}-N{N}-K{K}{split_note(s, -(-K // KB))}")
            for T, s, N, K in cases]


@pytest.mark.parametrize("T,splits,N,K", _dense_cases())
def test_dense(C, T, splits, N, K):
    x, w, bias = rnd(T, K, seed=T), weight(N, K, seed=N + K), rnd(N, scale=0.5, seed=7)
    check(run_linear(C, x, w, splits, bias=bias), reference(x, w, bias=bias))


def _dual_cases():
    nk = [(1408, 2048), (576, 2056), (1408, 1408)]
    out = []
    for i, (act, T, s) in enumerate(itertools.product(ACT, (3, 64, 65, 200, 300), (1, 2, 4))):
        N, K = nk[i % len(nk)]
        out.append(pytest.param(act, T, s, N, K, id=f"{dense_path(T, s, K, dual=True)}-bn{pick_bn(T)}-{act}-T{T}-s{s}-N{N}-K{K}"))
    return out


@pytest.mark.parametrize("act,T,splits,N,K", _dual_cases())
def test_dual(C, act, T, splits, N, K):
    """Gate/up pair: bf16(act(x wg^T) * (x wu^T)), both accumulators in fp32."""
    x, wg, wu = rnd(T, K, seed=T), weight(N, K, seed=1), weight(N, K, seed=2)
    check(run_linear(C, x, wg, splits, w2=wu, act=ACT[act]), reference(x, wg, wu, act=ACT[act]))


REDUCTIONS = {"persistent": (257, 1), "cluster": (33, 3), "workspace": (33, 12)}
EPILOGUES = ["plain", "bias", "residual", "softcap-bf16", "softcap-fp32", "fp32-residual", "strided-nan"]


@pytest.mark.parametrize("option", EPILOGUES)
@pytest.mark.parametrize("reduction", list(REDUCTIONS))
def test_epilogue(C, reduction, option):
    T, splits = REDUCTIONS[reduction]
    N, K = 576, 2056                                   # a 64-column tail past the last 128-row tile, a k-block tail of 8
    assert dense_path(T, splits, K) == reduction
    x, w = rnd(T, K, seed=3), weight(N, K, seed=4)
    kw = dict(bias=rnd(N, scale=0.5, seed=5))
    if option == "plain":
        kw = {}
    elif option == "residual":
        kw = dict(residual=rnd(T, N, seed=6))
    elif option.startswith("softcap"):
        kw.update(softcap=2.0, out_fp32=option.endswith("fp32"))
    elif option == "fp32-residual":
        kw = dict(residual=rnd(T, N, seed=6), out_fp32=True)
    elif option == "strided-nan":
        # operands are views whose rows continue with NaN past K (and x with NaN rows past T): nothing beyond them may be read
        xb = torch.full((T + 5, K + 64), NAN, dtype=torch.bfloat16, device=DEV)
        wb = torch.full((N + 64, K + 64), NAN, dtype=torch.bfloat16, device=DEV)
        xb[:T, :K], wb[:N, :K] = x, w
        x, w = xb[:T, :K], wb[:N, :K]
    check(run_linear(C, x, w, splits, **kw), reference(x, w, **kw))


# ------------------------------------------------------------------------------------------------ determinism, ticket reset
SPLIT_PATHS = {"cluster": (17, 4), "workspace-bn256": (200, 2), "workspace-bn32": (17, 12)}


@pytest.mark.parametrize("path", list(SPLIT_PATHS))
def test_split_k_repeatable(C, path):
    """Split-K results are bitwise repeatable, and a launch of another shape in between changes nothing.  Every launch writes
    into a fresh NaN buffer, so an epilogue skipped because a tile ticket or done counter was left non-zero shows up."""
    T, splits = SPLIT_PATHS[path]
    N, K = 1408, 2048
    assert dense_path(T, splits, K) == dense_path(T + 40, splits, 1024) == path.split("-")[0]
    x, w, bias = rnd(T, K, seed=11), weight(N, K, seed=12), rnd(N, scale=0.5, seed=13)
    first = run_linear(C, x, w, splits, bias=bias)
    check(first, reference(x, w, bias=bias))
    assert torch.equal(run_linear(C, x, w, splits, bias=bias), first)
    x2, w2 = rnd(T + 40, 1024, seed=14), weight(3648, 1024, seed=15)
    check(run_linear(C, x2, w2, splits), reference(x2, w2))
    assert torch.equal(run_linear(C, x, w, splits, bias=bias), first)


@pytest.mark.parametrize("path", ["workspace", "cluster"])
def test_split_k_graph_replay(C, path):
    """A captured split-K launch replayed three times equals the eager launch bit for bit (tickets reset inside the graph)."""
    T, splits = (200, 2) if path == "workspace" else (17, 4)
    N, K = 1408, 2048
    assert dense_path(T, splits, K) == path
    x, w = rnd(T, K, seed=21), weight(N, K, seed=22)
    out = torch.full((T, N), NAN, dtype=torch.bfloat16, device=DEV)
    C.linear(x, w, out=out, splits=splits)
    eager = out.clone()
    check(eager, reference(x, w))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        C.linear(x, w, out=out, splits=splits)
    for _ in range(3):
        out.fill_(NAN)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)


# ------------------------------------------------------------------------------------------------ grouped bf16
def offsets_of(counts):
    return torch.tensor([0] + list(itertools.accumulate(counts)), dtype=torch.int32, device=DEV)


GROUPED = {"empty-first-middle-last": [0, 37, 5, 0, 64, 1, 60, 0], "one-expert-300-of-400": [30, 0, 300, 10, 0, 25, 35, 0],
           "decode": [1, 0, 2, 0, 0, 1, 0, 3]}


@pytest.mark.parametrize("name", list(GROUPED))
def test_grouped_offsets(C, name):
    """Offsets layout, as moe_experts runs it: dual gate/up (N = 1408) then the down projection (N = 2048) with fp32 output."""
    counts = GROUPED[name]
    E, R, H, I = len(counts), sum(counts), 2048, 1408
    x = rnd(R, H, seed=31)
    wg, wu, wd = (torch.stack([weight(n, k, seed=100 * j + e) for e in range(E)]) for j, (n, k) in enumerate([(I, H), (I, H), (H, I)]))
    offs = offsets_of(counts)
    segs = [(e, int(offs[e]), c) for e, c in enumerate(counts)]
    h = C.grouped_linear(x, wg, wu, offs, R, ACT["silu"], False)
    rows, refs = grouped_reference(x, wg, wu, ACT["silu"], False, segs)
    check(h[rows], refs)
    y = C.grouped_linear(h, wd, None, offs, R, 0, True)
    rows, refs = grouped_reference(h, wd, None, 0, True, segs)
    check(y[rows], refs)


@pytest.mark.parametrize("stride", [64, 128], ids=["stride64", "stride128"])
def test_grouped_counts_layout(C, stride):
    """Counts (scatter) layout: expert e owns rows [e * stride, e * stride + counts[e]); the rows past each count are NaN and
    must not leak into any stored row."""
    counts = [0, 5, stride, 17, 0, 1, stride - 1, 33]
    E, H, I = len(counts), 1024, 1408
    x = torch.full((E * stride, H), NAN, dtype=torch.bfloat16, device=DEV)
    for e, c in enumerate(counts):
        x[e * stride:e * stride + c] = rnd(c, H, seed=40 + e)
    wg, wu, wd = (torch.stack([weight(n, k, seed=100 * j + e) for e in range(E)]) for j, (n, k) in enumerate([(I, H), (I, H), (H, I)]))
    cnt = torch.tensor(counts, dtype=torch.int32, device=DEV)
    segs = [(e, e * stride, c) for e, c in enumerate(counts)]
    h = C.grouped_linear(x, wg, wu, cnt, stride, ACT["gelu_tanh"], False, None, None, None, sum(counts), stride)
    rows, refs = grouped_reference(x, wg, wu, ACT["gelu_tanh"], False, segs)
    check(h[rows], refs)
    y = C.grouped_linear(h, wd, None, cnt, stride, 0, True, None, None, None, sum(counts), stride)
    rows, refs = grouped_reference(h, wd, None, 0, True, segs)
    check(y[rows], refs)


# ------------------------------------------------------------------------------------------------ quantised
def q_path(splits):
    return "qpersistent" if splits == 1 else "qsplit"


def _quant_cases():
    out = []
    for (bi, bits), (gi, group) in itertools.product(enumerate((4, 8)), enumerate((64, 128))):
        for ti, T in enumerate((1, 17, 32, 33, 300)):
            s = (1, 2, 3, 4)[(ti + bi + gi) % 4]
            N, K = (576, 2048) if ti % 2 == 0 else (1408, 1408)
            out.append((bits, group, T, s, N, K))
    out += [(4, 128, 17, 2, 1408, 1408), (8, 128, 300, 2, 576, 1408)]   # a split boundary in the middle of a 128-wide group
    return [pytest.param(bits, group, T, s, N, K,
                         id=f"{q_path(s)}-bn{pick_bn(T)}-int{bits}-g{group}-T{T}-s{s}-N{N}-K{K}{split_note(s, K // KB, group // KB)}")
            for bits, group, T, s, N, K in out]


@pytest.mark.parametrize("bits,group,T,splits,N,K", _quant_cases())
def test_quantized(B, C, bits, group, T, splits, N, K):
    q, w = qweight(B, N, K, bits, group, seed=N + K + bits)
    x, bias = rnd(T, K, seed=T), rnd(N, scale=0.5, seed=8)
    check(run_linear_q(C, x, q, bits, group, N, splits, bias=bias), reference(x, w, bias=bias))


def _q_variants(splits, formats):
    return [pytest.param(bits, group, s, id=f"{q_path(s)}-int{bits}-g{group}-s{s}") for (bits, group), s in itertools.product(formats, splits)]


@pytest.mark.parametrize("bits,group,splits", _q_variants((1, 2), [(4, 64), (8, 128)]))
def test_quantized_dual(B, C, bits, group, splits):
    T, N, K = 17, 1408, 2048
    (qg, wg), (qu, wu) = qweight(B, N, K, bits, group, seed=1), qweight(B, N, K, bits, group, seed=2)
    x = rnd(T, K, seed=9)
    got = run_linear_q(C, x, qg, bits, group, N, splits, q2=qu, act=ACT["silu"])
    check(got, reference(x, wg, wu, act=ACT["silu"]))


@pytest.mark.parametrize("bits,group,splits", _q_variants((1, 3), [(4, 128), (8, 64)]))
def test_quantized_bias_residual_fp32(B, C, bits, group, splits):
    T, N, K = 33, 576, 2048
    q, w = qweight(B, N, K, bits, group, seed=3)
    x, bias, res = rnd(T, K, seed=10), rnd(N, scale=0.5, seed=11), rnd(T, N, seed=12)
    got = run_linear_q(C, x, q, bits, group, N, splits, bias=bias, residual=res, out_fp32=True)
    check(got, reference(x, w, bias=bias, residual=res, out_fp32=True))


@pytest.mark.parametrize("bits,group", [(4, 64), (8, 128)], ids=["int4-g64", "int8-g128"])
def test_grouped_quantized_empty_experts(B, C, bits, group):
    counts = [0, 20, 0, 9, 41, 0]
    E, R, H, I = len(counts), sum(counts), 1024, 1408
    qs = [[qweight(B, n, k, bits, group, seed=100 * j + e) for e in range(E)] for j, (n, k) in enumerate([(I, H), (I, H), (H, I)])]
    (qg, wg), (qu, wu), (qd, wd) = ((tuple(torch.cat([q[0][i] for q in bank], dim=1 if i else 0) for i in range(3)),
                                     torch.stack([q[1] for q in bank])) for bank in qs)
    x, offs = rnd(R, H, seed=50), offsets_of(counts)
    segs = [(e, int(offs[e]), c) for e, c in enumerate(counts)]
    h = C.grouped_linear_q(x, *qg, *qu, bits, group, E, I, offs, R, ACT["silu"], False)
    rows, refs = grouped_reference(x, wg, wu, ACT["silu"], False, segs)
    check(h[rows], refs)
    y = C.grouped_linear_q(h, *qd, None, None, None, bits, group, E, H, offs, R, 0, True)
    rows, refs = grouped_reference(h, wd, None, 0, True, segs)
    check(y[rows], refs)


# ------------------------------------------------------------------------------------------------ fused stage-boundary signal
SIGNAL_PATHS = ["persistent", "cluster", "workspace", "qpersistent", "qsplit", "rmsnorm"]


def rmsnorm_reference(x, w, eps):
    xd = x.double()
    y = xd * torch.rsqrt(xd.pow(2).mean(-1, keepdim=True) + eps) * w.double()
    return {"exact": rounded(y, ACC * y.abs(), False)}


@pytest.mark.parametrize("mode", ["count", "value"])
@pytest.mark.parametrize("path", SIGNAL_PATHS)
def test_stage_signal(B, C, path, mode):
    """One GPU, no consumer: the flag is read by the host after a synchronize.  Counting mode adds 1 per launch, so two launches
    leave 2 only if the grid-completion counter came back to zero after the first; value mode stores the value."""
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    value = 0 if mode == "count" else 7
    sig = dict(flag=flag.data_ptr(), value=value)
    for _ in range(2):
        if path == "rmsnorm":
            x, w = rnd(37, 2048, seed=60), rnd(2048, scale=0.3, seed=61)
            buf, out = guarded(37, 2048, torch.bfloat16)
            C.rmsnorm(x, w, 1e-6, False, None, out, flag.data_ptr(), value)
            check_guard(buf, 37, 2048)
            check(out[:37], rmsnorm_reference(x, w, 1e-6))
        elif path.startswith("q"):
            T, splits, N, K = (300, 1, 3648, 1024) if path == "qpersistent" else (17, 2, 1408, 2048)
            q, w = qweight(B, N, K, 4, 64, seed=62)
            x = rnd(T, K, seed=63)
            check(run_linear_q(C, x, q, 4, 64, N, splits, **sig), reference(x, w))
        else:
            # the persistent case has more tiles (3 x 56) than the B200 has SMs: CTAs report several tiles each
            T, splits, N, K = {"persistent": (600, 1, 7168, 512), "cluster": (17, 4, 1408, 2048),
                               "workspace": (200, 2, 1408, 2048)}[path]
            assert dense_path(T, splits, K) == path
            x, w = rnd(T, K, seed=64), weight(N, K, seed=65)
            check(run_linear(C, x, w, splits, **sig), reference(x, w))
    torch.cuda.synchronize()
    assert flag.item() == (2 if mode == "count" else 7)


# ------------------------------------------------------------------------------------------------ operand validation
def bad_view(rows, cols, dtype, kind):
    """A [rows, cols] view whose first element is not 16-byte aligned ("base") or whose row stride is not a multiple of 16
    bytes ("stride")."""
    el = 16 // torch.empty(0, dtype=dtype).element_size()
    if kind == "base":
        return torch.zeros(rows, cols + 2 * el, dtype=dtype, device=DEV)[:, 1:1 + cols]
    return torch.zeros(rows, cols + el // 2, dtype=dtype, device=DEV)[:, :cols]


MISALIGNED = [(op, operand, kind) for op, operands in (("linear", ("out", "out-fp32", "residual")), ("linear_q", ("out", "residual")),
                                                        ("rmsnorm", ("x", "out", "residual")))
              for operand in operands for kind in ("base", "stride")]


@pytest.mark.parametrize("op,operand,kind", MISALIGNED, ids=["-".join(c) for c in MISALIGNED])
def test_misaligned_operand_rejected(B, C, op, operand, kind):
    """residual / out (and x of rmsnorm) are accessed as 16-byte vectors: a misaligned view must raise, not reach a kernel.  The
    zero-row call comes first, so a build without the check fails on it before launching anything misaligned."""
    T, N, K = 4, 576, 512
    dtype = torch.float32 if operand == "out-fp32" else torch.bfloat16
    bad = bad_view(T, N if op != "rmsnorm" else K, dtype, kind)
    if op == "rmsnorm":
        x, w = rnd(T, K, seed=70), rnd(K, seed=71)
        args = {"x": x, "out": None, "residual": None}
        args[operand] = bad

        def call(rows):
            return C.rmsnorm(args["x"][:rows], w, 1e-6, False, None if args["residual"] is None else args["residual"][:rows],
                             None if args["out"] is None else args["out"][:rows], 0, 0)
    else:
        x = rnd(T, K, seed=72)
        out = bad if operand.startswith("out") else None
        res = bad if operand == "residual" else None
        fp32 = operand == "out-fp32"
        if op == "linear":
            w = weight(N, K, seed=73)

            def call(rows):
                return C.linear(x[:rows], w, residual=None if res is None else res[:rows], out_fp32=fp32,
                                out=None if out is None else out[:rows], splits=1)
        else:
            q, _ = qweight(B, N, K, 4, 64, seed=74)

            def call(rows):
                return C.linear_q(x[:rows], *q, None, None, None, 4, 64, N, None if res is None else res[:rows], None, 0, 0.0,
                                  fp32, None if out is None else out[:rows], 1, 0, 0)
    with pytest.raises(RuntimeError, match="16-byte|16 bytes"):
        call(0)
    with pytest.raises(RuntimeError, match="16-byte|16 bytes"):
        call(T)
