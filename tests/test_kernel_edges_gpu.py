"""Element-wise checks of the sm_100a kernels against float64 references at ragged, multi-batch and model-config shapes.

Every reference is computed in float64 from the bf16 values the kernel actually read, and every output element is held to
its own error bound (never one norm over the whole tensor), so a wrong tile edge or a dropped K-block fails.  A leaked
attention key fails the element-wise check only where it carries a real share of a row's softmax mass: at long T one extra
key moves a row by about 1/T, below the bf16 rounding of P, and there the bitwise batch-isolation and causality tests are
what catch it.  The bounds have the form

    |got - ref| <= c_out * 2^-8 * |ref|  +  c_acc * K * 2^-24 * (|A| |B|^T)

(bf16 output rounding plus fp32 accumulation over K), with the magnitude product computed in float64 next to the
reference.  Each case prints ``max err/bound``: near 1 the bound is tight, far below it would be vacuous.  Outputs are
written through views into larger buffers filled with a NaN bit pattern, and padded input columns / rows hold NaN, so a
kernel that writes outside its output or reads past K shows up.  The negative controls at the end plant a plausible
kernel bug into the reference and assert that the comparator rejects it.
"""
import math

import pytest
import torch

import edge_checks
from edge_checks import (BF, CANARY16, CANARY32, F64, U8, U24, _assert_outside_untouched, _canary_out, _excess, _operand,
                         _padded, _where_tile, check)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    edge_checks.worst.clear()
    yield
    edge_checks.print_worst()


@pytest.fixture(scope="module")
def C():
    from relora_b200.ops import native

    return native.require()


@pytest.fixture(scope="module")
def F():
    from relora_b200.ops import fused

    return fused


# ----------------------------------------------------------------------------------------------------------------- helpers
def _randn(*shape, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(BF)


def _where_attn(shape, i):
    b, h, t, d = torch.unravel_index(torch.tensor(i), shape)
    return f"(batch {int(b)}, head {int(h)}, row {int(t)}, dim {int(d)})"


def gemm_bound(ref, mag, K, *, out_bf16=True, extra=0.0):
    """bf16 (or fp32) output rounding + fp32 accumulation of K exact bf16 products.  The worst-case accumulation error of a
    length-K fp32 sum is K * 2^-24 * sum|a_k b_k| (c_acc = 1); ``extra`` counts further fp32 roundings in the epilogue
    (alpha, residual, bias, the split-K atomics), each at most 2^-24 of the magnitude.  ``mag`` carries everything that
    was summed in absolute value."""
    b = (K + 2 + extra) * U24 * mag
    if out_bf16:
        b = b + U8 * ref.abs()
    return b


def _mm(a, b):
    return a.to(F64) @ b.to(F64)


# ---------------------------------------------------------------------------------------------------------------- GEMM
# K, N and M from the model configs: hidden sizes 416 (llama_40m) / 640 (llama_100m), intermediate sizes 688 / 1368 /
# 1376 / 2736 / 5504, the LM-head tail chunk (4097 rows = one full 4096 chunk + 1), and the smallest legal widths.
_GEMM_CASES = sorted({
    *[(189, 688, k) for k in (8, 24, 416, 640, 1368, 2736, 5504)],
    *[(257, n, 416) for n in (8, 264, 688, 1376, 2736)],
    *[(m, 264, 640) for m in (1, 7, 65, 129, 189, 257, 4097)],
    (4097, 2736, 1368), (129, 1376, 5504), (65, 8, 2736), (7, 2736, 24),
})


@pytest.mark.parametrize("block_n", [128, 256])
@pytest.mark.parametrize("M,N,K", _GEMM_CASES)
def test_gemm_plain_elementwise(F, M, N, K, block_n):
    torch.manual_seed(M * 7 + N * 3 + K)
    a, b = _operand(_randn(M, K)), _operand(_randn(N, K, scale=0.05))
    buf, out = _canary_out(M, N)
    F.gemm(a, b, out, M=M, N=N, K1=K, block_n=block_n, pair=0)
    ref = _mm(a, b.t())
    mag = _mm(a.abs(), b.abs().t())
    check("gemm", f"M{M} N{N} K{K} bn{block_n}", out, ref, gemm_bound(ref, mag, K))
    _assert_outside_untouched(buf, M, N, "gemm out")


@pytest.mark.parametrize("M,N,K,a_mn,b_mn", [
    (189, 688, 416, True, False), (257, 1376, 24, False, True), (4097, 264, 1368, True, True), (65, 2736, 640, True, True),
    (1, 264, 5504, False, True), (129, 8, 2736, True, False),
])
def test_gemm_mn_major_elementwise(F, M, N, K, a_mn, b_mn):
    """MN-major operands are ``[K, rows]``: their padding columns lie past M / N and their padding rows past K."""
    torch.manual_seed(M + N + K)
    a, b = _randn(M, K), _randn(N, K, scale=0.05)
    a_in = _operand(a.t()) if a_mn else _operand(a)
    b_in = _operand(b.t()) if b_mn else _operand(b)
    buf, out = _canary_out(M, N)
    F.gemm(a_in, b_in, out, M=M, N=N, K1=K, a1_mn=a_mn, b1_mn=b_mn, block_n=128)
    ref = _mm(a, b.t())
    check("gemm", f"mn-major M{M} N{N} K{K} a{int(a_mn)} b{int(b_mn)}", out, ref, gemm_bound(ref, _mm(a.abs(), b.abs().t()), K))
    _assert_outside_untouched(buf, M, N, "gemm out")


@pytest.mark.parametrize("block_n", [128, 256])
@pytest.mark.parametrize("M,N,K", [(189, 688, 1368), (4097, 264, 416), (1, 2736, 640), (257, 8, 24)])
def test_gemm_residual_alpha_bias(F, M, N, K, block_n):
    torch.manual_seed(K + N)
    a, b = _operand(_randn(M, K)), _operand(_randn(N, K, scale=0.05))
    res = _operand(_randn(M, N))
    bias = _randn(N)
    alpha = 0.37
    buf, out = _canary_out(M, N)
    F.gemm(a, b, out, M=M, N=N, K1=K, residual=res, alpha=alpha, bias=bias, block_n=block_n, pair=0)
    ref = alpha * _mm(a, b.t()) + res.to(F64) + bias.to(F64)
    mag = alpha * _mm(a.abs(), b.abs().t()) + res.to(F64).abs() + bias.to(F64).abs()
    check("gemm", f"residual+alpha+bias M{M} N{N} K{K} bn{block_n}", out, ref, gemm_bound(ref, mag, K, extra=3))
    _assert_outside_untouched(buf, M, N, "gemm out")


@pytest.mark.parametrize("out_dtype", [torch.float32, BF])
@pytest.mark.parametrize("M,N,K", [(257, 688, 416), (4097, 264, 24), (65, 1376, 2736), (1, 8, 5504)])
def test_gemm_accumulate(F, M, N, K, out_dtype):
    """``out += alpha * a b^T`` into an fp32 or bf16 output."""
    torch.manual_seed(M + K)
    a, b = _operand(_randn(M, K)), _operand(_randn(N, K, scale=0.05))
    buf, out = _canary_out(M, N, dtype=out_dtype)
    out.copy_(torch.randn(M, N, device="cuda"))
    before = out.to(F64)
    alpha = 2.0
    F.gemm(a, b, out, M=M, N=N, K1=K, accumulate=True, alpha=alpha, block_n=128)
    ref = before + alpha * _mm(a, b.t())
    mag = before.abs() + alpha * _mm(a.abs(), b.abs().t())
    check("gemm-accumulate", f"{str(out_dtype)[6:]} M{M} N{N} K{K}", out, ref,
          gemm_bound(ref, mag, K, out_bf16=out_dtype == BF, extra=2))
    _assert_outside_untouched(buf, M, N, "gemm accumulate out")


@pytest.mark.parametrize("split", [2, 7])
@pytest.mark.parametrize("M,N,K,mn", [(264, 416, 4097, True), (128, 688, 1368, True), (189, 264, 24, False), (65, 2736, 416, False)])
def test_gemm_split_k(F, M, N, K, mn, split):
    """Split-K with K not a multiple of split * 64 (uneven k-block shares, and splits that own no k-block at all when
    K = 24): the weight-gradient form reads both operands MN-major over the token dimension."""
    torch.manual_seed(K + split)
    a, b = _randn(M, K, scale=0.3), _randn(N, K)
    a_in = _operand(a.t()) if mn else _operand(a)
    b_in = _operand(b.t()) if mn else _operand(b)
    buf, out = _canary_out(M, N, dtype=torch.float32)
    out.copy_(torch.randn(M, N, device="cuda"))
    before = out.to(F64)
    F.gemm(a_in, b_in, out, M=M, N=N, K1=K, a1_mn=mn, b1_mn=mn, accumulate=True, split_k=split)
    ref = before + _mm(a, b.t())
    mag = before.abs() + _mm(a.abs(), b.abs().t())
    check("gemm-split-k", f"split{split} M{M} N{N} K{K} mn{int(mn)}", out, ref, gemm_bound(ref, mag, K, out_bf16=False, extra=split))
    _assert_outside_untouched(buf, M, N, "split-K out")


@pytest.mark.parametrize("G,Ng,K,M,r,block_n", [(2, 5504, 416, 189, 128, 256), (3, 1344, 640, 257, 64, 128), (2, 320, 24, 4097, 128, 0),
                                                  (3, 5504, 416, 65, 64, 128)])
def test_gemm_fused_lora_groups_elementwise(F, G, Ng, K, M, r, block_n):
    """``y_g = x W_g^T + u_g B_g^T`` per group; groups with a ragged last tile (5504 = 21.5 x 256)."""
    torch.manual_seed(G * Ng + M)
    N = G * Ng
    x, W = _operand(_randn(M, K)), _operand(_randn(N, K, scale=0.03))
    u, B = _operand(_randn(M, G * r)), _operand(_randn(N, r, scale=0.05))
    buf, out = _canary_out(M, N)
    F.gemm(x, W, out, M=M, N=N, K1=K, a2=u, b2=B, K2=r, n_per_group=Ng, a2_group_kofs=r, block_n=block_n)
    ref, mag = _mm(x, W.t()), _mm(x.abs(), W.abs().t())
    for g in range(G):
        sl, ul = slice(g * Ng, (g + 1) * Ng), slice(g * r, (g + 1) * r)
        ref[:, sl] += _mm(u[:, ul], B[sl].t())
        mag[:, sl] += _mm(u[:, ul].abs(), B[sl].abs().t())
    check("gemm-groups", f"G{G} Ng{Ng} K{K} M{M} r{r} bn{block_n}", out, ref, gemm_bound(ref, mag, K + r))
    _assert_outside_untouched(buf, M, N, "grouped gemm out")


def test_gemm_group_width_not_multiple_of_64_is_rejected(F):
    """An intermediate size such as 688 cannot be a group width of the stacked GEMM: the binding says so."""
    x, W = _randn(64, 128), _randn(2 * 688, 128)
    with pytest.raises(RuntimeError, match="n_per_group must be a multiple of 64"):
        F.gemm(x, W, M=64, N=2 * 688, K1=128, n_per_group=688)


@pytest.mark.parametrize("M,N,K,a_mn,b_mn", [(257, 688, 416, False, False), (189, 1376, 1368, False, True), (4097, 2736, 640, True, False),
                                             (129, 264, 2736, True, True), (1, 8, 24, False, False)])
def test_gemm_cta_pair_ragged(F, M, N, K, a_mn, b_mn):
    """CTA pairs (256-row tiles) with M not a multiple of 256, plus a residual."""
    torch.manual_seed(M * 3 + K)
    a, b = _randn(M, K), _randn(N, K, scale=0.05)
    a_in = _operand(a.t()) if a_mn else _operand(a)
    b_in = _operand(b.t()) if b_mn else _operand(b)
    res = _operand(_randn(M, N))
    buf, out = _canary_out(M, N)
    F.gemm(a_in, b_in, out, M=M, N=N, K1=K, a1_mn=a_mn, b1_mn=b_mn, residual=res, block_n=256, pair=1)
    ref = _mm(a, b.t()) + res.to(F64)
    mag = _mm(a.abs(), b.abs().t()) + res.to(F64).abs()
    check("gemm-pair", f"M{M} N{N} K{K} a{int(a_mn)} b{int(b_mn)}", out, ref, gemm_bound(ref, mag, K, extra=1))
    _assert_outside_untouched(buf, M, N, "pair out")


@pytest.mark.parametrize("M,N,K,pair", [(189, 688, 416, 0), (4097, 1376, 640, 1), (1, 264, 1376, 0), (257, 2736, 2736, 1)])
def test_gemm_fp8_ragged(C, F, M, N, K, pair):
    """E4M3 frozen-weight GEMM with the bf16 LoRA branch and a residual, against the float64 product of the *dequantised*
    operands (the quantisation itself is not an error of the GEMM)."""
    torch.manual_seed(K + M)
    r = 128
    x, W = _randn(M, K), _randn(N, K, scale=0.05)
    u, B = _operand(_randn(M, r)), _operand(_randn(N, r, scale=0.05))
    res = _operand(_randn(M, N))
    f32 = lambda v: torch.tensor([v], dtype=torch.float32, device="cuda")  # noqa: E731
    scratch, sw, inv_sw = f32(0.0), f32(0.0), f32(0.0)
    # byte operands in padded buffers too; 0x7F is an E4M3 NaN
    _, W8 = _padded(N, K, pad_cols=16, dtype=torch.uint8, fill=0x7F)
    C.fp8_quantize_weight(W, W8, scratch, sw, inv_sw)
    sx = float(x.float().abs().max()) / 448.0
    _, x8 = _padded(M, K, pad_cols=16, dtype=torch.uint8, fill=0x7F)
    C.fp8_quantize_act(x, x8, f32(1.0 / sx), f32(0.0))
    xq = x8.view(torch.float8_e4m3fn).to(F64) * sx
    Wq = W8.view(torch.float8_e4m3fn).to(F64) * float(sw)
    alpha = sx * float(sw)
    u_s = (u.float() / alpha).to(BF)
    buf, out = _canary_out(M, N)
    F.gemm(x8, W8, out, M=M, N=N, K1=K, a2=u_s, b2=B, K2=r, residual=res, fp8=True, alpha_dev=f32(alpha),
           block_n=256 if pair else 0, pair=pair)
    ref = xq @ Wq.t() + alpha * _mm(u_s, B.t()) + res.to(F64)
    mag = xq.abs() @ Wq.abs().t() + alpha * _mm(u_s.abs(), B.abs().t()) + res.to(F64).abs()
    check("gemm-fp8", f"M{M} N{N} K{K} pair{pair}", out, ref, gemm_bound(ref, mag, K + r, extra=2))
    _assert_outside_untouched(buf, M, N, "fp8 out")


# ------------------------------------------------------------------------------------------------------------- lora_dx
def _lora_dx_ref(dy, W, du, A, G, r, p, seed, keys):
    M, N = du.shape[0], A.shape[1]
    ref, mag = None, None
    if dy is not None:
        ref, mag = _mm(dy, W), _mm(dy.abs(), W.abs())
    lora_ref = torch.zeros(M, N, dtype=F64, device="cuda")
    lora_mag = torch.zeros_like(lora_ref)
    from relora_b200.ops import reference as rf

    for g in range(G):
        sl = slice(g * r, (g + 1) * r)
        part, pmag = _mm(du[:, sl], A[sl]), _mm(du[:, sl].abs(), A[sl].abs())
        if p > 0:
            keep = rf.dropout_keep_mask(rf.mix_seed(seed, keys[g]), M, N, p, device="cuda").to(F64)
            part, pmag = part * keep / (1.0 - p), pmag * keep / (1.0 - p)
        lora_ref += part
        lora_mag += pmag
    return ref, mag, lora_ref, lora_mag


@pytest.mark.parametrize("G,r,M,N,Kb,p", [
    (1, 128, 189, 416, 1376, 0.1), (2, 64, 4097, 640, 1368, 0.0), (3, 128, 4097, 2048, 2736, 0.1), (1, 64, 1, 5504, 2048, 0.1),
    (3, 64, 189, 5504, 2048, 0.1), (2, 128, 1, 416, 688, 0.1), (3, 128, 189, 640, 416, 0.0),
])
def test_lora_dx_elementwise(C, G, r, M, N, Kb, p):
    """dx = dy W + sum_g keep_g * (du_g A_g) / (1 - p) (fused form; Kb >= 1536 with M > 128 takes the CTA-pair kernel), and
    the two-kernel form that adds the masked low-rank terms to a given bf16 base."""
    torch.manual_seed(G * 11 + M + N)
    dy, W = _operand(_randn(M, Kb)), _operand(_randn(Kb, N, scale=0.05))
    du, A = _operand(_randn(M, G * r)), _operand(_randn(G * r, N, scale=0.05))
    seed_v, keys = 1234567, [11, 22, 33][:G]
    seed = torch.tensor([seed_v], dtype=torch.int32, device="cuda")
    base_ref, base_mag, lora_ref, lora_mag = _lora_dx_ref(dy, W, du, A, G, r, p, seed_v, keys)
    buf, out = _canary_out(M, N, pad_rows=2, pad_cols=8)
    C.lora_dx(dy, W, du, A, out, seed if p > 0 else None, keys, p)
    ref = base_ref + lora_ref
    # two accumulators (Kb and r long) summed in fp32 with the 1/(1-p) scale: 3 more fp32 roundings; the fused kernel also
    # keeps the masked low-rank sum packed as bf16 in registers until the frozen-path product is ready (one more 2^-8)
    lora_acc = (r + 4) * U24 * lora_mag
    bound = U8 * ref.abs() + (Kb + 2) * U24 * base_mag + lora_acc + U8 * (lora_ref.abs() + lora_acc)
    check("lora_dx", f"fused G{G} r{r} M{M} N{N} Kb{Kb} p{p}", out, ref, bound)
    _assert_outside_untouched(buf, M, N, "lora_dx out")
    base = _operand(base_ref.to(BF))
    buf2, out2 = _canary_out(M, N, pad_rows=2, pad_cols=8)
    C.lora_dx(None, None, du, A, out2, seed if p > 0 else None, keys, p, base)
    ref2 = base.to(F64) + lora_ref
    bound2 = U8 * ref2.abs() + 2 * U24 * base.to(F64).abs() + (r + 4) * U24 * lora_mag
    check("lora_dx", f"base G{G} r{r} M{M} N{N} p{p}", out2, ref2, bound2)
    _assert_outside_untouched(buf2, M, N, "lora_dx (base) out")


# ----------------------------------------------------------------------------------------------------------- attention
def _qkv_views(q_all, B, T, nh, hd):
    x = q_all.to(F64).view(B, T, 3, nh, hd)
    return tuple(x[:, :, i].transpose(1, 2) for i in range(3))  # [B, nh, T, hd]


def _attn_ref(qkv, dout, out_k, B, T, nh, hd, scale):
    """float64 causal attention, its lse (log2 units, as the kernel stores it) and gradients, with per-element bounds."""
    q, k, v = _qkv_views(qkv, B, T, nh, hd)
    causal = torch.ones(T, T, dtype=torch.bool, device="cuda").tril()
    s = (q @ k.transpose(-1, -2)) * scale
    s = s.masked_fill(~causal, float("-inf"))
    m = s.amax(-1, keepdim=True)
    e = torch.exp(s - m)
    l = e.sum(-1, keepdim=True)
    P = e / l
    o = P @ v
    lse = (m + torch.log(l)).squeeze(-1) / math.log(2.0)
    # fp32 error of a score: hd products and the scale; it moves exp(s) by that much relative
    qk_abs = (q.abs() @ k.abs().transpose(-1, -2)) * scale
    sig = float(((hd + 2) * U24 * qk_abs).masked_fill(~causal, 0).amax())
    # relative error of one probability as the kernel uses it: bf16 rounding of P (2^-8), ex2.approx (2^-22), the running
    # max rescales (one per 64-key block), the row sum (T terms) and the score error
    eps_p = U8 + (T / 64 + 4) * 2.0 ** -22 + (T + 2) * U24 + 2 * sig
    bnd = {}
    bnd["out"] = U8 * o.abs() + eps_p * (P @ v.abs())
    bnd["lse"] = 4 * 2.0 ** -22 + (T + 2) * U24 + U24 * lse.abs() + 2 * sig / math.log(2.0)
    ref = {"out": o, "lse": lse}
    if dout is not None:
        do = dout.to(F64).view(B, T, nh, hd).transpose(1, 2)
        ok = out_k.to(F64).view(B, T, nh, hd).transpose(1, 2)
        dP = do @ v.transpose(-1, -2)
        delta = (do * o).sum(-1, keepdim=True)
        dS = P * (dP - delta)
        # the kernel's delta comes from its own bf16 output: |do|.|o| * 2^-8 covers that, hd-term fp32 sums the rest
        D = (do.abs() * ok.abs()).sum(-1, keepdim=True)
        dov = do.abs() @ v.abs().transpose(-1, -2)
        E = P * ((U8 + eps_p) * (dP.abs() + delta.abs()) + (U8 + (hd + 2) * U24) * D + (hd + 2) * U24 * dov)
        dSa = dS.abs()
        ref["dq"] = scale * dS @ k
        ref["dk"] = scale * dS.transpose(-1, -2) @ q
        ref["dv"] = P.transpose(-1, -2) @ do
        acc = (T + 2) * U24
        bnd["dq"] = U8 * ref["dq"].abs() + scale * (E @ k.abs() + acc * dSa @ k.abs())
        bnd["dk"] = U8 * ref["dk"].abs() + scale * (E.transpose(-1, -2) @ q.abs() + acc * dSa.transpose(-1, -2) @ q.abs())
        bnd["dv"] = U8 * ref["dv"].abs() + (eps_p + acc) * (P.transpose(-1, -2) @ do.abs())
    return ref, bnd


class _Attn:
    """Runs the kernels on NaN-padded inputs with canary-filled outputs (``buf[:B*T]`` views, padded leading dimensions)."""

    def __init__(self, C, B, T, nh, hd):
        self.C, self.B, self.T, self.nh, self.hd = C, B, T, nh, hd
        self.h = nh * hd
        self.scale = 1.0 / math.sqrt(hd)

    def fwd(self, qkv):
        B, T, nh, h = self.B, self.T, self.nh, self.h
        obuf, out = _canary_out(B * T, h, pad_rows=5, pad_cols=8)
        lbuf = torch.empty(B * nh * T + 37, device="cuda", dtype=torch.float32)
        lbuf.view(torch.int32).fill_(CANARY32)
        lse = lbuf[: B * nh * T].view(B, nh, T)
        self.C.attention_fwd(qkv, out, lse, B, T, nh, self.hd, self.scale)
        _assert_outside_untouched(obuf, B * T, h, "attention out")
        assert bool((lbuf[B * nh * T:].view(torch.int32) == CANARY32).all()), "attention lse: wrote past B*nh*T"
        return out, lse

    def bwd(self, qkv, out, dout, lse, use_ws):
        B, T, nh, h = self.B, self.T, self.nh, self.h
        dbuf, dqkv = _canary_out(B * T, 3 * h, pad_rows=5, pad_cols=8)
        delta = torch.empty(B, nh, T, device="cuda", dtype=torch.float32)
        ws = None
        if use_ws:
            ws = torch.full((self.C.attention_ds_workspace_elems(B, T, nh),), float("nan"), device="cuda", dtype=BF)
        self.C.attention_bwd(qkv, out, dout, lse, delta, dqkv, B, T, nh, self.hd, self.scale, ws)
        _assert_outside_untouched(dbuf, B * T, 3 * h, "attention dqkv")
        return dqkv


_ATTN_CASES = sorted({
    *[(3 if T < 1000 else 2, T, 3 if T < 1000 else 2, 64) for T in (1, 7, 63, 65, 127, 129, 200, 1000, 2048, 2049)],
    *[(3, 129, 2, hd) for hd in (8, 16, 24, 32, 40, 48, 56, 64)],
    (2, 2049, 2, 48), (2, 200, 3, 40),
})


@pytest.mark.parametrize("B,T,nh,hd", _ATTN_CASES)
def test_attention_elementwise(C, B, T, nh, hd):
    """Forward (out, lse) and both backward forms (dQ recomputed / dQ from the stored dS^T tiles) against float64."""
    torch.manual_seed(T * 13 + hd + B)
    run = _Attn(C, B, T, nh, hd)
    h = nh * hd
    qkv = _operand(_randn(B * T, 3 * h), pad_rows=70)
    dout = _operand(_randn(B * T, h, scale=0.5), pad_rows=70)
    out, lse = run.fwd(qkv)
    ref, bnd = _attn_ref(qkv, dout, out, B, T, nh, hd, run.scale)
    case = f"B{B} T{T} nh{nh} hd{hd}"
    check("attention-fwd", case, out.view(B, T, nh, hd).transpose(1, 2), ref["out"], bnd["out"], _where_attn)
    check("attention-lse", case, lse, ref["lse"], bnd["lse"], lambda s, i: _where_attn(s + (1,), i))
    for use_ws in (False, True):
        d5 = run.bwd(qkv, out, dout, lse, use_ws).view(B, T, 3, nh, hd)
        for i, name in enumerate(("dq", "dk", "dv")):
            check("attention-bwd", f"{case} {name} {'dS-ws' if use_ws else 'recompute'}", d5[:, :, i].transpose(1, 2),
                  ref[name], bnd[name], _where_attn)


def _perturbed(qkv, rows, cols, factor=30.0):
    """``qkv`` (padded like the original) with ``[rows, cols]`` multiplied by ``factor``."""
    t = qkv.clone()
    t[rows, cols] = (t[rows, cols].float() * factor).to(BF)
    return _operand(t, pad_rows=70)


@pytest.mark.parametrize("B,T,nh,hd", [(3, 65, 2, 64), (3, 200, 2, 40), (2, 1000, 2, 64), (3, 129, 2, 8), (2, 2049, 2, 48), (3, 7, 2, 24)])
def test_attention_batch_isolation_bitwise(C, B, T, nh, hd):
    """The tail tile of batch b reads rows of batch b+1 through the packed [B*T, 3*nh*hd] tensor map; only the kernel's
    masks keep them out.  Scaling batch b+1's q/k/v (and dO) by 30 must leave batch b's out, lse and dq/dk/dv identical."""
    torch.manual_seed(T + hd)
    run = _Attn(C, B, T, nh, hd)
    h = nh * hd
    qkv = _operand(_randn(B * T, 3 * h), pad_rows=70)
    dout = _operand(_randn(B * T, h, scale=0.5), pad_rows=70)
    out, lse = run.fwd(qkv)
    grads = {ws: run.bwd(qkv, out, dout, lse, ws) for ws in (False, True)}
    for b in sorted({0, B - 2}):
        nxt = slice((b + 1) * T, (b + 2) * T)
        qkv2 = _perturbed(qkv, nxt, slice(None))
        dout2 = _perturbed(dout, nxt, slice(None))
        out2, lse2 = run.fwd(qkv2)
        rows = slice(b * T, (b + 1) * T)
        assert torch.equal(out2[rows], out[rows]), f"batch {b} out changed with batch {b + 1}"
        assert torch.equal(lse2[b], lse[b]), f"batch {b} lse changed with batch {b + 1}"
        for ws in (False, True):
            d2 = run.bwd(qkv2, out2, dout2, lse2, ws)
            assert torch.equal(d2[rows], grads[ws][rows]), f"batch {b} dqkv (ds workspace {ws}) changed with batch {b + 1}"


@pytest.mark.parametrize("B,T,nh,hd", [(2, 65, 2, 64), (3, 200, 2, 40), (2, 1000, 2, 64), (2, 129, 3, 8), (2, 2049, 2, 48), (3, 7, 2, 24)])
def test_attention_causality_bitwise(C, B, T, nh, hd):
    """Keys / values after position t must not change out / lse rows <= t; queries / dO before position j must not
    change dk / dv (nor dq) of rows >= j.  Both positions sit inside a tile."""
    torch.manual_seed(T * 5 + hd)
    run = _Attn(C, B, T, nh, hd)
    h = nh * hd
    qkv = _operand(_randn(B * T, 3 * h), pad_rows=70)
    dout = _operand(_randn(B * T, h, scale=0.5), pad_rows=70)
    out, lse = run.fwd(qkv)
    t, j = (2 * T) // 3, (T + 1) // 3
    rows_after = torch.cat([torch.arange(b * T + t + 1, (b + 1) * T) for b in range(B)]).cuda()
    rows_upto = torch.cat([torch.arange(b * T, b * T + t + 1) for b in range(B)]).cuda()
    qkv_k = _perturbed(qkv, rows_after[:, None], torch.arange(h, 3 * h, device="cuda")[None, :])
    out_k, lse_k = run.fwd(qkv_k)
    assert torch.equal(out_k[rows_upto], out[rows_upto]), f"out rows <= {t} see later keys"
    assert torch.equal(lse_k[:, :, : t + 1], lse[:, :, : t + 1]), f"lse rows <= {t} see later keys"
    rows_before = torch.cat([torch.arange(b * T, b * T + j) for b in range(B)]).cuda()
    rows_from = torch.cat([torch.arange(b * T + j, (b + 1) * T) for b in range(B)]).cuda()
    qkv_q = _perturbed(qkv, rows_before[:, None], torch.arange(0, h, device="cuda")[None, :])
    dout_q = _perturbed(dout, rows_before[:, None], torch.arange(0, h, device="cuda")[None, :])
    out_q, lse_q = run.fwd(qkv_q)
    for ws in (False, True):
        g0 = run.bwd(qkv, out, dout, lse, ws)
        g1 = run.bwd(qkv_q, out_q, dout_q, lse_q, ws)
        assert torch.equal(g1[rows_from], g0[rows_from]), f"dq/dk/dv rows >= {j} (ds workspace {ws}) see earlier queries"


@pytest.mark.parametrize("hd", [72, 12])
def test_attention_unsupported_head_dim_is_rejected(C, hd):
    B, T, nh = 1, 64, 2
    qkv = _randn(B * T, 3 * nh * hd)
    out = torch.empty(B * T, nh * hd, device="cuda", dtype=BF)
    lse = torch.empty(B, nh, T, device="cuda", dtype=torch.float32)
    with pytest.raises(RuntimeError, match="head_dim"):
        C.attention_fwd(qkv, out, lse, B, T, nh, hd, 0.1)


# ------------------------------------------------------------------------------------------------------------- RMSNorm
_NORM_CASES = sorted({
    *[(33, H) for H in (128, 416, 640, 1000, 1032, 2048, 2056, 2560, 8192)],
    *[(M, 640) for M in (1, 5, 33, 4097)], *[(M, 2560) for M in (1, 5, 4097)], (4097, 416), (4097, 2048), (4097, 8192),
})


@pytest.mark.parametrize("M,H", _NORM_CASES)
def test_rmsnorm_elementwise(C, F, M, H):
    """Forward (+ two dropout copies, + the fp8 copy where H <= 2048) and backward with ``dx_add``, on both the warp-per-row
    kernels and the block-per-row fallback (taken for H > 2048, and for any H when dw is not 16-byte aligned).  Row 0 is
    all zeros (a padding row: rstd = 1/sqrt(eps))."""
    from relora_b200.ops import reference as rf

    torch.manual_seed(M + H)
    eps, p, keys = 1e-6, 0.1, [5, 9]
    x = _randn(M, H, scale=1.5)
    x[0] = 0
    w = (1 + 0.1 * torch.randn(H, device="cuda")).to(BF)
    ybuf = torch.empty(M + 2, H, device="cuda", dtype=BF)
    ybuf.view(torch.int16).fill_(CANARY16)
    y, rstd = ybuf[:M], torch.empty(M, device="cuda", dtype=torch.float32)
    xd = torch.empty(M, 2 * H, device="cuda", dtype=BF)
    seed = torch.tensor([4242], dtype=torch.int32, device="cuda")
    f32 = lambda v: torch.tensor([v], dtype=torch.float32, device="cuda")  # noqa: E731
    fp8 = H <= 2048 and H % 16 == 0  # the standalone quantiser, the bit-exact reference of this copy, takes multiples of 16
    q8, inv, am = (torch.empty(M, H, dtype=torch.uint8, device="cuda"), f32(448.0 / 8.0), f32(0.0)) if fp8 else (None, None, None)
    C.rmsnorm_fwd(x, w, y, rstd, eps, xd, seed, keys, p, q8, inv, am)
    assert bool((ybuf[M:].view(torch.int16) == CANARY16).all()), "rmsnorm y: wrote past M rows"
    # rstd against float64 (H-term fp32 sum, the division and rsqrt: a few ulp)
    xf = x.to(F64)
    rs_ref = 1.0 / torch.sqrt((xf * xf).mean(-1) + eps)
    check("rmsnorm-rstd", f"M{M} H{H}", rstd, rs_ref, (H + 8) * U24 * rs_ref)
    # y = bf16(w * bf16(x * rstd)) with the kernel's fp32 rstd: every rounding is mirrored, so it is exact
    xhat_b = (x.float() * rstd[:, None]).to(BF)
    y_ref = (w.float() * xhat_b.float()).to(BF)
    assert torch.equal(y, y_ref), f"rmsnorm y: first mismatch at {(y != y_ref).nonzero()[0].tolist()}"
    inv_keep = torch.tensor(1.0 / (1.0 - p), dtype=torch.float32, device="cuda")  # the kernel's fp32 1/(1-p)
    for g, k in enumerate(keys):
        keep = rf.dropout_keep_mask(rf.mix_seed(4242, k), M, H, p, device="cuda")
        want = torch.where(keep, (y.float() * inv_keep).to(BF), torch.zeros_like(y))
        assert torch.equal(xd.view(M, 2, H)[:, g], want), f"dropout copy {g}"
    if fp8:
        rq, ram = torch.empty_like(q8), f32(0.0)
        C.fp8_quantize_act(y, rq, inv, ram)
        assert torch.equal(q8, rq) and float(am) == float(ram)

    dy, add = _randn(M, H), _randn(M, H)
    rs = rstd.to(F64)[:, None]
    wf, dyf = w.to(F64), dy.to(F64)
    g_ = dyf * wf
    dot = (g_ * xf * rs).sum(-1, keepdim=True) / H
    dx_ref = rs * (g_ - xf * rs * dot) + add.to(F64)
    s_abs = (g_ * xf * rs).abs().sum(-1, keepdim=True)
    # fp32: the H-term dot (H * 2^-24 of sum|g x rstd|), then a handful of roundings per element
    dx_bound = U8 * dx_ref.abs() + U24 * (8 * rs * (g_.abs() + xf.abs() * rs * dot.abs()) + (H + 4) * rs * rs * xf.abs() * s_abs / H
                                          + 2 * add.to(F64).abs())
    dw_init = torch.randn(H, device="cuda")
    dw_ref = dw_init.to(F64) + (dyf * xhat_b.to(F64)).sum(0)
    dw_bound = (M + 4) * U24 * (dw_init.to(F64).abs() + (dyf * xhat_b.to(F64)).abs().sum(0))
    ws, tk = F.norm_workspace(x.device, H)
    for form in ("warp", "block") if H <= 2048 else ("block",):
        dxbuf = torch.empty(M + 2, H, device="cuda", dtype=BF)
        dxbuf.view(torch.int16).fill_(CANARY16)
        dx = dxbuf[:M]
        dwbuf = torch.empty(H + 8, device="cuda", dtype=torch.float32)
        dw = dwbuf[:H] if form == "warp" else dwbuf[1:H + 1]  # a dw that is not 16-byte aligned selects the block kernel
        dw.copy_(dw_init)
        C.rmsnorm_bwd(dy, x, w, rstd, add, dx, dw, ws, tk)
        check("rmsnorm-dx", f"{form} M{M} H{H}", dx, dx_ref, dx_bound)
        check("rmsnorm-dw", f"{form} M{M} H{H}", dw, dw_ref, dw_bound)
        assert bool((dxbuf[M:].view(torch.int16) == CANARY16).all()), "rmsnorm dx: wrote past M rows"


# -------------------------------------------------------------------------------------------------------- cross entropy
def _ce_eps(V):
    """Relative error of one softmax probability in the one-block-per-row kernel, apart from the exp argument's own
    rounding (2^-24 of |x - max|, added by the caller): __expf (2^-22) and the row sum, which each of the 512 threads
    accumulates over V/512 columns before a 512-way tree (V/512 + 10 fp32 additions on any path)."""
    return 4 * 2.0 ** -22 + (V / 512 + 12) * U24


def _ce_grad_bound(x, grad, gs, valid):
    """Per-element bound of the in-place gradient ``bf16(gs * (softmax(x) - onehot))`` of ``ce_kernel``.

    Every rounding in the kernel is relative: P carries ``_ce_eps`` plus 2^-24 of |x - max| (the exp argument is rounded
    once more when __expf scales it by log2 e), the ``- 1`` at the label and the ``* grad_scale`` add 2^-24 each, and the
    bf16 store 2^-8.  The only absolute errors come from underflow: __expf may flush a result below 2^-126 to zero, which
    after the multiplies by 1/sum (<= 1, the row maximum contributes exp(0) = 1 to the sum) and by grad_scale is at most
    gs * 2^-126; the fp32 multiplies underflow gradually (2^-150) and a bf16 subnormal rounds to within 2^-134 -- together
    below 2^-133.  Rows with an ignored label must be exactly zero."""
    V = x.shape[-1]
    mx = x.amax(-1, keepdim=True)
    P = torch.exp(x - mx - torch.log(torch.exp(x - mx).sum(-1, keepdim=True)))
    eps_p = _ce_eps(V) + 2 * U24 * (x - mx).abs()
    floor = gs * 2.0 ** -126 + 2.0 ** -133
    bound = (U8 + 2 * U24) * grad.abs() + (1 + U8) * gs * eps_p * P + floor
    return torch.where(valid[:, None], bound, torch.zeros_like(bound))


@pytest.mark.parametrize("V", [8, 1000, 32100, 50257, 50304, 65536])
def test_cross_entropy_elementwise(C, V):
    """Loss and in-place d(logits) against float64: labels V-1 and in the scalar tail (V % 8 columns), an ignored row,
    rows of +-80 with one +1e4 outlier, grad_scale != 1, and canaries in the padding columns [V, ld)."""
    torch.manual_seed(V)
    M, ld = 24, (V + 7) // 8 * 8 + 8
    buf = torch.empty(M + 1, ld, device="cuda", dtype=BF)
    buf.view(torch.int16).fill_(CANARY16)
    logits = buf[:M, :V]
    logits.copy_(_randn(M, V, scale=3.0))
    logits[3] = (torch.randint(0, 2, (V,), device="cuda") * 160 - 80).to(BF)
    logits[4] = logits[3]
    logits[4, V // 2] = 1e4
    labels = torch.randint(0, V, (M,), device="cuda")
    labels[0], labels[1], labels[2] = V - 1, V - 1 - (V % 8) // 2, -100
    labels[4] = V - 1 if V // 2 != V - 1 else 0
    x = logits.to(F64)
    loss, cnt = torch.tensor([1.5], device="cuda"), torch.tensor([2.0], device="cuda")
    gs = 0.37
    C.cross_entropy_fwd_bwd(logits, labels, V, gs, -100, loss, cnt)
    valid = labels != -100
    mx = x.amax(-1, keepdim=True)
    lse = mx + torch.log(torch.exp(x - mx).sum(-1, keepdim=True))
    P = torch.exp(x - lse)
    lab = labels.clamp(min=0)
    row_loss = (lse.squeeze(-1) - x.gather(1, lab[:, None]).squeeze(-1))[valid]
    grad = P.clone()
    grad[torch.arange(M, device="cuda"), lab] -= 1.0
    grad = torch.where(valid[:, None], grad * gs, torch.zeros_like(grad))
    check("cross-entropy-grad", f"V{V}", logits, grad, _ce_grad_bound(x, grad, gs, valid))
    assert float(cnt) == 2.0 + float(valid.sum())
    loss_ref = 1.5 + float(row_loss.sum())
    loss_bound = (M + 4) * U24 * (1.5 + float(row_loss.abs().sum())) + float(valid.sum()) * (
        _ce_eps(V) + U24 * float(lse.abs().max()) + 2 * U24 * float((x - mx).abs().max()))
    check("cross-entropy-loss", f"V{V}", loss, torch.tensor([loss_ref], dtype=F64, device="cuda"),
          torch.tensor([loss_bound], dtype=F64, device="cuda"))
    _assert_outside_untouched(buf, M, V, "cross entropy")


@pytest.mark.parametrize("V", [1000, 50257])
def test_cross_entropy_all_rows_ignored(C, V):
    M, ld = 9, (V + 7) // 8 * 8 + 8
    buf = torch.empty(M, ld, device="cuda", dtype=BF)
    buf.view(torch.int16).fill_(CANARY16)
    logits = buf[:, :V]
    logits.copy_(_randn(M, V))
    labels = torch.full((M,), -100, device="cuda", dtype=torch.long)
    loss, cnt = torch.zeros(1, device="cuda"), torch.zeros(1, device="cuda")
    C.cross_entropy_fwd_bwd(logits, labels, V, 1.0, -100, loss, cnt)
    assert float(loss) == 0.0 and float(cnt) == 0.0
    assert bool((logits.float() == 0).all())
    _assert_outside_untouched(buf, M, V, "cross entropy (all ignored)")


# ------------------------------------------------------------------------------------------------------ negative controls
def test_negative_control_gemm_comparator(F):
    """The GEMM comparator rejects (a) one 128x128 tile missing its last K-block and (b) the last 8 columns of a ragged N
    off by 1 %, while it accepts the kernel's own output."""
    torch.manual_seed(0)
    M, N, K = 1000, 520, 640
    a, b = _randn(M, K), _randn(N, K, scale=0.05)
    ref, mag = _mm(a, b.t()), _mm(a.abs(), b.abs().t())
    bound = gemm_bound(ref, mag, K)
    got = F.gemm(a, b, block_n=128)
    assert _excess(got, ref, bound)[0] <= 1.0
    wrong = ref.clone()
    wrong[128:256, 256:384] -= _mm(a[128:256, K - 64:], b[256:384, K - 64:].t())
    worst, i = _excess(wrong.to(BF), ref, bound)
    assert worst > 1.0, worst
    assert "tile_m 1, tile_n 2" in _where_tile((M, N), i)
    wrong = ref.clone()
    wrong[:, N - 8:] *= 1.01
    assert _excess(wrong.to(BF), ref, bound)[0] > 1.0
    # fp32 output (no 2^-8 term): a dropped K-block is far outside the accumulation bound
    bound32 = gemm_bound(ref, mag, K, out_bf16=False)
    wrong = ref.clone()
    wrong[:128, :128] -= _mm(a[:128, K - 64:], b[:128, K - 64:].t())
    assert _excess(wrong.float(), ref, bound32)[0] > 1.0


def test_negative_control_lora_dx_comparator(C):
    """A dropout mask applied to the wrong group (keys swapped) is rejected."""
    torch.manual_seed(1)
    G, r, M, N, Kb, p = 2, 64, 189, 416, 688, 0.1
    dy, W = _randn(M, Kb), _randn(Kb, N, scale=0.05)
    du, A = _randn(M, G * r), _randn(G * r, N, scale=0.05)
    base_ref, base_mag, lora_ref, lora_mag = _lora_dx_ref(dy, W, du, A, G, r, p, 77, [1, 2])
    ref = base_ref + lora_ref
    lora_acc = (r + 4) * U24 * lora_mag
    bound = U8 * ref.abs() + (Kb + 2) * U24 * base_mag + lora_acc + U8 * (lora_ref.abs() + lora_acc)
    _, _, lora_sw, _ = _lora_dx_ref(dy, W, du, A, G, r, p, 77, [2, 1])
    assert _excess((base_ref + lora_sw).to(BF), ref, bound)[0] > 1.0


def test_negative_control_attention_comparator():
    """One attention row that includes one extra (future) key, and dK / dV that miss the diagonal query (a causal mask off
    by one), are rejected.  The leaked key sits in row 5, where it takes about 1/7 of the row's mass; at T of a few hundred
    and more a single leaked key moves a row by about 1/T, inside the rounding bound of P, and only the bitwise isolation
    and causality tests see it."""
    torch.manual_seed(2)
    B, T, nh, hd = 2, 129, 2, 64
    scale = 1.0 / math.sqrt(hd)
    qkv = _randn(B * T, 3 * nh * hd)
    dout = _randn(B * T, nh * hd, scale=0.5)
    ref0, _ = _attn_ref(qkv, None, None, B, T, nh, hd, scale)
    out_bf = ref0["out"].transpose(1, 2).reshape(B * T, nh * hd).to(BF)
    ref, bnd = _attn_ref(qkv, dout, out_bf, B, T, nh, hd, scale)
    assert _excess(ref["out"].to(BF), ref["out"], bnd["out"])[0] <= 1.0
    # row t of batch 1, head 0 sees key t+1 as well
    q, k, v = _qkv_views(qkv, B, T, nh, hd)
    t = 5
    s = (q[1, 0, t] @ k[1, 0, : t + 2].t()) * scale
    leaked = torch.softmax(s, -1) @ v[1, 0, : t + 2]
    wrong = ref["out"].clone()
    wrong[1, 0, t] = leaked
    worst, i = _excess(wrong.to(BF), ref["out"], bnd["out"])
    assert worst > 1.0 and "batch 1, head 0, row 5" in _where_attn(tuple(wrong.shape), i), (worst, i)
    s_all = (q @ k.transpose(-1, -2)) * scale
    causal = torch.ones(T, T, dtype=torch.bool, device="cuda").tril()
    P = torch.softmax(s_all.masked_fill(~causal, float("-inf")), -1)
    do = dout.to(F64).view(B, T, nh, hd).transpose(1, 2)
    dS = P * (do @ v.transpose(-1, -2) - (do * ref["out"]).sum(-1, keepdim=True))
    P_diag, dS_diag = P.diagonal(dim1=-2, dim2=-1)[..., None], dS.diagonal(dim1=-2, dim2=-1)[..., None]
    assert _excess(ref["dk"] - scale * dS_diag * q, ref["dk"], bnd["dk"])[0] > 1.0
    assert _excess(ref["dv"] - P_diag * do, ref["dv"], bnd["dv"])[0] > 1.0


def test_negative_control_rmsnorm_and_ce_comparators():
    """RMSNorm dw that misses the last row is rejected.  The cross-entropy gradient bound (the one the kernel test uses)
    accepts the correctly rounded gradient but rejects scalar-tail columns with a 1 % wrong normaliser, a 10 % error on
    the small-probability columns (P < 1e-6, most of a large vocabulary) and small probabilities flushed to zero."""
    torch.manual_seed(3)
    M, H = 33, 1000
    dy = _randn(M, H).to(F64)
    xh = _randn(M, H).to(F64)
    dw_ref = (dy * xh).sum(0)
    bound = (M + 4) * U24 * (dy * xh).abs().sum(0)
    assert _excess((dy[:-1] * xh[:-1]).sum(0), dw_ref, bound)[0] > 1.0
    V, M, gs = 32100, 4, 0.37
    x = _randn(M, V, scale=3.0).to(F64)
    labels = torch.randint(0, V, (M,), device="cuda")
    P = torch.softmax(x, -1)
    grad = P.clone()
    grad[torch.arange(M, device="cuda"), labels] -= 1.0
    grad = grad * gs
    bound = _ce_grad_bound(x, grad, gs, torch.ones(M, dtype=torch.bool, device="cuda"))
    assert _excess(grad.to(BF), grad, bound)[0] <= 1.0
    wrong = grad.clone()
    wrong[:, V - V % 8:] *= 1.01
    assert _excess(wrong.to(BF), grad, bound)[0] > 1.0
    small = P < 1e-6
    assert float(small.double().mean()) > 0.5
    wrong = torch.where(small, grad * 1.1, grad)
    assert _excess(wrong.to(BF), grad, bound)[0] > 1.0
    wrong = torch.where(P < 1e-7, torch.zeros_like(grad), grad)
    assert _excess(wrong.to(BF), grad, bound)[0] > 1.0


# ------------------------------------------------------------------------------------------------ Pythia masked eval
def test_pythia_batched_eval_with_padding_mask_matches_reference():
    """Batched eval with a left-padded attention mask: the native (plain causal) attention must not be used, because it would
    attend to the padding.  Logits at the unpadded positions match the same model on the PyTorch reference path."""
    from relora_b200.models import GPTNeoXForCausalLM, SimpleConfig
    from relora_b200.ops import dispatch

    torch.manual_seed(0)
    cfg = SimpleConfig(model_type="gpt_neox", vocab_size=512, hidden_size=256, num_hidden_layers=2, num_attention_heads=4,
                       intermediate_size=1024, rotary_pct=0.25, max_position_embeddings=128, layer_norm_eps=1e-5,
                       use_parallel_residual=True, hidden_act="gelu", rotary_emb_base=10000, tie_word_embeddings=False)
    model = GPTNeoXForCausalLM(cfg).to("cuda", BF).eval()
    B, T = 3, 48
    ids = torch.randint(0, 512, (B, T), device="cuda")
    mask = torch.ones(B, T, dtype=torch.long, device="cuda")
    mask[1, :18] = 0
    mask[2, :31] = 0
    with torch.no_grad():
        got = model(input_ids=ids, attention_mask=mask).logits.float()
        dispatch.force_reference(True)
        try:
            want = model(input_ids=ids, attention_mask=mask).logits.float()
        finally:
            dispatch.force_reference(False)
    for b in range(B):
        keep = mask[b].bool()
        g, w = got[b, keep], want[b, keep]
        err = float((g - w).norm() / w.norm())
        assert err < 2e-2, (b, err)
