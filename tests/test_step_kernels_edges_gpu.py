"""Element-wise checks of the rest of the training step's kernels against float64: rotary, SwiGLU, dropout, embedding,
AdamW, the fp8 delayed-scaling state, the small utility kernels, and the Pythia block (layernorm, GELU, partial rotary).

The method is that of ``test_kernel_edges_gpu.py`` (helpers in ``edge_checks.py``): the reference is computed in float64
from the exact bf16 / fp32 values the kernel read, and every element is held to its own bound -- output rounding plus the
fp32 roundings of the kernel's own arithmetic, over float64 magnitudes.  Where the arithmetic allows it (rotary, the dropout
copies, embedding lookup, the fp32 -> bf16 cast, the seed stream) the result must be bit-exact.  The shapes come from
``configs/*.json``: hidden 416 / 640 / 768 / 2048, intermediate 688 / 1368 / 1376 / 2736 / 5504, head dim 64, vocabularies
32000 / 32100 (Llama) and 50304 (Pythia), M from 1 to 4097 and T up to 2049 at B = 2 and 3.  Each case prints its largest
``err/bound``; the negative controls at the end plant a plausible bug into a reference and check that the comparator
rejects it.
"""
import math

import pytest
import torch

import edge_checks
from edge_checks import BF, CANARY16, F64, U8, U24, _assert_outside_untouched, _canary_out, _excess, check

pytestmark = pytest.mark.gpu

F32 = torch.float32
ULP23 = 2.0 ** -23  # one fp32 ulp relative to the value (upper bound)


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    edge_checks.worst.clear()
    yield
    edge_checks.print_worst()


@pytest.fixture(scope="module")
def C():
    from relora_b200.ops import native

    return native.require()


def _randn(*shape, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(BF)


def _f32(v):
    """The fp32 value a kernel receives for a host double."""
    return float(torch.tensor(v, dtype=F32))


def _all_finite_bf16():
    """Every finite bf16 value (65280 of them), as a flat CUDA tensor."""
    bits = torch.arange(-32768, 32768, dtype=torch.int32, device="cuda").to(torch.int16)
    v = bits.view(BF)
    return v[torch.isfinite(v.float())].contiguous()


def _bf16_bits_equal(got, want, what):
    g, w = got.contiguous().view(torch.int16), want.contiguous().view(torch.int16)
    bad = (g != w).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} mismatches, first at {bad[0].tolist()}: got {float(got[tuple(bad[0])])!r}, " \
                             f"want {float(want[tuple(bad[0])])!r}"
    print(f"[edges] {what:<67s} mismatches 0")


def _canary_rows(rows, cols, ld, pad_rows=2):
    """(buffer, contiguous-rows view ``[rows, cols]`` with leading dimension ``ld``) filled with the bf16 canary."""
    buf = torch.empty(rows + pad_rows, ld, device="cuda", dtype=BF)
    buf.view(torch.int16).fill_(CANARY16)
    return buf, buf[:rows, :cols]


# ------------------------------------------------------------------------------------------------------------- rotary
def _rope_tables(n_pos, rot, seed):
    """bf16 tables ``[n_pos, rot]`` whose two halves are equal (the half-rotation layout), with values that change with
    every position so that a row read at the wrong position is visible."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ang = torch.rand(n_pos, rot // 2, device="cuda", generator=g, dtype=F64) * 2 * math.pi
    c, s = ang.cos().to(BF), ang.sin().to(BF)
    return torch.cat([c, c], 1).contiguous(), torch.cat([s, s], 1).contiguous()


def _rope_ref(x, pos, cos, sin, rot, sgn):
    """bf16(fp32(exact)) of the rotation of the first ``rot`` dims of every head of ``x [rows, heads, hd]`` at positions
    ``pos [rows]``: the products of two bf16 values are exact in fp32, so ``a c - b s`` is one fp32 rounding of the exact
    value whether or not the kernel contracts it into an FMA."""
    half = rot // 2
    xf = x.to(F64)
    c = cos.to(F64)[pos, :half][:, None, :]
    s = sgn * sin.to(F64)[pos, :half][:, None, :]
    a, b = xf[..., :half], xf[..., half:rot]
    out = x.clone()
    out[..., :half] = (a * c - b * s).to(F32).to(BF)
    out[..., half:rot] = (b * c + a * s).to(F32).to(BF)
    return out


def _rope_positions(B, T, pos0, shift_batch=None):
    pos = torch.arange(T, device="cuda").repeat(B) + pos0
    if shift_batch is not None:  # the bug of the negative control: one batch's positions off by one
        pos[shift_batch * T:(shift_batch + 1) * T] += 1
    return pos


_ROPE_CASES = [
    # B, T, nh, hd, rot, pos0, misalign: (65 / 1000 / 2049 tokens at B = 3; rot < hd; hd 24 / 40 have half % 8 != 0)
    (3, 65, 4, 64, 64, 0, False), (3, 1000, 2, 64, 64, 0, False), (3, 2049, 2, 64, 64, 0, False), (3, 2049, 2, 64, 64, 37, False),
    (3, 1000, 2, 64, 32, 5, False), (3, 65, 3, 64, 16, 0, False), (3, 2049, 2, 64, 64, 3, True), (3, 1000, 2, 24, 24, 0, False),
    (3, 65, 4, 40, 40, 11, False), (2, 2049, 2, 40, 24, 0, True),
]


@pytest.mark.parametrize("B,T,nh,hd,rot,pos0,misalign", _ROPE_CASES)
def test_rope_inplace_bitexact(C, B, T, nh, hd, rot, pos0, misalign):
    """Forward and inverse rotation of q and k inside the packed ``[B*T, 3*nh*hd]`` buffer (v and the padding columns and
    rows must not change), bit-exact.  A buffer that is not 16-byte aligned, or half = rot/2 not a multiple of 8, takes the
    scalar ``rope_kernel``.  Forward then inverse returns the input to within the rounding of the two passes."""
    torch.manual_seed(T + hd + rot + pos0)
    M, h3 = B * T, 3 * nh * hd
    ld = (h3 + 7) // 8 * 8 + 8
    ofs = 2 if misalign else 0  # 4 bytes: a bf16x2-aligned but not 16-byte aligned view
    buf = torch.empty((M + 2) * ld + 8, device="cuda", dtype=BF)
    buf.view(torch.int16).fill_(CANARY16)
    full = buf[ofs:ofs + (M + 2) * ld].view(M + 2, ld)
    x = full[:M, :h3]
    x.copy_(_randn(M, h3))
    x0 = x.clone()
    cos, sin = _rope_tables(T + pos0, rot, T + rot)
    pos = _rope_positions(B, T, pos0)
    case = f"B{B} T{T} nh{nh} hd{hd} rot{rot} pos0 {pos0}{' misaligned' if misalign else ''}"
    qk = lambda t: t.view(M, 3 * nh, hd)[:, : 2 * nh]  # noqa: E731
    C.rope_inplace(x, T, 2 * nh, hd, rot, cos, sin, False, pos0)
    want = _rope_ref(qk(x0), pos, cos, sin, rot, 1.0)
    _bf16_bits_equal(qk(x), want, f"rope forward {case}")
    assert torch.equal(x.view(M, 3 * nh, hd)[:, 2 * nh:], x0.view(M, 3 * nh, hd)[:, 2 * nh:]), "v changed"
    _assert_outside_untouched(full, M, h3, "rope buffer")
    assert bool((buf[:ofs].view(torch.int16) == CANARY16).all()), "rope wrote before the buffer"
    y = x.clone()
    C.rope_inplace(x, T, 2 * nh, hd, rot, cos, sin, True, pos0)
    _bf16_bits_equal(qk(x), _rope_ref(qk(y), pos, cos, sin, rot, -1.0), f"rope inverse {case}")
    # round trip: x' = R^T (R x + e1) + e2 with R^T R = (c^2 + s^2) I for the bf16 table values
    half = rot // 2
    c, s = cos.to(F64)[pos, :half][:, None, :], sin.to(F64)[pos, :half][:, None, :]
    x0f, yf = qk(x0).to(F64), qk(y).to(F64)
    e1 = (U8 + 2 * U24) * yf.abs()  # bf16(fp32(.)) of the forward
    n2 = (c * c + s * s - 1).abs()
    r = qk(x).to(F64)
    ref = x0f[..., :rot]
    bound = torch.cat([n2 * x0f[..., :half].abs() + c.abs() * e1[..., :half] + s.abs() * e1[..., half:rot],
                       n2 * x0f[..., half:rot].abs() + c.abs() * e1[..., half:rot] + s.abs() * e1[..., :half]], -1)
    bound = bound + (U8 + 2 * U24) * r[..., :rot].abs()
    check("rope-roundtrip", case, r[..., :rot], ref, bound)
    assert torch.equal(r[..., rot:], x0f[..., rot:])


@pytest.mark.parametrize("B,T,nh,hd,rot,pos0,contig", [
    (3, 65, 4, 64, 64, 0, False), (3, 2049, 2, 64, 64, 9, False), (3, 1000, 2, 64, 32, 0, True), (2, 2049, 3, 64, 16, 4, False),
    (3, 129, 2, 64, 64, 0, True),
])
def test_rope_pack_bwd_bitexact(C, B, T, nh, hd, rot, pos0, contig):
    """Gather of dq / dk / dv into the packed dQKV buffer with the inverse rotation of dq and dk, bit-exact: inputs with
    the strides attention backward returns (``[B, T, nh, hd]`` memory seen as ``[B, nh, T, hd]``) or contiguous; dims past
    ``rot`` and all of dv pass through unchanged."""
    torch.manual_seed(T * 3 + rot)
    M, hs = B * T, nh * hd
    if contig:
        dq, dk, dv = (_randn(B, nh, T, hd) for _ in range(3))
    else:
        dq, dk, dv = (_randn(B, T, nh, hd).transpose(1, 2) for _ in range(3))
    cos, sin = _rope_tables(T + pos0, rot, 2 * T + rot)
    buf, out = _canary_rows(M, 3 * hs, 3 * hs + 16)
    C.rope_pack_bwd(dq, dk, dv, out, rot, cos, sin, pos0)
    _assert_outside_untouched(buf, M, 3 * hs, "rope_pack_bwd out")
    pos = _rope_positions(B, T, pos0)
    tok = lambda t: t.transpose(1, 2).reshape(M, nh, hd)  # noqa: E731
    o5 = out.view(M, 3, nh, hd)
    case = f"B{B} T{T} nh{nh} hd{hd} rot{rot} pos0 {pos0} {'contiguous' if contig else 'attention strides'}"
    _bf16_bits_equal(o5[:, 0], _rope_ref(tok(dq), pos, cos, sin, rot, -1.0), f"rope_pack_bwd dq {case}")
    _bf16_bits_equal(o5[:, 1], _rope_ref(tok(dk), pos, cos, sin, rot, -1.0), f"rope_pack_bwd dk {case}")
    assert torch.equal(o5[:, 2], tok(dv)), "dv is a plain gather"


def _pack_args(B=2, T=64, nh=2, hd=64):
    """Inputs of ``rope_pack_bwd`` that live inside larger allocations, so that even a call the binding should have refused
    reads and writes only memory it owns."""
    big = torch.zeros(3, B, T + 8, nh, hd, device="cuda", dtype=BF)
    dq, dk, dv = (big[i, :, :T].transpose(1, 2) for i in range(3))
    out = torch.zeros(B * T + 8, 3 * nh * hd + 64, device="cuda", dtype=BF)[: B * T, : 3 * nh * hd]
    return dq, dk, dv, out


@pytest.mark.parametrize("bad", ["short table", "pos0 past the table", "width", "fp32 table", "strided table", "rot > hd"])
def test_rope_pack_bwd_rejects_bad_tables(C, bad):
    """The rotary tables of ``rope_pack_bwd`` are validated like those of ``rope_inplace``: bf16, contiguous, ``[n_pos,
    rotary_dim]`` with ``T + pos0 <= n_pos`` and ``rotary_dim <= head_dim``.  Each error is raised on the host, before
    any launch."""
    T, hd = 64, 64
    dq, dk, dv, out = _pack_args(T=T, hd=hd)
    cos_big, sin_big = _rope_tables(4 * T, 2 * hd, 1)
    view = lambda t, r, c: t.view(-1)[: r * c].view(r, c)  # noqa: E731  (a contiguous table inside the big one)
    rot, pos0 = hd, 0
    cos, sin = view(cos_big, T, hd), view(sin_big, T, hd)
    if bad == "short table":
        cos, sin = view(cos_big, T - 1, hd), view(sin_big, T - 1, hd)
    elif bad == "pos0 past the table":
        pos0 = 1
    elif bad == "width":
        cos, sin = view(cos_big, T, 2 * hd)[:, :hd + 8].contiguous(), view(sin_big, T, 2 * hd)[:, :hd + 8].contiguous()
    elif bad == "fp32 table":
        cos, sin = cos.float(), sin.float()
    elif bad == "strided table":
        cos, sin = cos_big[:T, :hd], sin_big[:T, :hd]
    elif bad == "rot > hd":
        rot = 2 * hd
        cos, sin = view(cos_big, T, 2 * hd), view(sin_big, T, 2 * hd)
    with pytest.raises(RuntimeError, match="rotary|cos|sin"):
        C.rope_pack_bwd(dq, dk, dv, out, rot, cos, sin, pos0)


# ------------------------------------------------------------------------------------------------------------- SwiGLU
def _silu64(g):
    return g * torch.sigmoid(g)


# __fdividef(x, y) returns 0 for 2^126 < |y| < 2^128, and 1 + __expf(-g) passes 2^126 for g <= -87.34 (it is inf below
# -88.72).  There the kernel's silu(g) is 0 while the true value, about g e^g, is a normal number down to about 1e-36.
# The bounds below admit exactly that: an absolute floor of |ref| on those elements and nowhere else.
_FDIV_ZERO_G = -87.3


def _swiglu_eps(g):
    """Relative error of the kernel's fp32 sigmoid(g) = 1 / (1 + __expf(-g)) (and of g / (1 + __expf(-g))): __expf is
    within 2 + 1.16 |x| ulp, the addition adds one rounding, scaled by e / (1 + e) of the exponential's own error, and
    __fdividef is within 2 ulp."""
    e = torch.exp(-g)
    w = torch.where(torch.isfinite(e), e / (1 + e), torch.ones_like(e))
    return w * (2 + 1.16 * g.abs()) * ULP23 + U24 + 2 * ULP23


def _swiglu_fwd_ref(g, u):
    gf, uf = g.to(F64), u.to(F64)
    ref = _silu64(gf) * uf
    bound = ref.abs() * (U8 + (1 + U8) * (_swiglu_eps(gf) + U24)) + 2.0 ** -133  # bf16 subnormal spacing / 2
    bound = torch.where(gf <= _FDIV_ZERO_G, torch.maximum(bound, ref.abs() * (1 + U8)), bound)
    return ref, bound


def _swiglu_bwd_ref(g, u, d, scale3=True):
    gf, uf, df = g.to(F64), u.to(F64), d.to(F64)
    sg = torch.sigmoid(gf)
    silu = gf * sg
    inner = sg + silu * (1 - sg)
    du = df * silu
    dg = df * uf * inner
    es = _swiglu_eps(gf)
    # du = d * (g * sg): sg's error, two multiplies, the bf16 store
    du_b = du.abs() * (U8 + (1 + U8) * (es + 2 * U24))
    # inner = sg + silu * (1 - sg): the absolute error of sg enters 1 - sg as well (cancellation for large g)
    err_sg = sg * es
    e_inner = err_sg * (1 + silu.abs()) + silu.abs() * (1 - sg) * (es + 2 * U24) + U24 * (1 - sg) * silu.abs() + U24 * inner.abs()
    dg_b = U8 * dg.abs() + (1 + U8) * ((df * uf).abs() * e_inner + 2 * U24 * dg.abs())
    floor = 2.0 ** -133
    tail = gf <= _FDIV_ZERO_G
    du_b = torch.where(tail, torch.maximum(du_b, du.abs() * (1 + U8)), du_b) + floor
    dg_b = torch.where(tail, torch.maximum(dg_b, dg.abs() * (1 + U8)), dg_b) + floor
    return du, du_b, dg, dg_b


def _swiglu_run_fwd(C, gu, M, Fd, p=0.0, seed=None, key=0):
    hbuf, h = _canary_rows(M, Fd, Fd + 24)
    dbuf, hd = _canary_rows(M, Fd, Fd + 40) if p > 0 else (None, None)
    C.swiglu_fwd(gu, h, hd, seed, key, p)
    _assert_outside_untouched(hbuf, M, Fd, "swiglu h")
    if hd is not None:
        _assert_outside_untouched(dbuf, M, Fd, "swiglu dropout copy")
    return h, hd


@pytest.mark.parametrize("M,Fd", [(1, 688), (189, 1368), (4097, 1376), (257, 2736), (4097, 5504), (7, 5504), (65, 688)])
def test_swiglu_elementwise(C, M, Fd):
    """h = silu(g) u and its backward at every intermediate size, ragged M, leading dimensions larger than the row
    (``gu``, ``h``, the dropout copy and ``dgu``); the grid-stride tail of the two-vectors-in-flight forward is hit at
    4097 x 5504.  The dropout copy is ``bf16(fp32(h) * fp32(1/(1-p)))`` bit for bit where kept and exactly 0 elsewhere."""
    from relora_b200.ops import reference as rf

    torch.manual_seed(M + Fd)
    gbuf = torch.full((M + 2, 2 * Fd + 16), float("nan"), device="cuda", dtype=BF)
    gu = gbuf[:M, : 2 * Fd]
    gu.copy_(_randn(M, 2 * Fd, scale=3.0))
    p, key, seed_v = 0.1, 7, 99991
    seed = torch.tensor([seed_v], dtype=torch.int32, device="cuda")
    h, hd = _swiglu_run_fwd(C, gu, M, Fd, p, seed, key)
    ref, bound = _swiglu_fwd_ref(gu[:, :Fd], gu[:, Fd:])
    check("swiglu-fwd", f"M{M} F{Fd}", h, ref, bound)
    keep = rf.dropout_keep_mask(rf.mix_seed(seed_v, key), M, Fd, p, device="cuda")
    ik = torch.tensor(1.0 / (1.0 - p), dtype=F32, device="cuda")
    want = torch.where(keep, (h.float() * ik).to(BF), torch.zeros_like(h))
    _bf16_bits_equal(hd, want, f"swiglu dropout copy M{M} F{Fd}")
    dh = torch.full((M + 1, Fd + 8), float("nan"), device="cuda", dtype=BF)[:M, :Fd]
    dh.copy_(_randn(M, Fd))
    dbuf, dgu = _canary_rows(M, 2 * Fd, 2 * Fd + 32)
    C.swiglu_bwd(dh, gu, dgu)
    _assert_outside_untouched(dbuf, M, 2 * Fd, "swiglu dgu")
    du, du_b, dg, dg_b = _swiglu_bwd_ref(gu[:, :Fd], gu[:, Fd:], dh)
    check("swiglu-bwd", f"dg M{M} F{Fd}", dgu[:, :Fd], dg, dg_b)
    check("swiglu-bwd", f"du M{M} F{Fd}", dgu[:, Fd:], du, du_b)


@pytest.mark.parametrize("u_kind", ["one", "random"])
def test_swiglu_every_bf16_gate(C, u_kind):
    """Every finite bf16 g (|g| up to 3.4e38, where __expf and __fdividef leave their accurate range), with u = 1 or u
    uniform in [-1, 1] (so that g u stays finite), forward and backward."""
    torch.manual_seed(5)
    g = _all_finite_bf16()
    Fd = 2736
    M = (g.numel() + Fd - 1) // Fd
    gflat = torch.zeros(M * Fd, device="cuda", dtype=BF)
    gflat[: g.numel()] = g
    u = torch.ones(M, Fd, device="cuda", dtype=BF) if u_kind == "one" else (torch.rand(M, Fd, device="cuda") * 2 - 1).to(BF)
    gu = torch.cat([gflat.view(M, Fd), u], 1).contiguous()
    h, _ = _swiglu_run_fwd(C, gu, M, Fd)
    ref, bound = _swiglu_fwd_ref(gu[:, :Fd], gu[:, Fd:])
    check("swiglu-fwd", f"every bf16 g, u {u_kind}", h, ref, bound)
    dh = torch.ones(M, Fd, device="cuda", dtype=BF) if u_kind == "one" else (torch.rand(M, Fd, device="cuda") * 2 - 1).to(BF)
    dgu = torch.empty_like(gu)
    C.swiglu_bwd(dh, gu, dgu)
    du, du_b, dg, dg_b = _swiglu_bwd_ref(gu[:, :Fd], gu[:, Fd:], dh)
    check("swiglu-bwd", f"dg every bf16 g, u {u_kind}", dgu[:, :Fd], dg, dg_b)
    check("swiglu-bwd", f"du every bf16 g, u {u_kind}", dgu[:, Fd:], du, du_b)


# ----------------------------------------------------------------------------------------------------- dropout kernels
def _combine_ref(base, parts, G, M, H, seed_v, keys, p):
    """float64 base + sum_g keep_g * part_g * fp32(1/(1-p)) and its bound: the bf16 store plus up to G + 1 fp32
    roundings (a product and an addition per group) over the magnitude of the terms."""
    from relora_b200.ops import reference as rf

    ik = _f32(1.0 / (1.0 - p))
    ref = torch.zeros(M, H, dtype=F64, device="cuda") if base is None else base.to(F64)
    mag = ref.abs()
    for g in range(G):
        keep = rf.dropout_keep_mask(rf.mix_seed(seed_v, keys[g]), M, H, p, device="cuda").to(F64)
        term = keep * parts[g].to(F64) * ik
        ref = ref + term
        mag = mag + term.abs()
    return ref, U8 * ref.abs() + (2 * G + 1) * U24 * mag


_DROP_CASES = [(G, M, H, base, form) for (G, M, H) in [(1, 4097, 416), (2, 189, 5504), (3, 257, 640), (3, 4097, 768), (2, 1, 2048)]
               for base in (True, False) for form in ("stacked", "strided")]


@pytest.mark.parametrize("G,M,H,base,form", _DROP_CASES)
def test_dropout_combine_elementwise(C, G, M, H, base, form):
    """``out = base + sum_g keep_g * part_g / (1-p)`` for G = 1, 2, 3 (the qkv backward uses 3), with and without a base,
    parts as ``[G, M, H]`` or as a ``[M, G*H]`` view with a leading dimension larger than G*H."""
    torch.manual_seed(G * 100 + M + H)
    p, seed_v, keys = 0.1, 424242, [3, 17, 99][:G]
    seed = torch.tensor([seed_v], dtype=torch.int32, device="cuda")
    b = _randn(M, H) if base else None
    if form == "stacked":
        parts = _randn(G, M, H)
        plist = [parts[g] for g in range(G)]
    else:
        pbuf = torch.full((M + 1, G * H + 24), float("nan"), device="cuda", dtype=BF)
        parts = pbuf[:M, : G * H]
        parts.copy_(_randn(M, G * H))
        plist = [parts[:, g * H:(g + 1) * H] for g in range(G)]
    obuf = torch.empty(M + 3, H, device="cuda", dtype=BF)
    obuf.view(torch.int16).fill_(CANARY16)
    out = obuf[:M]
    C.dropout_combine(b, parts, out, seed, keys, p)
    assert bool((obuf[M:].view(torch.int16) == CANARY16).all()), "dropout_combine wrote past M rows"
    ref, bound = _combine_ref(b, plist, G, M, H, seed_v, keys, p)
    check("dropout-combine", f"G{G} M{M} H{H} base{int(base)} {form}", out, ref, bound)


@pytest.mark.parametrize("G,M,H", [(1, 4097, 416), (2, 189, 5504), (3, 257, 640), (4, 7, 2048)])
def test_dropout_expand_bitexact(C, G, M, H):
    """``xd[:, g] = keep_g ? bf16(fp32(x) * fp32(1/(1-p))) : 0`` bit for bit, for every group."""
    from relora_b200.ops import reference as rf

    torch.manual_seed(G + M + H)
    p, seed_v, keys = 0.1, 777, [5, 6, 7, 8][:G]
    seed = torch.tensor([seed_v], dtype=torch.int32, device="cuda")
    x = _randn(M, H, scale=2.0)
    xbuf = torch.empty(M * G * H + 64, device="cuda", dtype=BF)
    xbuf.view(torch.int16).fill_(CANARY16)
    xd = xbuf[: M * G * H].view(M, G * H)
    C.dropout_expand(x, xd, seed, keys, p)
    assert bool((xbuf[M * G * H:].view(torch.int16) == CANARY16).all()), "dropout_expand wrote past its output"
    ik = torch.tensor(1.0 / (1.0 - p), dtype=F32, device="cuda")
    for g in range(G):
        keep = rf.dropout_keep_mask(rf.mix_seed(seed_v, keys[g]), M, H, p, device="cuda")
        want = torch.where(keep, (x.float() * ik).to(BF), torch.zeros_like(x))
        _bf16_bits_equal(xd.view(M, G, H)[:, g], want, f"dropout_expand G{G} M{M} H{H} group {g}")


# ---------------------------------------------------------------------------------------------------------- embedding
def _zipf_ids(M, V, pad, hot, n_hot, seed):
    """Token ids with a Zipf-like tail, one id repeated ``n_hot`` times, and the ids 0, V-1 and ``pad`` present."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = torch.rand(M, device="cuda", generator=g, dtype=F64)
    ids = (torch.exp(r * math.log(V)) - 1).long().clamp(0, V - 1)  # density ~ 1/id
    perm = torch.randperm(M, device="cuda", generator=g)
    ids[perm[:n_hot]] = hot
    ids[perm[n_hot:n_hot + 3]] = torch.tensor([0, V - 1, pad], device="cuda")
    return ids


def _embedding_bwd_ref(ids, dout, init, pad, drop=None):
    """float64 ``init + index_add(dout)`` with the padding row left alone, and the per-row bound
    (count + 1) * 2^-24 * (|init| + sum |dout|): the fp32 additions into one row, in any order."""
    V, H = init.shape
    keep = ids != pad
    if drop is not None:
        keep = keep.clone()
        keep[drop] = False
    idk, dk = ids[keep], dout.to(F64)[keep]
    ref = init.to(F64).index_add(0, idk, dk)
    mag = init.to(F64).abs().index_add(0, idk, dk.abs())
    cnt = torch.zeros(V, dtype=F64, device="cuda").index_add_(0, idk, torch.ones_like(idk, dtype=F64))
    return ref, (cnt[:, None] + 1) * U24 * mag


@pytest.mark.parametrize("V,H,M,pad", [(32000, 416, 6147, 0), (32100, 640, 4097, 31999), (50304, 2048, 2 * 2049, 1),
                                       (32000, 768, 4098, 0)])
def test_embedding_elementwise(C, V, H, M, pad):
    """Lookup bit-exact (ids 0, V-1 and the padding id present); the atomic and the sorted (deterministic) backward on a
    non-zero table with one id repeated 3000 times and a Zipf-like rest, the padding row untouched; the sorted form
    bit-identical across calls."""
    torch.manual_seed(V + H)
    ids = _zipf_ids(M, V, pad, hot=V // 3, n_hot=3000, seed=V + M)
    table = _randn(V, H)
    obuf = torch.empty(M + 2, H, device="cuda", dtype=BF)
    obuf.view(torch.int16).fill_(CANARY16)
    out = obuf[:M]
    C.embedding_fwd(ids, table, out)
    _bf16_bits_equal(out, table[ids], f"embedding_fwd V{V} H{H} M{M}")
    assert bool((obuf[M:].view(torch.int16) == CANARY16).all())
    dout = _randn(M, H)
    init = torch.randn(V, H, device="cuda")
    ref, bound = _embedding_bwd_ref(ids, dout, init, pad)
    d1 = init.clone()
    C.embedding_bwd(ids, dout, d1, pad)
    check("embedding-bwd", f"atomic V{V} H{H} M{M}", d1, ref, bound)
    assert torch.equal(d1[pad], init[pad]), "padding row changed"
    sid, perm = torch.sort(ids, stable=True)
    runs = []
    for _ in range(2):
        d2 = init.clone()
        C.embedding_bwd_sorted(sid, perm, dout, d2, pad)
        runs.append(d2)
    check("embedding-bwd", f"sorted V{V} H{H} M{M}", runs[0], ref, bound)
    assert torch.equal(runs[0], runs[1]), "sorted embedding backward is not bit-reproducible"
    assert torch.equal(runs[0][pad], init[pad]), "padding row changed"


# -------------------------------------------------------------------------------------------------------------- AdamW
def _adam_hyper(lr, b1, b2, eps, wd):
    return tuple(_f32(v) for v in (lr, b1, b2, eps, wd))


def _adamw_ref(p, g, m, v, *, lr, b1, b2, eps, wd, t, gs, gs_rel=0.0, bc_t=None):
    """float64 AdamW step from the stored p / g / m / v and the fp32 hyper-parameters the kernel reads, and per-element
    bounds for the stored p', m', v'.  ``gs_rel`` is a relative uncertainty of the gradient scale itself (0 when the
    kernel's own fp32 scale is used).  ``bc_t`` overrides the step count of the bias corrections (negative control)."""
    lr, b1, b2, eps, wd = _adam_hyper(lr, b1, b2, eps, wd)
    pf, gf, mf, vf = (t_.to(F64) for t_ in (p, g, m, v))
    tb = t if bc_t is None else bc_t
    gr = gf * gs
    mm = b1 * mf + (1 - b1) * gr
    vv = b2 * vf + (1 - b2) * gr * gr
    bc1, bc2 = 1 - b1 ** tb, 1 - b2 ** tb
    s = vv.sqrt()
    denom = s / math.sqrt(bc2) + eps
    upd = (lr / bc1) * mm / denom
    decay = 1 - lr * wd
    pn = pf * decay - upd
    # fp32 errors of the kernel: gr = g * gs (1 rounding), the moment updates (2 products and a sum; gr^2 one more)
    err_m = (3 * U24 + gs_rel) * (b1 * mf).abs() + (4 * U24 + gs_rel) * ((1 - b1) * gr).abs()
    err_v = 3 * U24 * (b2 * vf).abs() + (6 * U24 + 2 * gs_rel) * (1 - b2) * gr * gr
    # bias corrections: powf (within 4 ulp) amplified by b^t / (1 - b^t) in 1 - b^t, then a division or a rsqrt of a sqrt
    e_bc1 = 4 * ULP23 * (b1 ** t) / bc1 + 3 * U24
    e_bc2 = 0.5 * (4 * ULP23 * (b2 ** t) / bc2 + U24) + 3 * U24
    e_s = torch.where(s > 0, 0.5 * err_v / torch.where(s > 0, s, torch.ones_like(s)) + U24 * s, torch.zeros_like(s))
    e_den = (e_s + s * e_bc2) / math.sqrt(bc2) + 2 * U24 * denom
    rel_den = e_den / denom
    # p' = p * decay - step * (m / denom): decay (2 roundings), the product, the step size, the division, the difference
    e_upd = (lr / bc1) * err_m / denom + upd.abs() * (rel_den + e_bc1 + 3 * U24)
    e_p = 3 * U24 * (pf * decay).abs() + e_upd + U24 * pn.abs()
    bounds = {"p": U8 * pn.abs() + (1 + U8) * e_p}
    for name, ref, err, st in (("m", mm, err_m, m), ("v", vv, err_v, v)):
        bounds[name] = err + (U8 * ref.abs() * (1 + U8) + U8 * err if st.dtype == BF else U24 * ref.abs())
    return {"p": pn, "m": mm, "v": vv}, bounds


def _adam_inputs(n, gdt, sdt, seed):
    """p, g, m, v with four kinds of slices: generic; p = 0 (p' = -update, so a wrong bias correction, eps placement or
    gradient scale fails the 2^-8 relative bound); g = m = v = 0 (weight decay alone); gradients of the size of eps
    (where eps inside the square root would show)."""
    g_ = torch.Generator(device="cuda").manual_seed(seed)
    p = torch.randn(n, device="cuda", generator=g_).to(BF)
    g = torch.randn(n, device="cuda", generator=g_)
    m = 0.1 * torch.randn(n, device="cuda", generator=g_)
    v = 0.01 * torch.rand(n, device="cuda", generator=g_) + 1e-4
    q = n // 4
    p[q:2 * q] = 0
    g[2 * q:3 * q], m[2 * q:3 * q], v[2 * q:3 * q] = 0, 0, 0
    g[3 * q:] *= 1e-8
    m[3 * q:] *= 1e-7
    v[3 * q:] = v[3 * q:] * 1e-14
    return p, g.to(gdt), m.to(sdt), v.to(sdt)


_ADAM_DT = [(BF, BF), (F32, BF), (BF, F32), (F32, F32)]


@pytest.mark.parametrize("gdt,sdt", _ADAM_DT, ids=["g-bf16 s-bf16", "g-f32 s-bf16", "g-bf16 s-f32", "g-f32 s-f32"])
@pytest.mark.parametrize("n,step,dev_step", [(8 * 1001, 1, False), (8 * (148 * 8 * 256 + 1237), 7, True), (8 * 77, 1000, True)])
def test_adamw_flat_elementwise(C, gdt, sdt, n, step, dev_step):
    """One update of every grad / state dtype pair, n not a multiple of the grid stride, the step count from the host or
    from the device (the host value is then ignored), a device gradient scale times a host one."""
    hp = dict(lr=1e-2, b1=0.9, b2=0.95, eps=1e-8, wd=0.1)
    p, g, m, v = _adam_inputs(n, gdt, sdt, seed=n + step)
    gs_dev, gs_host = 0.37, 2.0
    gs = _f32(_f32(gs_host) * _f32(gs_dev))  # the kernel multiplies the two in fp32
    ref, bnd = _adamw_ref(p, g, m, v, t=step, gs=gs, **hp)
    step_dev = torch.tensor([float(step)], device="cuda") if dev_step else None
    C.adamw_flat(p, g, m, v, hp["lr"], hp["b1"], hp["b2"], hp["eps"], hp["wd"], 12345 if dev_step else step,
                 torch.tensor([gs_dev], device="cuda"), gs_host, None, step_dev)
    case = f"{str(gdt)[6:]}/{str(sdt)[6:]} n{n} t{step}"
    for k, got in (("p", p), ("m", m), ("v", v)):
        check(f"adamw-{k}", case, got, ref[k], bnd[k])


def test_adamw_trajectory_through_flat_adamw(C):
    """Six updates driven the way the fused stepper drives them -- fp32 gradients, bf16 moments, the clip coefficient as a
    device scale, ``FlatAdamW.step(grad_scale=..., skip=...)``: step 3 has a non-finite gradient norm (NaN scale) and step
    5 ``skip = 1``; both must leave p / m / v bit-identical and not advance the device step count.  Every other step is
    replayed in float64 from the state the previous step left, with the bias corrections of the number of updates
    actually applied; the clip coefficient is checked against ``clip_grad_norm_`` semantics in float64."""
    from relora_b200.ops.fused import NativeOptim
    from relora_b200.parallel.flat import FlatAdamW, FlatParamStore

    torch.manual_seed(11)
    shapes = [(416, 688), (1368,), (5, 7), (640, 416)]
    params = [torch.nn.Parameter(torch.randn(*s, device="cuda").to(BF)) for s in shapes]
    store = FlatParamStore([(f"p{i}", p) for i, p in enumerate(params)], grad_dtype=F32)
    hp = dict(lr=3e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.1)
    opt = FlatAdamW(store, lr=hp["lr"], betas=(hp["b1"], hp["b2"]), eps=hp["eps"], weight_decay=hp["wd"], state_dtype=BF,
                    native=NativeOptim())
    clip, applied = 1.0, 0
    for k in range(1, 7):
        store.grads.normal_()
        store.grads[store.used:] = 0  # alignment padding holds no gradient
        if k == 3:
            store.grads[5] = float("nan")
        g64 = store.grads.to(F64)
        total64 = float(g64.norm())
        # FusedLlamaStepper.update with one rank: norm -> clip coefficient -> NaN when the norm is not finite
        total = torch.linalg.vector_norm(store.grads, 2, dtype=F32)
        coef = torch.clamp(clip / (total + 1e-6), max=1.0)
        scale = torch.where(torch.isfinite(total), coef, torch.full_like(coef, float("nan")))
        skip = torch.tensor(1.0 if k == 5 else 0.0, device="cuda")
        before = (store.params.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone(), float(opt._step_t))
        opt.step(grad_scale=scale, skip=skip)
        if k in (3, 5):
            assert torch.equal(store.params, before[0]) and torch.equal(opt.exp_avg, before[1]) and torch.equal(opt.exp_avg_sq, before[2]), \
                f"step {k}: a skipped update changed the state"
            assert float(opt._step_t) == before[3] == applied, f"step {k}: the device step count moved"
            continue
        applied += 1
        assert float(opt._step_t) == applied
        coef64 = min(clip / (total64 + 1e-6), 1.0)
        gs = float(scale)
        # torch's fp32 norm: an n-term fp32 sum of squares (worst case n * 2^-24 relative), then sqrt, add, divide
        n = store.numel
        check("adamw-clip-coef", f"step {k}", scale.reshape(1), torch.tensor([coef64], dtype=F64, device="cuda"),
              torch.tensor([(0.5 * n * U24 + 4 * U24) * coef64], dtype=F64, device="cuda"))
        ref, bnd = _adamw_ref(before[0], store.grads, before[1], before[2], t=applied, gs=gs, **hp)
        for name, got in (("p", store.params), ("m", opt.exp_avg), ("v", opt.exp_avg_sq)):
            check(f"adamw-{name}", f"trajectory step {k} (update {applied})", got, ref[name], bnd[name])
    assert applied == 4 and opt.step_count == 6


# ------------------------------------------------------------------------------------------------------------ fp8 prep
def _fp8_prep_model(state, w_scale, margin, n_e4m3):
    """Python model of ``prep_kernel``: the recorded amax replaces the estimate only when it is finite and positive;
    nothing recorded (0), NaN or inf keep the previous estimate.  Returns the new state and float64 scales."""
    n = w_scale.numel()
    st = state.double().cpu().view(n, 2).clone()
    cur, old = st[:, 1], st[:, 0]
    prev = torch.where(torch.isfinite(cur) & (cur > 0), cur, old)
    new_state = torch.stack([prev, torch.zeros_like(prev)], 1).reshape(-1)
    fmax = torch.where(torch.arange(n) < n_e4m3, torch.tensor(448.0, dtype=F64), torch.tensor(57344.0, dtype=F64))
    sx = torch.clamp(prev, min=_f32(1e-12)) * _f32(margin) / fmax
    a = sx * w_scale.double().cpu()
    return new_state, {"inv_sx": 1 / sx, "alpha_main": a, "alpha_inv": 1 / a}


@pytest.mark.parametrize("margin,n_e4m3", [(1.0, -1), (2.0, 20), (1.25, 0), (3.7, 33)])
def test_fp8_prep_state_machine(C, margin, n_e4m3):
    """Four calls of ``fp8_prep`` over 37 sites (E4M3 sites below ``n_e4m3``, E5M2 above), with the amax recorded in
    between: sites that recorded a value, sites that recorded nothing (keep the estimate), a NaN and an inf (an overflowed
    activation: also keep the estimate, otherwise the next micro-step quantises everything to 0 with alpha = inf).
    ``inv_sx``, ``alpha_main`` and ``alpha_inv`` to within a few fp32 ulp; the state exactly."""
    n = 37
    ne = n if n_e4m3 < 0 else n_e4m3
    torch.manual_seed(n_e4m3 + 100)
    state = torch.zeros(2 * n, device="cuda")
    w_scale = (torch.rand(n, device="cuda") * 0.01 + 1e-4)
    outs = {k: torch.empty(n, device="cuda") for k in ("inv_sx", "alpha_main", "alpha_inv")}
    for call in range(4):
        rec = torch.rand(n, device="cuda") * 50
        rec[call::5] = 0.0  # nothing recorded
        if call >= 1:
            rec[3 + call] = float("inf")
            rec[10 + call] = float("nan")
        if call == 0:
            rec[7] = 0.0  # a site that never records: the estimate stays 0, the scale uses the 1e-12 floor
        state.view(n, 2)[:, 1] = rec
        want_state, want = _fp8_prep_model(state, w_scale, margin, ne)
        C.fp8_prep(state, w_scale, outs["inv_sx"], outs["alpha_main"], outs["alpha_inv"], margin, n_e4m3)
        got_state = state.double().cpu()
        bad = sorted({i // 2 for i in (got_state != want_state).nonzero().view(-1).tolist()})
        assert not bad, f"call {call}: sites {bad}: state {[got_state.view(n, 2)[i].tolist() for i in bad]}, " \
                        f"expected {[want_state.view(n, 2)[i].tolist() for i in bad]} (recorded {[float(rec[i]) for i in bad]})"
        for k, ulps in (("inv_sx", 4), ("alpha_main", 4), ("alpha_inv", 6)):
            ref = want[k].cuda()
            check("fp8-prep", f"{k} call {call} margin {margin} n_e4m3 {n_e4m3}", outs[k], ref, ulps * U24 * ref.abs())


# ---------------------------------------------------------------------------------------------- cast, seed, sum of squares
def _cast_inputs():
    """fp32 values at the edges of the bf16 rounding: +-0, fp32 subnormals, values that become bf16 subnormals, exact bf16
    midpoints (low half 0x8000) with odd and even upper halves and their +-1 ulp neighbours, the largest finite values
    (0x7F7F8000 rounds up to inf), +-inf, NaN, and random normals."""
    hi = torch.tensor([0x0000, 0x0001, 0x007F, 0x0080, 0x0081, 0x3F80, 0x3F81, 0x4049, 0x7F7E, 0x7F7F, 0x0100, 0x1234],
                      dtype=torch.int64)
    lo = torch.tensor([0x0000, 0x0001, 0x7FFF, 0x8000, 0x8001, 0xFFFF, 0x4000, 0xC000], dtype=torch.int64)
    bits = (hi[:, None] << 16 | lo[None, :]).reshape(-1)
    bits = torch.cat([bits, bits | (1 << 31), torch.tensor([0x7F800000, 0xFF800000, 0x7FC00000, 0x7F800001, 0xFFC00001])])
    x = bits.to(torch.int32).view(F32)
    rnd = torch.randn(4096, generator=torch.Generator().manual_seed(3))
    x = torch.cat([x, rnd, rnd * 1e-39, rnd * 3e38])
    pad = (-x.numel()) % 8
    return torch.cat([x, torch.zeros(pad)]).cuda()


@pytest.mark.parametrize("scale", [1.0, 0.37, 2.0, 1e-30])
def test_cast_f32_to_bf16_bitexact(C, scale):
    """``bf16_rn(fp32(x * scale))`` bit for bit (the products of two fp32 values are exact in float64); NaN stays NaN."""
    x = _cast_inputs()
    out = torch.empty(x.numel(), device="cuda", dtype=BF)
    C.cast_f32_to_bf16(x, out, scale)
    want = (x.double() * _f32(scale)).float().to(BF)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(out), nan), "NaN positions differ"
    _bf16_bits_equal(out[~nan], want[~nan], f"cast_f32_to_bf16 scale {scale}")


def test_seed_advance_sequence(C):
    """seed <- lowbias32(seed + 0x9E3779B9) over 300 launches, bit for bit, from a seed with the sign bit set."""
    from relora_b200.ops import reference as rf

    seed = torch.tensor([-123456789], dtype=torch.int32, device="cuda")
    got = []
    for _ in range(300):
        C.seed_advance(seed)
        got.append(seed.clone())
    got = (torch.cat(got).cpu().to(torch.int64) & 0xFFFFFFFF).tolist()
    x = -123456789 & 0xFFFFFFFF
    for i, gv in enumerate(got):
        x = int(rf._lowbias32(torch.tensor((x + 0x9E3779B9) & 0xFFFFFFFF, dtype=torch.int64)))
        assert gv == x, f"iteration {i}: {gv:#x} != {x:#x}"


def _sumsq_depth(n):
    """Longest chain of fp32 additions in ``sumsq``: each of grid * 256 threads (grid = min(ceil(n / 256), 1024)) sums a
    strided chunk serially, a 256-thread block tree (warp shuffles, then the warp sums: 10 levels), the final block adds
    ceil(grid / 256) partials per thread and another 10-level tree, and the result is added to ``out``."""
    grid = min((n + 255) // 256, 1024)
    return math.ceil(n / (grid * 256)) + 10 + math.ceil(grid / 256) + 10 + 1


@pytest.mark.parametrize("dtype", [BF, F32])
@pytest.mark.parametrize("n", [1, 255, 100_003, 12_582_917])
def test_sumsq_bound_and_determinism(C, dtype, n):
    torch.manual_seed(n)
    x = torch.randn(n, device="cuda").to(dtype)
    x[0] = 3.0
    out = torch.tensor([1.5], device="cuda")
    C.sumsq(x, out)
    again = torch.tensor([1.5], device="cuda")
    C.sumsq(x, again)
    assert torch.equal(out, again), "sumsq is not bit-reproducible"
    ref = 1.5 + (x.to(F64) ** 2).sum()
    bound = (_sumsq_depth(n) + 1) * 1.001 * U24 * ref  # the terms are >= 0: every partial sum is <= the total
    check("sumsq", f"{str(dtype)[6:]} n{n}", out, ref.reshape(1), bound.reshape(1))


# ------------------------------------------------------------------------------------------------------ Pythia: layernorm
def _ln_fwd_ref(x, w, b, eps, vpl):
    """float64 layernorm and the bound of the kernel's fp32 pipeline: the mean over H (each lane sums vpl * 8 values,
    then a 5-level warp tree), the two-pass variance around the fp32 mean (its error enters only to second order),
    rsqrtf (2 ulp), then (x - mean) * rstd * w + b and the bf16 store."""
    H = x.shape[1]
    xf, wf = x.to(F64), w.to(F64)
    bf = b.to(F64) if b is not None else torch.zeros_like(wf)
    mu = xf.mean(1, keepdim=True)
    d = xf - mu
    var = (d * d).mean(1, keepdim=True)
    rs = 1 / torch.sqrt(var + eps)
    y = d * rs * wf + bf
    depth = vpl * 8 + 6
    e_mu = depth * U24 * xf.abs().mean(1, keepdim=True)
    e_var = (depth + 4) * U24 * var + e_mu ** 2 + 2 * U24 * (var + eps)
    e_rs = rs * (0.5 * e_var / (var + eps) + 2 * ULP23 + U24)
    e_y = wf.abs() * (e_mu * rs + d.abs() * e_rs + 3 * U24 * (d * rs).abs()) + U24 * (y.abs() + bf.abs())
    return {"y": y, "mean": mu.squeeze(1), "rstd": rs.squeeze(1)}, {
        "y": U8 * y.abs() + (1 + U8) * e_y, "mean": (e_mu + U24 * mu.abs()).squeeze(1), "rstd": e_rs.squeeze(1)}


def _vpl(H):
    need = (H // 8 + 31) // 32
    return next(v for v in (1, 2, 3, 4, 8, 16) if need <= v)


def _ln_inputs(M, H, seed):
    """Rows of N(0, 1.5^2), one constant row, and rows with mean about 1000 and a spread of a few bf16 ulps (where a
    one-pass E[x^2] - E[x]^2 would cancel)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (torch.randn(M, H, device="cuda", generator=g) * 1.5).to(BF)
    x[1] = 1.3
    x[2:5] = (1000 + 8 * torch.randn(3, H, device="cuda", generator=g)).to(BF)
    w = (1 + 0.2 * torch.randn(H, device="cuda", generator=g)).to(BF)
    b = (0.1 * torch.randn(H, device="cuda", generator=g)).to(BF)
    return x, w, b


_LN_CASES = [(33, 200), (189, 416), (7, 640), (65, 768), (33, 1000), (189, 1024), (257, 1368), (4097, 2048), (33, 2560), (9, 4096)]


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("M,H", _LN_CASES)
def test_layernorm_fwd_elementwise(C, M, H, bias):
    """Every VPL instantiation (1 at H 200; 2 at 416; 3 at 640, 768; 4 at 1000, 1024; 8 at 1368, 2048; 16 at 2560, 4096),
    lanes with a ragged last vector, M not a multiple of the 8 rows of a block."""
    x, w, b = _ln_inputs(M, H, M * 7 + H)
    b = b if bias else None
    eps = 1e-5
    ybuf = torch.empty(M + 2, H, device="cuda", dtype=BF)
    ybuf.view(torch.int16).fill_(CANARY16)
    y = ybuf[:M]
    mean, rstd = torch.empty(M, device="cuda"), torch.empty(M, device="cuda")
    C.layernorm_fwd(x, w, b, y, mean, rstd, eps)
    assert bool((ybuf[M:].view(torch.int16) == CANARY16).all()), "layernorm y: wrote past M rows"
    ref, bnd = _ln_fwd_ref(x, w, b, eps, _vpl(H))
    case = f"M{M} H{H} vpl{_vpl(H)} bias{int(bias)}"
    check("layernorm-fwd", case, y, ref["y"], bnd["y"])
    check("layernorm-stats", f"mean {case}", mean, ref["mean"], bnd["mean"])
    check("layernorm-stats", f"rstd {case}", rstd, ref["rstd"], bnd["rstd"])


def _ln_bwd_ref(dy, x, w, mu, rs, dw0, db0, M, H, vpl, var_h=None):
    """float64 layernorm backward from the kernel's fp32 mean / rstd, and bounds.  dx: the two row means (H-term fp32 sums
    over vpl * 8 serial terms and a 5-level tree) and a handful of roundings per element.  dw / db: every column is a sum
    over rows -- serially within a warp (rows strided by grid * 8), then 8 warps into shared memory and grid blocks into
    global memory on top of the initial value."""
    dyf, xf, wf = dy.to(F64), x.to(F64), w.to(F64)
    mu, rs = mu.to(F64)[:, None], rs.to(F64)[:, None]
    xh = (xf - mu) * rs
    g = dyf * wf
    n = H if var_h is None else var_h
    sg = g.sum(1, keepdim=True) / H
    sgx = (g * xh).sum(1, keepdim=True) / n
    dx = rs * (g - sg - xh * sgx)
    depth = vpl * 8 + 6
    e_xh = 2 * U24 * xh.abs()
    e_sg = depth * U24 * g.abs().sum(1, keepdim=True) / H + U24 * sg.abs()
    e_sgx = (depth + 3) * U24 * (g * xh).abs().sum(1, keepdim=True) / H + U24 * sgx.abs()
    e_in = e_sg + e_xh * sgx.abs() + xh.abs() * e_sgx + 3 * U24 * (g.abs() + sg.abs() + (xh * sgx).abs())
    dx_b = U8 * dx.abs() + (1 + U8) * (rs * e_in + U24 * dx.abs())
    grid = min((M + 7) // 8, 2 * 148)
    rdepth = math.ceil(M / (grid * 8)) + 8 + grid + 1
    dyxh = dyf * xh
    out = {"dx": dx, "dw": dw0.to(F64) + dyxh.sum(0), "db": db0.to(F64) + dyf.sum(0)}
    bnd = {"dx": dx_b,
           "dw": (rdepth + 3) * U24 * (dw0.to(F64).abs() + dyxh.abs().sum(0)),
           "db": (rdepth + 1) * U24 * (db0.to(F64).abs() + dyf.abs().sum(0))}
    return out, bnd


@pytest.mark.parametrize("with_db", [True, False])
@pytest.mark.parametrize("M,H", [(33, 200), (189, 416), (2373, 640), (65, 768), (33, 1000), (4097, 1024), (257, 1368), (2373, 2048)])
def test_layernorm_bwd_elementwise(C, M, H, with_db):
    """dx, dw, db (or ``db=None``) at VPL 1 / 2 / 3 / 4 / 8, M = 2373 and 4097 > 2 * 148 * 8 so that every warp strides
    over several rows, on top of non-zero dw / db."""
    x, w, b = _ln_inputs(M, H, M + H)
    y = torch.empty_like(x)
    mean, rstd = torch.empty(M, device="cuda"), torch.empty(M, device="cuda")
    C.layernorm_fwd(x, w, b, y, mean, rstd, 1e-5)
    dy = _randn(M, H)
    dw0, db0 = torch.randn(H, device="cuda"), torch.randn(H, device="cuda")
    dxbuf = torch.empty(M + 2, H, device="cuda", dtype=BF)
    dxbuf.view(torch.int16).fill_(CANARY16)
    dx = dxbuf[:M]
    dw, db = dw0.clone(), (db0.clone() if with_db else None)
    C.layernorm_bwd(dy, x, w, mean, rstd, dx, dw, db)
    assert bool((dxbuf[M:].view(torch.int16) == CANARY16).all()), "layernorm dx: wrote past M rows"
    ref, bnd = _ln_bwd_ref(dy, x, w, mean, rstd, dw0, db0, M, H, _vpl(H))
    case = f"M{M} H{H} vpl{_vpl(H)} db{int(with_db)}"
    check("layernorm-dx", case, dx, ref["dx"], bnd["dx"])
    check("layernorm-dw/db", f"dw {case}", dw, ref["dw"], bnd["dw"])
    if with_db:
        check("layernorm-dw/db", f"db {case}", db, ref["db"], bnd["db"])


def test_layernorm_2560_takes_the_pytorch_path(C):
    """Pythia-2.8b's hidden size 2560 is above the backward kernel's 2048: the binding refuses it on the host, the model's
    layernorm takes nn.LayerNorm instead, and that path is checked against float64 too (forward and input gradient)."""
    from relora_b200.models import pythia
    from relora_b200.ops import fused

    M, H = 129, 2560
    x, w, b = _ln_inputs(M, H, 9)
    mean, rstd = torch.empty(M, device="cuda"), torch.empty(M, device="cuda")
    with pytest.raises(RuntimeError, match="<= 2048"):
        C.layernorm_bwd(x, x, w, mean, rstd, torch.empty_like(x), torch.zeros(H, device="cuda"), None)
    assert not fused.layernorm_supported(x)
    mod = torch.nn.LayerNorm(H, eps=1e-5).to("cuda", BF)
    with torch.no_grad():
        mod.weight.copy_(w)
        mod.bias.copy_(b)
    xr = x.clone().requires_grad_()
    y = pythia._layer_norm(mod, xr)
    # PyTorch reduces in its own order: bound its sums by H-term chains (vpl = H / 8 gives depth H + 6)
    ref, bnd = _ln_fwd_ref(x, w, b, 1e-5, H // 8)
    check("layernorm-fwd", f"M{M} H{H} pytorch path", y, ref["y"], bnd["y"])
    dy = _randn(M, H)
    y.backward(dy)
    xf = x.to(F64)
    mu, var = xf.mean(1), xf.var(1, unbiased=False)
    rs64 = 1 / torch.sqrt(var + 1e-5)
    r, bd = _ln_bwd_ref(dy, x, w, mu, rs64, torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda"), M, H, H // 8)
    # PyTorch's own fp32 mean / rstd (H-term sums) instead of exact ones: they move xh and the rstd factor of dx
    g = dy.to(F64) * w.to(F64)
    xh = (xf - mu[:, None]) * rs64[:, None]
    sgx = (g * xh).sum(1, keepdim=True) / H
    stats = (H + 10) * U24 * (r["dx"].abs() + rs64[:, None] * (3 * (xh * sgx).abs() + xf.abs().mean(1, keepdim=True) * rs64[:, None] * sgx.abs()))
    check("layernorm-dx", f"M{M} H{H} pytorch path", xr.grad, r["dx"], bd["dx"] + stats)


# --------------------------------------------------------------------------------------------------------- Pythia: GELU
def _gelu_ref(z, tanh, bwd, da=None, drop_3k=False):
    """float64 GELU (erf or tanh form) or da * its derivative, with the bound of the kernel's fp32 evaluation: the scaled
    argument (constants rounded to fp32), erff / tanhf (2 ulp each), whose error is multiplied by 0.5 |z| and where 1 +- f
    cancels, __expf in the erf derivative (2 + 1.16 |x| ulp), a few more roundings and the bf16 store."""
    zf = z.to(F64)
    c, k = math.sqrt(2 / math.pi), 0.044715
    if tanh:
        u = c * (zf + k * zf ** 3)
        f = torch.tanh(u)
        e_u = 7 * U24 * c * (zf.abs() + k * zf.abs() ** 3)
        e_f = 2 * ULP23 * f.abs() + (1 - f * f) * e_u
    else:
        a = zf / math.sqrt(2)
        f = torch.erf(a)
        e_f = 2 * ULP23 * f.abs() + 2 / math.sqrt(math.pi) * torch.exp(-a * a) * 2 * U24 * a.abs()
    half1 = 0.5 * (1 + f)
    if not bwd:
        ref = zf * half1
        e = 0.5 * zf.abs() * (e_f + U24 * (1 + f).abs()) + 2 * U24 * ref.abs()
        return ref, U8 * ref.abs() + (1 + U8) * e + 2.0 ** -133
    if tanh:
        q = 1 + 3 * (0 if drop_3k else k) * zf * zf
        t2 = 0.5 * zf * (1 - f * f) * c * q
        e_t2 = 0.5 * zf.abs() * c * q * (2 * f.abs() * e_f + U24 * f * f) + 10 * U24 * t2.abs()
    else:
        phi = torch.exp(-0.5 * zf * zf) / math.sqrt(2 * math.pi)
        t2 = zf * phi
        x = 0.5 * zf * zf  # __expf(-x) within 2 + 1.16 x ulp, and the argument's 2 roundings move it by 2 x 2^-24 relative
        e_t2 = t2.abs() * ((2 + 1.16 * x) * ULP23 + (2 * x + 5) * U24)
    dg = half1 + t2
    e_dg = 0.5 * (e_f + U24 * (1 + f).abs()) + e_t2 + U24 * (half1.abs() + t2.abs() + dg.abs())
    daf = da.to(F64)
    ref = daf * dg
    e = daf.abs() * e_dg + U24 * ref.abs()
    return ref, U8 * ref.abs() + (1 + U8) * e + 2.0 ** -133


@pytest.mark.parametrize("tanh", [False, True], ids=["erf", "tanh"])
def test_gelu_every_bf16(C, tanh):
    """Forward and backward of both GELU forms at every finite bf16 z (|z| up to 3.4e38), da random."""
    torch.manual_seed(int(tanh))
    z = _all_finite_bf16()
    a = torch.empty_like(z)
    C.gelu_fwd(z, a, tanh)
    ref, bnd = _gelu_ref(z, tanh, False)
    name = "tanh" if tanh else "erf"
    check(f"gelu-{name}-fwd", "every bf16 z", a, ref, bnd)
    da = _randn(z.numel())
    dz = torch.empty_like(z)
    C.gelu_bwd(da, z, dz, tanh)
    ref, bnd = _gelu_ref(z, tanh, True, da)
    check(f"gelu-{name}-bwd", "every bf16 z", dz, ref, bnd)


# ---------------------------------------------------------------------------------------------------- Pythia: neox rope
def _neox_ref(x, pos, cos, sin, rot, sgn):
    """float64 rotation of the first ``rot`` dims of q and k of ``x [rows, nh, 3, hd]`` with the fp32 tables, and the bound:
    two products of a bf16 and an fp32 value and their difference in fp32 (3 roundings of the magnitudes), the bf16 store."""
    half = rot // 2
    xf = x.to(F64)
    c = cos.to(F64)[pos, :half][:, None, None, :]
    s = sgn * sin.to(F64)[pos, :half][:, None, None, :]
    a, b = xf[:, :, :2, :half], xf[:, :, :2, half:rot]
    y1, y2 = a * c - b * s, b * c + a * s
    m1, m2 = (a * c).abs() + (b * s).abs(), (b * c).abs() + (a * s).abs()
    return torch.cat([y1, y2], -1), torch.cat([U8 * y1.abs() + (1 + U8) * 3 * U24 * m1, U8 * y2.abs() + (1 + U8) * 3 * U24 * m2], -1)


@pytest.mark.parametrize("hd,rot", [(64, 16), (80, 20), (128, 32), (256, 64)])
def test_neox_rope_elementwise(C, hd, rot):
    """Partial rotary of Pythia (rot = hd / 4: 16 / 20 / 32 / 64), B = 3, T = 2049, pos0 > 0, forward and inverse, the
    rest of q / k and all of v unchanged."""
    from relora_b200.ops import reference as rf

    torch.manual_seed(hd)
    B, T, nh, pos0 = 3, 2049, 2, 5
    M = B * T
    cos, sin = rf.rope_tables(rot, T + pos0, device="cuda")
    cos, sin = cos.contiguous(), sin.contiguous()
    x = _randn(M, nh * 3 * hd)
    x0 = x.clone()
    pos = _rope_positions(B, T, pos0)
    for inverse in (False, True):
        before = x.clone()
        C.neox_rope(x, T, nh, hd, rot, cos, sin, pos0, inverse)
        x4, b4 = x.view(M, nh, 3, hd), before.view(M, nh, 3, hd)
        ref, bnd = _neox_ref(b4, pos, cos, sin, rot, -1.0 if inverse else 1.0)
        check("neox-rope", f"hd{hd} rot{rot} {'inverse' if inverse else 'forward'}", x4[:, :, :2, :rot], ref, bnd)
        assert torch.equal(x4[:, :, :2, rot:], b4[:, :, :2, rot:]) and torch.equal(x4[:, :, 2], b4[:, :, 2])
    del x0


# ------------------------------------------------------------------------------------------------------ negative controls
def test_negative_control_rope_second_batch_position(C):
    """A rotary reference whose second batch is one position late differs from the kernel there (and only there)."""
    torch.manual_seed(0)
    B, T, nh, hd = 3, 65, 2, 64
    M = B * T
    x = _randn(M, 3 * nh * hd)
    x0 = x.clone()
    cos, sin = _rope_tables(T + 1, hd, 5)
    C.rope_inplace(x, T, 2 * nh, hd, hd, cos, sin, False, 0)
    qk = lambda t: t.view(M, 3 * nh, hd)[:, : 2 * nh]  # noqa: E731
    wrong = _rope_ref(qk(x0), _rope_positions(B, T, 0, shift_batch=1), cos, sin, hd, 1.0)
    diff = (qk(x).view(torch.int16) != wrong.view(torch.int16)).view(B, T, -1).any(-1)
    assert bool(diff[1].all()) and not bool(diff[0].any()) and not bool(diff[2].any())


def test_negative_control_adamw_bias_correction_and_eps():
    """The AdamW comparator rejects bias corrections of step t - 1 and eps inside the square root, on the p = 0 and the
    small-gradient slices."""
    hp = dict(lr=1e-2, b1=0.9, b2=0.95, eps=1e-8, wd=0.1)
    n, t = 8 * 4000, 7
    p, g, m, v = _adam_inputs(n, F32, F32, seed=1)
    ref, bnd = _adamw_ref(p, g, m, v, t=t, gs=0.5, **hp)
    got = ref["p"].to(BF)
    assert _excess(got, ref["p"], bnd["p"])[0] <= 1.0
    wrong, _ = _adamw_ref(p, g, m, v, t=t, gs=0.5, bc_t=t - 1, **hp)
    assert _excess(wrong["p"].to(BF), ref["p"], bnd["p"])[0] > 1.0
    lr, b1, b2, eps, wd = _adam_hyper(**hp)
    mm, vv = ref["m"], ref["v"]
    upd = (lr / (1 - b1 ** t)) * mm / torch.sqrt(vv / (1 - b2 ** t) + eps)
    wrong_p = p.to(F64) * (1 - lr * wd) - upd
    w, i = _excess(wrong_p.to(BF), ref["p"], bnd["p"])
    assert w > 1.0 and i >= 3 * (n // 4), (w, i)  # caught in the small-gradient slice


def test_negative_control_layernorm_variance_over_h_minus_1(C):
    """A layernorm reference that divides the variance by H - 1 is rejected by the rstd comparator at H = 416: rstd moves
    by 1/832 relative, far outside its fp32 bound (in the bf16 y the same change is below one rounding)."""
    M, H = 33, 416
    x, w, b = _ln_inputs(M, H, 1)
    y = torch.empty_like(x)
    mean, rstd = torch.empty(M, device="cuda"), torch.empty(M, device="cuda")
    C.layernorm_fwd(x, w, b, y, mean, rstd, 1e-5)
    ref, bnd = _ln_fwd_ref(x, w, b, 1e-5, _vpl(H))
    assert _excess(y, ref["y"], bnd["y"])[0] <= 1.0
    assert _excess(rstd, ref["rstd"], bnd["rstd"])[0] <= 1.0
    xf = x.to(F64)
    d = xf - xf.mean(1, keepdim=True)
    assert _excess(rstd, 1 / torch.sqrt((d * d).sum(1) / (H - 1) + 1e-5), bnd["rstd"])[0] > 1.0


def test_negative_control_embedding_dropped_occurrence(C):
    """An embedding-backward reference that misses one occurrence of a repeated id is rejected."""
    V, H, M, pad = 32000, 416, 6147, 0
    ids = _zipf_ids(M, V, pad, hot=V // 3, n_hot=3000, seed=2)
    dout = _randn(M, H)
    init = torch.randn(V, H, device="cuda")
    d = init.clone()
    C.embedding_bwd(ids, dout, d, pad)
    ref, bound = _embedding_bwd_ref(ids, dout, init, pad)
    assert _excess(d, ref, bound)[0] <= 1.0
    counts = torch.bincount(ids, minlength=V)
    rep = int(((counts >= 2) & (counts <= 50) & (torch.arange(V, device="cuda") != pad)).nonzero()[0])
    occ = int((ids == rep).nonzero()[0])
    wrong, _ = _embedding_bwd_ref(ids, dout, init, pad, drop=occ)
    assert _excess(d, wrong, bound)[0] > 1.0
    hot_occ = int((ids == V // 3).nonzero()[0])
    wrong, _ = _embedding_bwd_ref(ids, dout, init, pad, drop=hot_occ)
    assert _excess(d, wrong, bound)[0] > 1.0  # even for the id repeated 3000 times


def test_negative_control_dropout_combine_swapped_masks(C):
    """A ``dropout_combine`` reference with the masks of groups 0 and 1 swapped is rejected."""
    G, M, H, p, seed_v, keys = 3, 257, 640, 0.1, 31337, [3, 17, 99]
    parts = _randn(G, M, H)
    base = _randn(M, H)
    out = torch.empty(M, H, device="cuda", dtype=BF)
    C.dropout_combine(base, parts, out, torch.tensor([seed_v], dtype=torch.int32, device="cuda"), keys, p)
    ref, bound = _combine_ref(base, list(parts), G, M, H, seed_v, keys, p)
    assert _excess(out, ref, bound)[0] <= 1.0
    wrong, _ = _combine_ref(base, list(parts), G, M, H, seed_v, [17, 3, 99], p)
    assert _excess(out, wrong, bound)[0] > 1.0


def test_negative_control_gelu_tanh_derivative_without_cubic_term(C):
    """A gelu-tanh derivative reference without its 3 * 0.044715 z^2 term is rejected."""
    z = _all_finite_bf16()
    z = z[z.float().abs() < 8]
    z = z[: z.numel() // 8 * 8].contiguous()
    da = torch.ones_like(z)
    dz = torch.empty_like(z)
    C.gelu_bwd(da, z, dz, True)
    ref, bnd = _gelu_ref(z, True, True, da)
    assert _excess(dz, ref, bnd)[0] <= 1.0
    wrong, _ = _gelu_ref(z, True, True, da, drop_3k=True)
    assert _excess(dz, wrong, bnd)[0] > 1.0
