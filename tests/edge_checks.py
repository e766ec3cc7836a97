"""Shared helpers of the element-wise kernel checks (``test_kernel_edges_gpu.py``, ``test_step_kernels_edges_gpu.py``).

Every check compares a kernel output with a float64 reference element by element against a per-element bound, records
the largest ``err/bound`` per kernel family, and prints it.  Outputs are written through views into canary-filled
buffers and inputs sit in NaN-padded buffers, so writes past an output and reads past an operand show up.
"""
import torch

BF = torch.bfloat16
F64 = torch.float64
U8 = 2.0 ** -8    # unit roundoff of bf16 (8 significant bits): |bf16(x) - x| <= 2^-8 |x|
U24 = 2.0 ** -24  # unit roundoff of fp32
TINY = 1e-300     # keeps the bound positive where the reference and all magnitudes are exactly zero
CANARY16 = 0x7FC1            # a quiet-NaN bf16 pattern no kernel produces by arithmetic
CANARY32 = 0x7FC00123        # the same for fp32 buffers

worst = {}  # kernel family -> largest err/bound seen in the running test module


def print_worst():
    for fam, v in sorted(worst.items()):
        print(f"[edges] largest err/bound  {fam:<22s} {v:.3g}")


def _padded(rows, cols, *, pad_rows=3, pad_cols=8, dtype=BF, fill=float("nan")):
    """A ``[rows, cols]`` view into a buffer of ``rows + pad_rows`` rows whose remainder holds ``fill``; the leading dimension
    is ``cols`` rounded up to 16 bytes plus ``pad_cols`` (the tensor maps need 16-byte row pitches)."""
    align = 16 // torch.tensor([], dtype=dtype).element_size()
    ld = (cols + align - 1) // align * align + pad_cols
    buf = torch.full((rows + pad_rows, ld), fill, device="cuda", dtype=dtype)
    return buf, buf[:rows, :cols]


def _operand(t, **kw):
    """Copy ``t`` into a NaN-padded buffer (padding columns and rows past the view): a kernel reading past the logical
    extent of an operand produces NaN."""
    _, v = _padded(t.shape[0], t.shape[1], **kw)
    v.copy_(t)
    return v


def _canary_out(rows, cols, dtype=BF, pad_rows=3, pad_cols=16):
    """(buffer, ``[rows, cols]`` view) with the whole buffer filled with a NaN bit pattern."""
    itype = torch.int16 if dtype == BF else torch.int32
    buf = torch.empty(rows + pad_rows, cols + pad_cols, device="cuda", dtype=dtype)
    buf.view(itype).fill_(CANARY16 if dtype == BF else CANARY32)
    return buf, buf[:rows, :cols]


def _assert_outside_untouched(buf, rows, cols, what):
    """Bytes of ``buf`` outside ``[:rows, :cols]`` still hold the canary pattern."""
    itype = torch.int16 if buf.dtype == BF else torch.int32
    pat = CANARY16 if buf.dtype == BF else CANARY32
    bits = buf.view(itype)
    bad_cols = (bits[:rows, cols:] != pat).nonzero()
    bad_rows = (bits[rows:] != pat).nonzero()
    assert bad_cols.numel() == 0, f"{what}: wrote past the last column at (row, col) {(bad_cols[0] + torch.tensor([0, cols], device='cuda')).tolist()}"
    assert bad_rows.numel() == 0, f"{what}: wrote past the last row at (row, col) {(bad_rows[0] + torch.tensor([rows, 0], device='cuda')).tolist()}"


def _excess(got, ref, bound):
    """(max err/bound, flat index of the worst element).  A non-finite output, reference or bound counts as infinitely
    wrong, so a reference that read NaN padding cannot pass silently."""
    got = got.to(F64)
    err = (got - ref).abs()
    ratio = err / (bound + TINY)
    finite = torch.isfinite(got) & torch.isfinite(ref) & torch.isfinite(bound + torch.zeros_like(err))
    ratio = torch.where(finite & ~torch.isnan(ratio), ratio, torch.full_like(ratio, float("inf")))
    i = int(ratio.reshape(-1).argmax())
    return float(ratio.reshape(-1)[i]), i


def _where_tile(shape, i):
    r, c = divmod(i, shape[-1]) if len(shape) == 2 else (i, 0)
    return f"(row {r}, col {c}) in 128x128 tile (tile_m {r // 128}, tile_n {c // 128})"


def check(family, case, got, ref, bound, where=_where_tile):
    """Assert ``|got - ref| <= bound`` element by element and record ``max err/bound``."""
    w, i = _excess(got, ref, bound)
    worst[family] = max(worst.get(family, 0.0), w)
    print(f"[edges] {family:<22s} {case:<44s} max err/bound {w:.3g}")
    if w > 1.0:
        g = float(got.reshape(-1)[i])
        r = float(ref.reshape(-1)[i])
        raise AssertionError(f"{family} {case}: worst element {where(tuple(got.shape), i)}: got {g!r}, ref {r!r}, "
                             f"bound {float(bound.reshape(-1)[i]):.3g} (err/bound {w:.3g})")
