"""Reference, error bound and CPU emulation of the tcgen05 attention kernels (csrc/attention_tcgen05.cuh, T <= 208, and
csrc/attention_long_tcgen05.cuh, 209 <= T <= 1025), shared by every attention test (TEST INFRASTRUCTURE).

What both kernels compute, per (image, head) and query row i, with c = fl32(log2(e) / 8):
  s_j  = q_i . k_j                       bf16 products summed in fp32 by the tensor core
  m    = the row's shift: the Cauchy-Schwarz bound |q_i| max_j |k_j| c (1 + 1e-4), or, on the exact route (some row of
         the warp / unit has a bound > 40 log2 units), fl32(max_j s_j * c) over the real keys
  e_j  = ex2.approx(fma(s_j, c, -m))    fp32, real keys only (padding keys are masked to 0)
  P_j  = bf16(e_j)                       round to nearest, written over S in TMEM
  l    = sum_j e_j                       fp32, of the UNROUNDED e_j
  O    = sum_j P_j v_j                   fp32 accumulation in the tensor core
  o    = bf16(O * fl32(1 / l))

Error bound. Let p_j = e_j / l, r = sum_j p_j v_j and A = sum_j p_j |v_j|. With u = 2^-8 (bf16 unit roundoff),
|P_j - e_j| <= u e_j, so |O / l - r| <= u A: one bf16 rounding of each P entry, not cancelled by the row sum because l
sums the unrounded values. The final bf16 rounding adds u |O / l| <= u |r| + u^2 A. Everything else is far smaller:
ex2.approx (2^-22 relative), the fp32 rounding of the exponent's argument (|arg| <= 2 * 40 * 1.0001 on the bound route,
2^-18.5 relative in e_j at most), the fp32 rounding of c (2^-24 relative on logit differences), fl32(1 / l) and the
product (2^-23 |r|), and the fp32 sums of S, l and O, whose rounding errors are unbiased and grow as sqrt(T) 2^-24. So

    |o - r| <= (2^-8 |r| + (2^-8 + 2^-18) A) (1 + 2^-7)

where the (1 + 2^-7) factor, u 2^-7 (|r| + A) = 2^-15 (|r| + A), holds the u^2 A = 2^-16 A of the output rounding and
the small terms above. The reference r and A are computed in fp64 from the same bf16 q, k, v.

Bias check. Errors that move a whole row's weights the same way (a key dropped or added, a wrong softmax scale, P
truncated instead of rounded) can stay inside the per-element bound at small input scales, but they pull the output
towards or away from zero together. slope = sum o r / sum r^2 over one call is 1 up to unbiased rounding noise; over at
least 1e5 outputs with inputs of scale <= 1, |slope - 1| <= 2e-4 (the emulation below stays under 1e-4, where a
padding key in the row sum, a 1 % scale error at scale 1 and a truncated P give 1e-3 and more).

`emulate` restates the kernels' arithmetic on the CPU, with switches for the faults a kernel change most often brings
in; test_host_logic.py::test_attention_checker_sensitivity pins that `check` sees each of them.
"""
from __future__ import annotations

import math

import torch

LOG2E = 1.4426950408889634
BOUND_LOG2 = 40.0          # ATC_BOUND_LOG2: the largest shift accepted without reading the row maximum
U = 2.0 ** -8              # bf16 unit roundoff
SLOPE_TOL = 2e-4
SLOPE_MIN_OUTPUTS = 100_000


def split_qkv(qkv: torch.Tensor, n: int, T: int, heads: int, dtype=torch.float64):
    """q, k, v [n, heads, T, 64] of the fused qkv [n*T, 3*heads*64]."""
    return qkv.to(dtype).view(n, T, 3, heads, 64).permute(2, 0, 3, 1, 4)


def _merge(x: torch.Tensor) -> torch.Tensor:
    """[n, heads, T, 64] -> [n*T, heads*64] (the ctx layout)."""
    n, h, T, d = x.shape
    return x.permute(0, 2, 1, 3).reshape(n * T, h * d)


def reference(qkv: torch.Tensor, n: int, T: int, heads: int):
    """(r, A) in fp64 on qkv's device, both [n*T, D]: r = softmax(Q K^T / 8) V and A = softmax(Q K^T / 8) |V|."""
    rs, As = [], []
    step = max(1, (1 << 27) // (heads * T * T))  # images per chunk: <= 1 GB of fp64 scores
    for i0 in range(0, n, step):
        i1 = min(n, i0 + step)
        q, k, v = split_qkv(qkv[i0 * T:i1 * T], i1 - i0, T, heads)
        p = torch.softmax((q @ k.transpose(-1, -2)) / 8.0, dim=-1)
        rs.append(_merge(p @ v))
        As.append(_merge(p @ v.abs()))
    return torch.cat(rs), torch.cat(As)


def error_bound(r: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    return (U * r.abs() + (U + 2.0 ** -18) * A) * (1 + 2.0 ** -7)


def slope(o: torch.Tensor, r: torch.Tensor) -> float:
    return float((o * r).sum() / (r * r).sum())


def check(ctx: torch.Tensor, qkv: torch.Tensor, n: int, T: int, heads: int, *, scale: float | None = None,
          rows: torch.Tensor | None = None, ref=None, what: str = "attention"):
    """Asserts ctx (bf16 [n*T, D]) is finite and within `error_bound` of the fp64 reference of qkv, and, when `scale`
    (the std of the i.i.d. inputs) is <= 1 and at least SLOPE_MIN_OUTPUTS outputs are checked, that the slope of ctx
    on the reference is within SLOPE_TOL of 1. `rows`: a bool mask over the n*T rows to check (default: all). `ref`:
    a precomputed (r, A). Returns (largest |o - r| / bound, slope or None)."""
    r, A = reference(qkv, n, T, heads) if ref is None else ref
    o = ctx.double()
    if rows is not None:
        o, r, A = o[rows], r[rows], A[rows]
    assert torch.isfinite(o).all(), f"{what}: {int((~torch.isfinite(o)).sum())} non-finite outputs"
    err = (o - r).abs()
    bound = error_bound(r, A)
    bad = err > bound
    if bad.any():
        i = int(bad.flatten().nonzero()[0])
        row, col = divmod(i, o.shape[1])
        raise AssertionError(f"{what}: {int(bad.sum())} of {o.numel()} outputs outside the bound; first at row {row} "
                             f"col {col}: got {float(o.flatten()[i]):.6g}, reference {float(r.flatten()[i]):.6g}, "
                             f"bound {float(bound.flatten()[i]):.3g}")
    ratio = float((err / bound.clamp_min(1e-300)).max())
    s = None
    if scale is not None and scale <= 1.0 and o.numel() >= SLOPE_MIN_OUTPUTS:
        s = slope(o, r)
        assert abs(s - 1.0) <= SLOPE_TOL, f"{what}: slope of the output on the reference is 1 {s - 1.0:+.2e}"
    return ratio, s


def emulate(qkv: torch.Tensor, n: int, T: int, heads: int, *, drop_last_key: bool = False, extra_padding_key: bool = False,
            scale_error: float = 1.0, truncate_p: bool = False) -> torch.Tensor:
    """The kernels' arithmetic (module docstring) on the CPU, bf16 ctx [n*T, D]. The route is decided per row (the
    kernels decide per warp or per unit; both routes give the same rounding model). Faults: `drop_last_key` masks key
    T-1 out; `extra_padding_key` counts one zero-filled key (score 0, v = 0) in the row sum; `scale_error` multiplies
    the softmax scale; `truncate_p` truncates P to bf16 instead of rounding it."""
    q, k, v = split_qkv(qkv.cpu(), n, T, heads, torch.float32)
    s = q @ k.transpose(-1, -2)
    c = torch.tensor(LOG2E / 8 * scale_error, dtype=torch.float32)
    kmax2 = k.pow(2).sum(-1).amax(-1, keepdim=True).unsqueeze(-1)
    bound = (q.pow(2).sum(-1, keepdim=True) * kmax2).sqrt() * c * 1.0001
    shift = torch.where(bound > BOUND_LOG2, s.amax(-1, keepdim=True) * c, bound)
    e = torch.exp2((s.double() * c.double() - shift.double()).float())  # fma: one rounding of the argument
    if drop_last_key:
        e[..., T - 1] = 0.0
    l = e.sum(-1, keepdim=True)
    if extra_padding_key:
        l = l + torch.exp2(-shift)
    if truncate_p:
        p = (e.view(torch.int32) & ~0xFFFF).view(torch.float32)
    else:
        p = e.bfloat16().float()
    o = (p @ v) * (1.0 / l)
    return _merge(o).bfloat16()


def iid_qkv(n: int, T: int, heads: int, scale: float, seed: int, device="cpu") -> torch.Tensor:
    """i.i.d. Gaussian qkv [n*T, 3*heads*64] of std `scale`, rounded to bf16."""
    g = torch.Generator(device=device).manual_seed(seed)
    return (torch.randn(n * T, 3 * heads * 64, device=device, generator=g) * scale).bfloat16()


def images_for(T: int, heads: int, outputs: int = SLOPE_MIN_OUTPUTS, units: int = 32) -> int:
    """Images for a bias check at (T, heads): at least `outputs` ctx values and `units` (image, head) pairs. At small
    input scales a row's weights lie within a few bf16 steps of each other, so the rounding error of P follows the
    logits instead of averaging out, with a sign set by where the unit's shift puts them on the bf16 grid; over a few
    units that alone moves the slope by 1e-4 (the emulation does the same), over 32 it averages out."""
    return max(math.ceil(outputs / (T * heads * 64)), math.ceil(units / heads))


def run_and_check(ops, qkv: torch.Tensor, n: int, T: int, heads: int, *, scale: float | None = None, **kwargs):
    """Two calls of ops.attention(qkv, n, T, heads, **kwargs): consecutive launches walk the units in opposite orders
    (chain_dir), so both results are checked against the reference and must be bit-identical. Returns the first ctx
    and `check`'s (ratio, slope)."""
    ctx = ops.attention(qkv, n, T, heads, **kwargs)
    again = ops.attention(qkv, n, T, heads, **kwargs)
    ref = reference(qkv, n, T, heads)
    stats = check(ctx, qkv, n, T, heads, scale=scale, ref=ref)
    check(again, qkv, n, T, heads, scale=scale, ref=ref, what="attention, second call")
    assert torch.equal(ctx, again), "two calls on the same input differ"
    return ctx, stats
