"""Attention inputs built so that the right answer is exact or impossible to mistake, run on both tcgen05 kernels
(T <= 208: attention_tcgen05.cuh; 209 <= T <= 1025: attention_long_tcgen05.cuh) through both ways the library launches
them: stand-alone (the kernel takes |q|^2 and |k|^2 from q and k itself) and as the engine does, with the norms of the
QKV GEMM's epilogue. i.i.d. inputs cannot see a wrong norm index or a wrong route decision (softmax does not depend on
its shift) and hide a key too many or too few inside rounding; these can't. The tolerance is the per-element bound of
tests/attention_ref.py throughout.

The norms route passes fp32 norms with a row pitch of 2*heads + 8 whose padding columns are NaN: a kernel that reads
outside the |q|^2 and |k|^2 columns of its (image, head) turns its output into NaN.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import attention_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu

C_LOG2 = R.LOG2E / 8  # log2 units of one unit of q.k
# T -> (images, heads): both kernels, one and two query tiles, padding keys after an odd and an even number of real
# ones (37, 38: the mask treats even and odd columns in separate lanes), a 16-wide last key chunk (144), the short
# kernel's limit (208), the long kernel's first T (209), key tiles holding a single real key (257, 1025), two
# query-tile groups (577)
SHAPES = {37: (5, 3), 38: (4, 2), 144: (3, 2), 197: (4, 3), 208: (2, 4), 209: (3, 2), 257: (2, 3), 577: (2, 2),
          1025: (2, 3)}
ROUTES = ["standalone", "norms"]


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    torch.cuda.set_device(0)
    from twossp_b200 import ops as o
    return o


def _pack(q, k, v):
    """[n, heads, T, 64] q, k, v -> the fused bf16 qkv [n*T, 3*heads*64] on the GPU."""
    n, h, T, _ = q.shape
    return torch.stack([q, k, v]).permute(1, 3, 0, 2, 4).reshape(n * T, 3 * h * 64).bfloat16().cuda()


def _norms(qkv, n, T, heads):
    """|q|^2 and |k|^2 per head in fp64, stored as fp32 [n*T, 2*heads + 8] with NaN in the 8 padding columns."""
    q, k, _ = R.split_qkv(qkv, n, T, heads)
    out = torch.full((n * T, 2 * heads + 8), float("nan"), device="cuda")
    out[:, :heads] = q.pow(2).sum(-1).permute(0, 2, 1).reshape(n * T, heads).float()
    out[:, heads:2 * heads] = k.pow(2).sum(-1).permute(0, 2, 1).reshape(n * T, heads).float()
    return out


def _run(ops, qkv, n, T, heads, route):
    kw = {"norms": _norms(qkv, n, T, heads)} if route == "norms" else {}
    return R.run_and_check(ops, qkv, n, T, heads, **kw)[0]


def _randn(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_every_real_key_is_counted_once(ops, T, route):
    """Q = 0 gives every key the same weight whatever ex2 returns. Each V column of each (image, head) holds +1 for one
    half of a random permutation of the keys and -1 for the other (0 for the odd one out): ctx is exactly 0, while one
    key missing, or one of another head or image, makes it +-1/T or more."""
    n, h = SHAPES[T]
    q = torch.zeros(n, h, T, 64)
    k = _randn(n, h, T, 64, seed=T)
    rank = torch.rand(n, h, T, 64, generator=torch.Generator().manual_seed(T + 1)).argsort(2).argsort(2)
    half = T // 2
    v = torch.where(rank < half, 1.0, torch.where(rank < 2 * half, -1.0, 0.0))
    ctx = _run(ops, _pack(q, k, v), n, T, h, route)
    assert (ctx == 0).all(), f"{int((ctx != 0).sum())} nonzero outputs, largest {float(ctx.float().abs().max())}"


@pytest.mark.parametrize("logit", [-30.0, -150.0])  # the bound route; the exact route (the bound would underflow)
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_padding_keys_stay_out_of_the_softmax(ops, T, route, logit):
    """Every real key anti-aligned with q, every real logit `logit` log2 units; V has mean 1. A zero-filled padding key
    scores 0: let into the row sum or the row maximum, it collapses ctx to about 0 (or to NaN at -150)."""
    n, h = SHAPES[T]
    a = 8.0 if logit == -30.0 else 16.0
    b = -logit / C_LOG2 / a
    q, k = torch.zeros(n, h, T, 64), torch.zeros(n, h, T, 64)
    for i in range(n):
        for j in range(h):
            d = (i * h + j) % 64  # a different direction per (image, head)
            q[i, j, :, d] = a
            k[i, j, :, d] = -b
    v = 1.0 + 0.5 * _randn(n, h, T, 64, seed=T)
    _run(ops, _pack(q, k, v), n, T, h, route)


@pytest.mark.parametrize("logit", [32.0, 48.0])  # the bound route; the exact route
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_each_row_lands_in_its_place(ops, T, route, logit):
    """One-hot q and k: token t is of class perm[t % 64], a different permutation per (image, head), and a query
    scores `logit` log2 units against keys of its class and 0 against the rest, so each row is the mean V of its class.
    A row written to the wrong place, or a head or image read for another, is off by O(1)."""
    n, h = SHAPES[T]
    alpha = (logit / C_LOG2) ** 0.5
    g = torch.Generator().manual_seed(T + 7)
    q, k = torch.zeros(n, h, T, 64), torch.zeros(n, h, T, 64)
    t = torch.arange(T)
    for i in range(n):
        for j in range(h):
            cls = torch.randperm(64, generator=g)[t % 64]
            q[i, j, t, cls] = alpha
            k[i, j, t, cls] = alpha
    v = _randn(n, h, T, 64, seed=T)
    _run(ops, _pack(q, k, v), n, T, h, route)


def _hot_onehot(T, logit):
    """q = k = one-hot rows of class t % 64 scoring `logit` log2 units within a class."""
    alpha = (logit / C_LOG2) ** 0.5
    x = torch.zeros(T, 64)
    x[torch.arange(T), torch.arange(T) % 64] = alpha
    return x


@pytest.mark.parametrize("case", ["hot_head", "hot_image", "hot_row", "hot_key", "cold_row"])
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_hot_and_cold_shifts(ops, T, route, case):
    """Ordinary i.i.d. (image, head) units next to ones whose softmax shift is far from theirs. Each must come out finite
    and within the bound: a norm read for the wrong head, image, row or operand, or a wrong choice between the bound
    and the exact route, overflows to inf or underflows to 0 / 0 here.
      hot_head / hot_image: one head of every image / every head of one image scores up to +150 log2 units;
      hot_row: one query row of one unit (one warp of one tile) has a bound of 200 log2 units over logits near 60: only
               that warp (short kernel) or unit (long kernel) may take the exact route, and it must;
      hot_key: one key of one unit, aligned with every query of it, scores 75 to 300: a |q|^2 read in place of |k|^2
               would pick the bound route;
      cold_row: one query row whose logits all lie in [-300, -150]."""
    n, h = SHAPES[T]
    q, k, v = _randn(n, h, T, 64, seed=T), _randn(n, h, T, 64, seed=T + 1), _randn(n, h, T, 64, seed=T + 2)
    if case == "hot_head":
        q[:, h - 1] = k[:, h - 1] = _hot_onehot(T, 150.0)
    elif case == "hot_image":
        q[n - 1] = k[n - 1] = _hot_onehot(T, 150.0)
    elif case == "hot_row":
        i0 = 128 + 40 if T > 168 else T // 2
        kmax = float(k[n - 1, 0].bfloat16().float().norm(dim=-1).max())
        q[n - 1, 0, i0] = 0.0
        q[n - 1, 0, i0, 0] = 200.0 / (C_LOG2 * kmax)
    elif case == "hot_key":
        q[0, h - 1, :, 0] = q[0, h - 1, :, 0].abs() + 1.0
        k[0, h - 1, T - 1] = 0.0
        k[0, h - 1, T - 1, 0] = 150.0 / (2 * C_LOG2)
    else:  # cold_row
        k[0, 0, :, 0] = 2.0 + k[0, 0, :, 0].abs()
        kmin = float(k[0, 0, :, 0].bfloat16().float().min())
        q[0, 0, T // 3] = 0.0
        q[0, 0, T // 3, 0] = -150.0 / (C_LOG2 * kmin)
    _run(ops, _pack(q, k, v), n, T, h, route)


@pytest.mark.parametrize("T", list(SHAPES))
def test_norms_from_the_qkv_gemm(ops, T):
    """The engine's launch: qkv and its norms (ld = 2*heads) from the QKV GEMM with the rownorm epilogue, the norms
    taken of the fp32 values before their bf16 rounding. The last head's weights are 20x larger, so its logits reach
    about +150 log2 units (the exact route) next to heads on the bound route: a norm read at the wrong index overflows."""
    from twossp_b200 import _lib as L

    n, h = SHAPES[T]
    D, K = 64 * h, 128
    g = torch.Generator().manual_seed(T)
    x = (torch.randn(n * T, K, generator=g) * 0.5).bfloat16().cuda()
    w = torch.randn(3 * D, K, generator=g) * 0.05
    for part in (0, 1):  # q and k of the last head
        w[part * D + (h - 1) * 64:part * D + h * 64] *= 20.0
    w = w.bfloat16().cuda()
    bias = (torch.randn(3 * D, generator=g) * 0.1).cuda()
    qkv = torch.empty(n * T, 3 * D, device="cuda", dtype=torch.bfloat16)
    norms = ops.gemm_rownorm(x, w, qkv, bias, 2 * h)
    assert norms.shape == (n * T, 2 * h) and torch.isfinite(norms).all()
    R.run_and_check(ops, qkv, n, T, h, norms=norms)
    with pytest.raises(L.TsspError, match="ld_norms"):
        ops.attention(qkv, n, T, h, norms=norms[:, :2 * h - 1].contiguous())


SENTINEL = 0x5A5A  # a finite bf16 (about 1.5e16) no attention output of these inputs can take


@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_cls_only_writes_the_first_query_tile_alone(ops, T, route, scale):
    """cls_only (the engine's last block): rows >= 128 of every image keep what `out` held, bit for bit, and rows < 128
    are within the bound. In the short kernel they are also the full call's bits: each row's arithmetic is the same.
    The long kernel splits a row's sum over its two warpgroups by item parity, which depends on the group's tile count,
    so there the bound is all that holds."""
    n, h = SHAPES[T]
    qkv = R.iid_qkv(n, T, h, scale, seed=T * 5 + n, device="cuda")
    kw = {"norms": _norms(qkv, n, T, h)} if route == "norms" else {}
    first = (torch.arange(n * T, device="cuda") % T) < 128
    full = ops.attention(qkv, n, T, h, **kw)
    ref = R.reference(qkv, n, T, h)
    for _ in range(2):  # consecutive launches walk the units in opposite orders
        out = torch.empty(n * T, 64 * h, device="cuda", dtype=torch.bfloat16)
        out.view(torch.int16).fill_(SENTINEL)
        ops.attention(qkv, n, T, h, cls_only=True, out=out, **kw)
        assert (out.view(torch.int16)[~first] == SENTINEL).all(), "cls_only wrote rows >= 128"
        R.check(out, qkv, n, T, h, rows=first, ref=ref, what="cls_only")
        if T <= 208:
            assert torch.equal(out[first], full[first]), "cls_only rows differ from the full call's"
