"""Kernel-level entry points of libtssp_b200.so on torch CUDA tensors (thin argument marshalling only).

These are what the parity tests drive one kernel at a time; the engine (engine.py) runs the same kernels
in sequence inside the library.
"""
from __future__ import annotations

import torch

from . import _lib as L


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise L.TsspError("libtssp_b200 kernels take CUDA tensors; there is no CPU path")


def check_gather_inputs(fc1_w, fc1_b, fc2_w, keep=None, where: str = "ffn_gather") -> None:
    """Explicit checks (not asserts: they must survive `python -O`, where half-precision data would otherwise be read as
    fp32). The gather kernel copies fp32 words; other parameter dtypes are refused with a message that says what to do."""
    _need_cuda(fc1_w, fc1_b, fc2_w, keep)
    for name, t in (("fc1.weight", fc1_w), ("fc1.bias", fc1_b), ("fc2.weight", fc2_w)):
        if t is not None and t.dtype != torch.float32:
            raise L.TsspError(f"{where}: {name} is {t.dtype}; the gather kernel moves float32 parameters "
                              "(the reference path prunes fp32 modules) -- call model.float() before pruning")
    if fc1_w.dim() != 2 or fc2_w.dim() != 2 or tuple(fc2_w.shape) != (int(fc1_w.shape[1]), int(fc1_w.shape[0])):
        raise ValueError(f"{where}: expected fc1.weight [F, D] and fc2.weight [D, F], got {tuple(fc1_w.shape)} and {tuple(fc2_w.shape)}")
    if int(fc1_w.shape[1]) % 4 != 0:
        raise L.TsspError(f"{where}: hidden size {int(fc1_w.shape[1])} is not a multiple of 4 (128-bit row copies)")
    if keep is not None and keep.dtype != torch.int64:
        raise ValueError(f"{where}: keep indices must be int64, got {keep.dtype}")


def _aligned(t):
    """Contiguous with a 16-byte aligned start (a view at an odd storage offset is copied)."""
    if t is None:
        return None
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def gemm(mode: int, a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, bias: torch.Tensor | None = None, *,
         m: int | None = None, partials: torch.Tensor | None = None, tokens_per_image: int = 0,
         reduce_add: bool = False) -> torch.Tensor:
    """out[M,N] (=|+=) epilogue(a[M,K] @ w[N,K]^T + bias). a, w bf16; out bf16 (modes 0-3, 5, 7, 8) or fp32 (mode 4)."""
    _need_cuda(a, w, out, bias, partials)
    if a.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise ValueError(f"gemm: operands must be bfloat16, got {a.dtype} and {w.dtype}")
    if a.stride(1) != 1 or w.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError("gemm: operands and output must be row-major (unit stride in the last dimension)")
    M = a.shape[0] if m is None else m
    N, K = w.shape
    if a.shape[1] != K:
        raise ValueError(f"gemm: a is [.., {a.shape[1]}] but w is [{N}, {K}]")
    lib = L.load()
    L.check(lib.tssp_op_gemm(mode, L.ptr(a), a.stride(0), L.ptr(w), w.stride(0), L.ptr(out), out.stride(0), M, N, K,
                             L.ptr(bias), L.ptr(partials), partials.stride(0) if partials is not None else 0,
                             tokens_per_image, 1 if reduce_add else 0, L.current_stream()))
    return out


def gemm_scaled(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, bias: torch.Tensor | None, col_scale: torch.Tensor, *,
                reduce_add: bool = False) -> torch.Tensor:
    """The LayerScale epilogue: out (fp32) (=|+=) col_scale * (a @ w^T + bias), column-wise."""
    _need_cuda(a, w, out, bias, col_scale)
    if out.dtype != torch.float32 or col_scale.dtype != torch.float32:
        raise ValueError("gemm_scaled: out and col_scale must be float32")
    M, K = a.shape
    N = w.shape[0]
    lib = L.load()
    L.check(lib.tssp_op_gemm_scaled(L.ptr(a), a.stride(0), L.ptr(w), w.stride(0), L.ptr(out), out.stride(0), M, N, K, L.ptr(bias),
                                    L.ptr(col_scale), 1 if reduce_add else 0, L.current_stream()))
    return out


def gemm_rownorm(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, bias: torch.Tensor | None, chunks: int) -> torch.Tensor:
    """The QKV epilogue: out (bf16) = a @ w^T + bias; returns [M, chunks] fp32 sums of squares of 64-column chunks."""
    _need_cuda(a, w, out, bias)
    M, K = a.shape
    N = w.shape[0]
    rownorm = torch.full((M, chunks), float("nan"), device=a.device, dtype=torch.float32)
    lib = L.load()
    L.check(lib.tssp_op_gemm_rownorm(L.ptr(a), a.stride(0), L.ptr(w), w.stride(0), L.ptr(out), out.stride(0), M, N, K, L.ptr(bias),
                                     L.ptr(rownorm), chunks, chunks, L.current_stream()))
    return rownorm


def score_finish(partials: torch.Tensor, n_img: int, T: int, F: int, scores: torch.Tensor | None = None) -> torch.Tensor:
    """partials [ceil(M/32)*2, ldp] -> per-image norms [n_img, F]; optionally scores[F] += sum over images."""
    _need_cuda(partials, scores)
    norms = torch.empty(n_img, F, device=partials.device, dtype=torch.float32)
    lib = L.load()
    L.check(lib.tssp_op_score_finish(L.ptr(partials), partials.stride(0), L.ptr(norms), norms.stride(0), n_img, T, F,
                                     L.ptr(scores), L.current_stream()))
    return norms


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, row_stride: int | None = None,
              rows: int | None = None) -> torch.Tensor:
    _need_cuda(x, gamma, beta)
    D = gamma.numel()
    rows = x.shape[0] if rows is None else rows
    stride = x.stride(0) if row_stride is None else row_stride
    out = torch.empty(rows, D, device=x.device, dtype=torch.bfloat16)
    lib = L.load()
    L.check(lib.tssp_op_layernorm(L.ptr(x), stride, L.ptr(gamma), L.ptr(beta), L.ptr(out), rows, D, float(eps), L.current_stream()))
    return out


def layernorm_f32(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, out: torch.Tensor | None = None) -> torch.Tensor:
    """The LayerNorm with fp32 output rows (the pre-norm of CLIP towers); `out` may be `x` itself (in place)."""
    _need_cuda(x, gamma, beta, out)
    if x.dtype != torch.float32 or x.stride(1) != 1:
        raise ValueError("layernorm_f32: x must be float32 with unit stride in the last dimension")
    D = gamma.numel()
    out = torch.empty(x.shape[0], D, device=x.device, dtype=torch.float32) if out is None else out
    if out.dtype != torch.float32 or out.stride(1) != 1:
        raise ValueError("layernorm_f32: out must be float32 with unit stride in the last dimension")
    lib = L.load()
    L.check(lib.tssp_op_layernorm_f32(L.ptr(x), x.stride(0), L.ptr(gamma), L.ptr(beta), L.ptr(out), out.stride(0), x.shape[0], D,
                                      float(eps), L.current_stream()))
    return out


def attention(qkv: torch.Tensor, n_img: int, T: int, heads: int, *, norms: torch.Tensor | None = None,
              cls_only: bool = False, out: torch.Tensor | None = None) -> torch.Tensor:
    """ctx [n*T, D] bf16 = softmax(Q K^T / 8) V per (image, head) of the fused qkv [n*T, 3*D].

    norms: fp32 [n*T, ld >= 2*heads] with |q|^2 of head h in column h and |k|^2 in column heads + h (the rownorm output
    of gemm_rownorm): the softmax shifts come from them, as in the engine's forward. cls_only: only rows [0, 128) of
    every image are written, as in the engine's last block. out: the ctx tensor to write into (rows the kernel does not
    write keep their contents)."""
    _need_cuda(qkv, norms, out)
    if qkv.dtype != torch.bfloat16 or not qkv.is_contiguous():
        raise ValueError("attention: qkv must be a contiguous bfloat16 tensor [n*T, 3*D]")
    D = qkv.shape[1] // 3
    if norms is not None and (norms.dtype != torch.float32 or norms.dim() != 2 or norms.stride(1) != 1
                              or norms.shape[0] != n_img * T):
        raise ValueError(f"attention: norms must be float32 [n*T, ld] with unit column stride, got {norms.dtype} "
                         f"{tuple(norms.shape)}")
    if out is None:
        out = torch.empty(n_img * T, D, device=qkv.device, dtype=torch.bfloat16)
    elif out.dtype != torch.bfloat16 or not out.is_contiguous() or tuple(out.shape) != (n_img * T, D):
        raise ValueError(f"attention: out must be a contiguous bfloat16 tensor [{n_img * T}, {D}]")
    lib = L.load()
    L.check(lib.tssp_op_attention(L.ptr(qkv), L.ptr(out), n_img, T, heads, D, L.ptr(norms),
                                  norms.stride(0) if norms is not None else 0, 1 if cls_only else 0, L.current_stream()))
    return out


def im2col(pixels: torch.Tensor, patch: int, prefix: int = 1, *, mean=None, std=None, rescale: float = 1 / 255) -> torch.Tensor:
    """[n * T, Kp] bf16 patch rows, `prefix` zero rows ahead of every image's patches (2 for DeiT, 1 + R with R register
    tokens); Kp = C*P*P rounded up to a multiple of 8, the columns past C*P*P zero (P = 14: 588 -> 592).
    uint8 pixels (C <= 4) need `mean` and `std` per channel and are normalised in the kernel, (float(u) * rescale -
    mean[c]) / std[c] in fp32: the bits of the fp32 form on api.normalize_pixels(pixels, mean, std, rescale)."""
    _need_cuda(pixels)
    u8 = pixels.dtype == torch.uint8
    if not (u8 or pixels.dtype == torch.float32) or not pixels.is_contiguous():
        raise ValueError("im2col: pixels must be a contiguous float32 or uint8 tensor [n, C, H, W]")
    if u8 and (mean is None or std is None):
        raise ValueError("im2col: uint8 pixels need the per-channel mean and std they are normalised with")
    n, c, h, w = pixels.shape
    T = (h // patch) * (w // patch) + prefix
    out = torch.empty(n * T, (c * patch * patch + 7) // 8 * 8, device=pixels.device, dtype=torch.bfloat16)
    norm = L.pixel_input(L.PIXELS_U8, [float(v) for v in mean], [float(v) for v in std], float(rescale)) if u8 else None
    L.check(L.load().tssp_op_im2col(L.ptr(pixels), L.ptr(out), n, c, h, w, patch, prefix, norm, L.current_stream()))
    return out


def cast_bf16(x: torch.Tensor, rows_pad: int | None = None, cols_pad: int | None = None) -> torch.Tensor:
    _need_cuda(x)
    if x.dtype != torch.float32 or x.stride(1) != 1:
        raise ValueError("cast_bf16: input must be float32 with unit stride in the last dimension")
    r, c = x.shape
    rp = r if rows_pad is None else rows_pad
    cp = c if cols_pad is None else cols_pad
    out = torch.empty(rp, cp, device=x.device, dtype=torch.bfloat16)
    lib = L.load()
    L.check(lib.tssp_op_cast_bf16(L.ptr(x), r, c, x.stride(0), L.ptr(out), rp, cp, cp, L.current_stream()))
    return out


def argmax_count(logits: torch.Tensor, labels: torch.Tensor | None, n_classes: int | None = None):
    _need_cuda(logits, labels)
    n = logits.shape[0]
    C_ = logits.shape[1] if n_classes is None else n_classes
    preds = torch.empty(n, device=logits.device, dtype=torch.int32)
    correct = torch.zeros(1, device=logits.device, dtype=torch.int64)
    lib = L.load()
    L.check(lib.tssp_op_argmax_count(L.ptr(logits), logits.stride(0), n, C_, L.ptr(labels), L.ptr(preds), L.ptr(correct), L.current_stream()))
    return preds, correct


def ffn_gather(fc1_w: torch.Tensor, fc1_b: torch.Tensor | None, fc2_w: torch.Tensor, keep: torch.Tensor):
    """(W1[keep], b1[keep], W2[:, keep]) as fresh fp32 tensors -- src/vit_pruning.py:297-299, bit-exact."""
    check_gather_inputs(fc1_w, fc1_b, fc2_w, keep)
    fc1_w = _aligned(fc1_w)
    fc2_w = _aligned(fc2_w)
    F, D = fc1_w.shape
    k = keep.numel()
    w1 = torch.empty(k, D, device=fc1_w.device, dtype=torch.float32)
    b1 = torch.empty(k, device=fc1_w.device, dtype=torch.float32) if fc1_b is not None else None
    w2 = torch.empty(D, k, device=fc1_w.device, dtype=torch.float32)
    lib = L.load()
    L.check(lib.tssp_ffn_gather(L.ptr(fc1_w), L.ptr(fc1_b.contiguous() if fc1_b is not None else None), L.ptr(fc2_w), F, D,
                                L.ptr(keep.contiguous()), k, L.ptr(w1), L.ptr(b1), L.ptr(w2), L.current_stream()))
    return w1, b1, w2


def ffn_gather_batch_plan(blocks):
    """Allocates the outputs and builds the host pointer tables of tssp_ffn_gather_batch for `blocks`.

    Returns (args, outs, hold): `lib.tssp_ffn_gather_batch(*args, stream)` runs the gather (any number of times),
    `outs` are the output tensors, `hold` keeps the contiguous inputs alive."""
    import ctypes as C

    blocks = list(blocks)
    n = len(blocks)
    hold, outs = [], []
    D = int(blocks[0][0].shape[1])
    P = C.c_void_p * n
    w1p, b1p, w2p, kp, o1p, obp, o2p = P(), P(), P(), P(), P(), P(), P()
    Fs, ks = (C.c_int32 * n)(), (C.c_int32 * n)()
    for i, (fc1_w, fc1_b, fc2_w, keep) in enumerate(blocks):
        check_gather_inputs(fc1_w, fc1_b, fc2_w, keep, "ffn_gather_batch")
        if int(fc1_w.shape[1]) != D:
            raise ValueError("ffn_gather_batch: every block needs fc1_w [F, D] and fc2_w [D, F] with the same D")
        fc1_w, fc2_w, keep = _aligned(fc1_w), _aligned(fc2_w), keep.contiguous()
        fc1_b = fc1_b.contiguous() if fc1_b is not None else None
        F, k = int(fc1_w.shape[0]), int(keep.numel())
        w1 = torch.empty(k, D, device=fc1_w.device, dtype=torch.float32)
        b1 = torch.empty(k, device=fc1_w.device, dtype=torch.float32) if fc1_b is not None else None
        w2 = torch.empty(D, k, device=fc1_w.device, dtype=torch.float32)
        hold.append((fc1_w, fc1_b, fc2_w, keep))
        outs.append((w1, b1, w2))
        w1p[i], b1p[i], w2p[i], kp[i] = fc1_w.data_ptr(), (fc1_b.data_ptr() if fc1_b is not None else None), fc2_w.data_ptr(), keep.data_ptr()
        o1p[i], obp[i], o2p[i] = w1.data_ptr(), (b1.data_ptr() if b1 is not None else None), w2.data_ptr()
        Fs[i], ks[i] = F, k
    return (n, w1p, b1p, w2p, Fs, D, kp, ks, o1p, obp, o2p), outs, hold


def ffn_gather_batch(blocks):
    """The gather of `ffn_gather` for several blocks in ONE kernel launch (tssp_ffn_gather_batch).

    blocks: sequence of (fc1_w [F,D], fc1_b [F] or None, fc2_w [D,F], keep int64 [k]) -- F and k may differ per block.
    Returns a list of (W1[keep], b1[keep] or None, W2[:, keep]) as fresh fp32 tensors, bit-exact
    (src/vit_pruning.py:297-299)."""
    blocks = list(blocks)
    if not blocks:
        return []
    args, outs, hold = ffn_gather_batch_plan(blocks)
    lib = L.load()
    L.check(lib.tssp_ffn_gather_batch(*args, L.current_stream()))
    del hold
    return outs
