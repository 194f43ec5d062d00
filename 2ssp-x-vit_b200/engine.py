"""Host-side wrapper of one libtssp_b200 engine handle bound to one torch ViT module.

All arithmetic happens inside the library (hand-written sm_100a kernels). This file only walks the module
for parameter addresses, slices batches to the engine's capacity and marshals pointers.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _lib as L
from .anatomy import Anatomy, describe

# the weight table (include/tssp.h: tssp_weight_index / tssp_block_weight_index); a key the anatomy lacks is NULL
_GLOBAL_ORDER = ["patch_w", "patch_b", "cls", "pos", "final_ln_w", "final_ln_b", "head0_w", "head_w", "head_b",
                 "dist", "head_dist_w", "head_dist_b", "reg", "norm_pre_w", "norm_pre_b"]
_BLOCK_ORDER = ["ln1_w", "ln1_b", "q_w", "q_b", "k_w", "k_b", "v_w", "v_b", "proj_w", "proj_b",
                "ln2_w", "ln2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "ls1", "ls2"]


def _cuda_device(device) -> torch.device:
    d = torch.device(device if device is not None else "cuda")
    if d.type != "cuda":
        raise L.TsspError(f"device {device!r}: the B200 backend runs on CUDA devices only (no CPU path)")
    if not torch.cuda.is_available():
        raise L.TsspError("CUDA is not available: the B200 backend has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device() if d.index is None else d.index)


class Engine:
    def __init__(self, vit_model, device="cuda", max_images: int = 128, cache_blocks: bool = False):
        self.lib = L.load()
        self.device = _cuda_device(device)
        self.anatomy: Anatomy = describe(vit_model)
        self.max_images = int(max_images)
        self.cache_blocks = bool(cache_blocks)
        a = self.anatomy
        cfg = L.TsspConfig()
        cfg.n_blocks, cfg.hidden, cfg.heads = a.n_blocks, a.hidden, a.heads
        cfg.image_size, cfg.patch_size, cfg.channels = a.image_size, a.patch_size, a.channels
        cfg.n_classes, cfg.head_hidden = a.n_classes, a.head_hidden
        cfg.max_images, cfg.score_point, cfg.cache_blocks = self.max_images, a.score_point, int(self.cache_blocks)
        cfg.ln_eps = a.ln_eps
        cfg.dist_token, cfg.register_tokens, cfg.pos_patches_only = int(a.dist_token), a.register_tokens, int(not a.pos_covers_prefix)
        cfg.layer_scale, cfg.pre_norm, cfg.ffn_act = int(a.layer_scale), int(a.pre_norm), L.FFN_ACTS[a.ffn_act]
        if a.n_blocks > L.TSSP_MAX_BLOCKS:
            raise L.TsspError(f"{a.n_blocks} blocks exceed TSSP_MAX_BLOCKS={L.TSSP_MAX_BLOCKS}")
        for i in range(a.n_blocks):
            cfg.ffn_dims[i] = a.ffn_dims[i]
            cfg.attn_present[i] = 1 if a.attn_present[i] else 0
        self._handle = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_create(C.byref(cfg), self.device.index, C.byref(self._handle)))
        self.ffn_dims = list(a.ffn_dims)
        self.pixel_norm = None                # (mean, std, rescale): see set_pixel_normalization
        self._pixel_format = (L.PIXELS_F32, None)  # what the library engine reads its `pixels` pointers as
        self.load_weights(a)
        self.anatomy.globals_.clear()
        self.anatomy.blocks.clear()  # do not keep parameter references alive

    # ------------------------------------------------------------------ weights
    def _dev32(self, t: Optional[torch.Tensor], keep: list) -> C.c_void_p:
        if t is None:
            return C.c_void_p(0)
        u = t.to(device=self.device, dtype=torch.float32).contiguous()
        keep.append(u)
        return C.c_void_p(u.data_ptr())

    def load_weights(self, a: Anatomy) -> None:
        keep: list = []
        entries = [self._dev32(a.globals_.get(k), keep) for k in _GLOBAL_ORDER]
        for blk in a.blocks:
            entries += [self._dev32(blk.get(k), keep) for k in _BLOCK_ORDER]
        table = (C.c_void_p * len(entries))(*entries)
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_load_weights(self._handle, table, len(entries), L.current_stream()))
            torch.cuda.current_stream().synchronize()  # staging copies in `keep` may now be released

    def update_ffn(self, block: int, fc1_w: torch.Tensor, fc1_b: Optional[torch.Tensor], fc2_w: torch.Tensor) -> None:
        keep: list = []
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_update_ffn(self._handle, block, int(fc1_w.shape[0]), self._dev32(fc1_w, keep),
                                             self._dev32(fc1_b, keep), self._dev32(fc2_w, keep), L.current_stream()))
            torch.cuda.current_stream().synchronize()
        self.ffn_dims[block] = int(fc1_w.shape[0])

    def set_attention(self, present: Sequence[bool]) -> None:
        arr = (C.c_int32 * len(present))(*[1 if p else 0 for p in present])
        L.check(self.lib.tssp_set_attention(self._handle, arr))

    def set_pixel_normalization(self, norm) -> None:
        """norm = (mean, std, rescale), one mean and std per channel: uint8 batches are then sent as bytes and normalised on
        the device, (float(u) * rescale - mean[c]) / std[c] in fp32. None: uint8 batches are converted with .float() on the
        host and not normalised. fp32 batches are fed as they are either way."""
        self.pixel_norm = None if norm is None else (tuple(float(m) for m in norm[0]), tuple(float(s) for s in norm[1]), float(norm[2]))

    def _use_format(self, u8: bool) -> None:
        want = (L.PIXELS_U8, self.pixel_norm) if u8 else (L.PIXELS_F32, None)
        if want != self._pixel_format:
            mean, std, rescale = self.pixel_norm if u8 else ((), (), 1.0)
            L.check(self.lib.tssp_set_pixel_input(self._handle, C.byref(L.pixel_input(want[0], mean, std, rescale))))
            self._pixel_format = want

    # ------------------------------------------------------------------ batches
    def _pixels(self, px: torch.Tensor) -> torch.Tensor:
        """The batch as the engine reads it; also sets the engine's pixel format for it (uint8 stays uint8 only with a
        normalisation set)."""
        u8 = px.dtype == torch.uint8 and self.pixel_norm is not None
        if px.dtype != torch.float32 and not u8:
            px = px.float()
        a = self.anatomy
        if px.dim() != 4 or px.shape[1] != a.channels or px.shape[2] != a.image_size or px.shape[3] != a.image_size:
            raise ValueError(f"pixel_values of shape {tuple(px.shape)} do not match the model "
                             f"([n,{a.channels},{a.image_size},{a.image_size}])")
        if px.is_cuda and px.device != self.device:
            px = px.to(self.device)
        self._use_format(u8)
        return px.contiguous()

    def _chunks(self, n: int):
        for s in range(0, n, self.max_images):
            yield s, min(n, s + self.max_images)

    def _skip(self, skip_attn: Optional[Sequence[int]]):
        if skip_attn is None:
            return None
        flags = [0] * self.anatomy.n_blocks
        for i in skip_attn:
            flags[int(i)] = 1
        return (C.c_int32 * len(flags))(*flags)

    # ------------------------------------------------------------------ stage 1
    def s1_reset(self) -> None:
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_s1_reset(self._handle, L.current_stream()))

    def s1_batch(self, pixel_values: torch.Tensor, img_norms: Optional[torch.Tensor] = None) -> int:
        px = self._pixels(pixel_values)
        with torch.cuda.device(self.device):
            for s, e in self._chunks(px.shape[0]):
                part = px[s:e]
                norms_ptr = L.ptr(img_norms[s:e]) if img_norms is not None else C.c_void_p(0)
                L.check(self.lib.tssp_s1_batch(self._handle, L.ptr(part), e - s, 0 if part.is_cuda else 1, norms_ptr, L.current_stream()))
        return int(px.shape[0])

    def s1_score_sums(self, on_device: bool = False) -> torch.Tensor:
        """Concatenated per-block sums over images of the token norms (not yet divided by the image count)."""
        total = sum(self.ffn_dims)
        with torch.cuda.device(self.device):
            if on_device:
                out = torch.empty(total, device=self.device, dtype=torch.float32)
                L.check(self.lib.tssp_s1_scores(self._handle, L.ptr(out), 0, L.current_stream()))
            else:
                out = torch.empty(total, dtype=torch.float32).pin_memory()
                L.check(self.lib.tssp_s1_scores(self._handle, L.ptr(out), 1, L.current_stream()))
        return out

    def split_blocks(self, flat: torch.Tensor) -> List[torch.Tensor]:
        return list(torch.split(flat, self.ffn_dims))

    # ------------------------------------------------------------------ forward / evaluation
    def logits(self, pixel_values: torch.Tensor, skip_attn: Optional[Sequence[int]] = None) -> torch.Tensor:
        px = self._pixels(pixel_values)
        out = torch.empty(px.shape[0], self.anatomy.n_classes, device=self.device, dtype=torch.float32)
        skip = self._skip(skip_attn)
        with torch.cuda.device(self.device):
            for s, e in self._chunks(px.shape[0]):
                part = px[s:e]
                L.check(self.lib.tssp_forward_logits(self._handle, L.ptr(part), e - s, 0 if part.is_cuda else 1, skip,
                                                     L.ptr(out[s:e]), 0, L.current_stream()))
        return out

    @staticmethod
    def _labels(labels: torch.Tensor, px: torch.Tensor) -> torch.Tensor:
        lb = labels.to(torch.int64).contiguous().view(-1)
        if lb.shape[0] != px.shape[0]:
            raise ValueError(f"{lb.shape[0]} labels for a batch of {px.shape[0]} images")
        return lb.to(px.device) if lb.is_cuda != px.is_cuda else lb

    def eval_batch(self, pixel_values: torch.Tensor, labels: torch.Tensor, correct_dev: torch.Tensor,
                   skip_attn: Optional[Sequence[int]] = None) -> int:
        px = self._pixels(pixel_values)
        lb = self._labels(labels, px)
        skip = self._skip(skip_attn)
        with torch.cuda.device(self.device):
            for s, e in self._chunks(px.shape[0]):
                L.check(self.lib.tssp_eval_batch(self._handle, L.ptr(px[s:e]), L.ptr(lb[s:e]), e - s, 0 if px.is_cuda else 1,
                                                 skip, L.ptr(correct_dev), L.current_stream()))
        return int(px.shape[0])

    # ------------------------------------------------------------------ stage 2
    def s2_reset(self) -> None:
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_s2_reset(self._handle, L.current_stream()))

    def s2_batch(self, pixel_values: torch.Tensor, labels: torch.Tensor, candidates: Optional[Sequence[int]] = None,
                 run_baseline: bool = True, with_scores: bool = False) -> int:
        """One batch of the attention-removal search. with_scores: the baseline pass also accumulates the Stage-1 score
        sums (s1_reset() before the first batch, s1_score_sums() after the last)."""
        px = self._pixels(pixel_values)
        lb = self._labels(labels, px)
        mask = self._skip(candidates)  # same [B] 0/1 layout; None = every block is a candidate
        with torch.cuda.device(self.device):
            for s, e in self._chunks(px.shape[0]):
                L.check(self.lib.tssp_s2_batch(self._handle, L.ptr(px[s:e]), L.ptr(lb[s:e]), e - s, 0 if px.is_cuda else 1,
                                               mask, (1 if run_baseline else 0) | (2 if with_scores else 0), L.current_stream()))
        return int(px.shape[0])

    def s2_counts(self) -> List[int]:
        n = self.anatomy.n_blocks + 1
        arr = (C.c_int64 * n)()
        with torch.cuda.device(self.device):
            L.check(self.lib.tssp_s2_counts(self._handle, arr, L.current_stream()))
        return [int(v) for v in arr]

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self.lib.tssp_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
