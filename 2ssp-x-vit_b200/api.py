"""Drop-in for the reference's ViT pruning API (src/vit_pruning.py `__all__` + the underscored helpers that
experiments/vit_pruning/auto_2ssp.py:44-56 imports), backed by libtssp_b200.so.

Same names, argument meaning, return types and error behaviour as the reference; the calibration forward
sweep, the top-1 evaluation, the Stage-2 candidate search and the Stage-1 gather run as sm_100a kernels.
What stays in Python/torch is what is not on the hot path and is parity-critical to keep identical:
`torch.argsort`/`torch.sort` for the neuron selection (unstable tie order, src/vit_pruning.py:286-287), the
integer planner, parameter accounting and JSON writing.

There is no CPU fallback: a model or device that is not CUDA raises TsspError.
"""
from __future__ import annotations

import json
import math
import os
import re
import weakref
from dataclasses import dataclass
from enum import Enum
from typing import Any, Dict, List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib as L
from . import distributed as D
from . import ops
from .anatomy import (attention_module, describe, ffn_act_signature, gather_mlp_pairs, get_blocks, get_encoder, has_attention,
                      install_bypass)
from .engine import Engine, _cuda_device

__all__ = [
    "prune_vit_mlp_width", "evaluate_top1", "prune_vit_attention_blocks", "plan_2ssp_allocation",
    "count_total_params", "count_block_params", "compute_actual_sparsity", "TwoSSPPlan",
    "B200Auto2SSPInterface", "PruningTypes", "PruningInterface",
    "save_ffn_importances", "save_ffn_masks", "save_attention_indices", "save_framework_export",
    "load_ffn_mask", "mask_to_importance", "apply_ffn_mask", "attention_removal_counts", "attention_removal_iterative",
    "measure_latency", "engine_for", "release_engine", "trim_pool",
    "set_pixel_normalization", "clear_pixel_normalization", "normalize_pixels",
]

# reference-named helpers (src/vit_pruning.py:28-75)
_get_encoder = get_encoder
_gather_mlp_pairs = gather_mlp_pairs


def _get_hidden_and_inter_sizes(vit_model):
    pairs = gather_mlp_pairs(vit_model)
    hidden = pairs[0][0].weight.size(1) if pairs else getattr(vit_model.config, "hidden_size", None)
    return hidden, [fc1.weight.size(0) for fc1, _ in pairs]


# ------------------------------------------------------------------------------------------ accounting
def count_total_params(model: nn.Module) -> int:
    """src/vit_pruning.py:81-83."""
    return sum(p.numel() for p in model.parameters())


def count_block_params(model: nn.Module) -> List[int]:
    """src/vit_pruning.py:85-98."""
    _, blocks = get_blocks(model)
    return [sum(p.numel() for p in b.parameters()) for b in blocks]


def compute_actual_sparsity(before_params: int, after_params: int) -> float:
    """src/vit_pruning.py:100-105."""
    return 0.0 if before_params <= 0 else (before_params - after_params) / before_params


def _count_attention_params_per_block(vit_model) -> List[int]:
    """src/vit_pruning.py:522-537 (a bypassed attention counts 0)."""
    kind, blocks = get_blocks(vit_model)
    out = []
    for b in blocks:
        m = attention_module(kind, b)
        out.append(0 if m is None else sum(p.numel() for p in m.parameters()))
    return out


def _count_ffn_params_per_block(vit_model) -> List[int]:
    """src/vit_pruning.py:539-558."""
    return [sum(p.numel() for p in fc1.parameters()) + sum(p.numel() for p in fc2.parameters())
            for fc1, fc2 in gather_mlp_pairs(vit_model)]


# ------------------------------------------------------------------------------------------ engine cache
_ENGINES: "weakref.WeakKeyDictionary[nn.Module, Dict[str, Any]]" = weakref.WeakKeyDictionary()
# model -> (mean, std, rescale) registered by set_pixel_normalization; applied to every engine engine_for returns, so an
# engine rebuilt after a pruning step or a parameter change keeps it
_PIXEL_NORMS: "weakref.WeakKeyDictionary[nn.Module, tuple]" = weakref.WeakKeyDictionary()


def _signature(model) -> tuple:
    """What a cached engine's weights were packed from: address, in-place version and shape of every parameter (a rebound
    Parameter changes the address, an in-place update the version, a view of the same storage the shape), and the MLP
    activation of every block (a parameter-free module: a swapped `mlp.act` changes nothing above)."""
    sig = []
    stack = [model]  # a plain walk of the module tree: model.parameters() spends 4x as long building names and a de-dup set
    while stack:
        mod = stack.pop()
        for p in mod._parameters.values():
            if p is not None:
                sig.append((p.data_ptr(), p._version, p.shape))
        stack.extend(m for m in mod._modules.values() if m is not None)
    sig.append(ffn_act_signature(model))
    return tuple(sig)


def engine_for(model, device="cuda", batch_hint: int = 128, need_cache: bool = False) -> Engine:
    """One engine per live module; rebuilt when the module's parameters changed or more capacity is needed."""
    dev = _cuda_device(device)
    sig = _signature(model)
    slot = _ENGINES.get(model)
    if slot is not None:
        eng: Engine = slot["engine"]
        if slot["sig"] == sig and eng.device == dev and (eng.cache_blocks or not need_cache):
            eng.set_pixel_normalization(_PIXEL_NORMS.get(model))
            return eng
        eng.close()
    cap = min(max(int(batch_hint), 16), 256)
    eng = Engine(model, device=dev, max_images=cap, cache_blocks=need_cache)
    eng.set_pixel_normalization(_PIXEL_NORMS.get(model))
    _ENGINES[model] = {"engine": eng, "sig": sig}
    return eng


def release_engine(model, trim: bool = False) -> None:
    """Drop the engine cached for `model`. Its device buffers are parked in the library's block pool (the next engine of
    the same shape takes them back without a cudaMalloc); trim=True returns the pool to the driver as well."""
    slot = _ENGINES.pop(model, None)
    if slot is not None:
        slot["engine"].close()
    if trim:
        trim_pool()


def trim_pool() -> None:
    """Give every device buffer parked by closed engines back to the CUDA driver. torch's caching allocator cannot see
    or reclaim that memory (up to TSSP_POOL_MB, default 16 GB): call this before fine-tuning the pruned model in the
    same process, or when torch reports out-of-memory."""
    L.check(L.load().tssp_trim_pool())


def set_pixel_normalization(model, mean: Sequence[float], std: Sequence[float], rescale: float = 1 / 255) -> None:
    """Let `model`'s batches arrive as uint8 [n, C, H, W] (what JPEG decoders produce) and normalise them on the device:
    x = (float(u) * rescale - mean[c]) / std[c] in fp32, the per-channel arithmetic of HF image processors and timm
    transforms. Every result is then bit for bit that of the fp32 batch `normalize_pixels(u, mean, std, rescale)`, and
    each image crosses PCIe as a quarter of the bytes. fp32 batches are unaffected. Pass the processor's numbers
    (e.g. image_mean / image_std of an HF processor). Raises ValueError, before any device work, unless there is one
    finite mean and one finite std > 0 per channel (at most four channels) and rescale is finite."""
    import ctypes as C
    channels = describe(model).channels
    f32 = lambda v: C.c_float(float(v)).value  # noqa: E731  (the values the device computes with)
    mean = [f32(m) for m in mean]
    std = [f32(s) for s in std]
    rescale = f32(rescale)
    if not 1 <= channels <= L.TSSP_MAX_PIXEL_CHANNELS:
        raise ValueError(f"uint8 pixel input supports 1 to {L.TSSP_MAX_PIXEL_CHANNELS} channels; the model has {channels}")
    if len(mean) != channels or len(std) != channels:
        raise ValueError(f"mean and std need one value per channel ({channels}), got {len(mean)} and {len(std)}")
    if not all(math.isfinite(v) for v in mean + std + [rescale]):
        raise ValueError(f"mean, std and rescale must be finite, got mean={mean} std={std} rescale={rescale}")
    if not all(s > 0 for s in std):
        raise ValueError(f"std must be > 0 in every channel, got {std}")
    _PIXEL_NORMS[model] = (tuple(mean), tuple(std), rescale)
    slot = _ENGINES.get(model)
    if slot is not None:
        slot["engine"].set_pixel_normalization(_PIXEL_NORMS[model])


def clear_pixel_normalization(model) -> None:
    """Undo set_pixel_normalization: uint8 batches of `model` are converted with .float() again, without normalisation."""
    _PIXEL_NORMS.pop(model, None)
    slot = _ENGINES.get(model)
    if slot is not None:
        slot["engine"].set_pixel_normalization(None)


def normalize_pixels(pixels: torch.Tensor, mean: Sequence[float], std: Sequence[float], rescale: float = 1 / 255) -> torch.Tensor:
    """The fp32 image a uint8 batch [n, C, H, W] stands for under set_pixel_normalization:
    (u.float() * rescale - mean[c]) / std[c], each operation in fp32, on the batch's device."""
    C = pixels.shape[1]
    dev = pixels.device
    r = torch.tensor(float(rescale), dtype=torch.float32, device=dev)
    m = torch.tensor([float(v) for v in mean], dtype=torch.float32, device=dev).view(1, C, 1, 1)
    s = torch.tensor([float(v) for v in std], dtype=torch.float32, device=dev).view(1, C, 1, 1)
    return (pixels.float() * r - m) / s


def _engine_in_step(model):
    """The cached engine of `model`, if its weights still are the module's (signature taken BEFORE a mutation)."""
    slot = _ENGINES.get(model)
    if slot is not None and slot["sig"] == _signature(model):
        return slot
    return None


def _peek(dataloader):
    """First batch (to size the engine) and an iterator that replays it followed by the rest."""
    it = iter(dataloader)
    try:
        first = next(it)
    except StopIteration:
        return None, iter(())

    def chain():
        yield first
        yield from it
    return first, chain()


# ------------------------------------------------------------------------------------------ stage 1: scores
@torch.no_grad()
def _compute_ffn_activation_importance(vit_model, dataloader, device: str = "cuda", batch_limit: Optional[int] = None,
                                       progress: bool = False, *, group=None, exact: bool = False) -> List[torch.Tensor]:
    """Per-neuron FFN importance = mean over calibration images of the L2 norm over tokens of the hooked
    activation (src/vit_pruning.py:111-201). Returns List[B] of CPU fp32 tensors [d_int].

    `group`: optional torch.distributed process group. Each rank passes the dataloader of ITS shard of the
    calibration set; the per-block sums are all-reduced (one NCCL collective) before the division by the
    global image count. `exact=True` (batches must carry "index" = global image ids) all-gathers per-image norms
    and adds them in global image order instead, so the bits do not depend on the number of GPUs.
    """
    if vit_model.training:
        vit_model.eval()
    first, batches = _peek(dataloader)
    if first is None or (batch_limit is not None and batch_limit <= 0):
        return [torch.zeros(fc1.out_features) for fc1, _ in gather_mlp_pairs(vit_model)]
    eng = engine_for(vit_model, device, batch_hint=int(first["pixel_values"].shape[0]))
    eng.s1_reset()
    seen = 0
    norm_parts, index_parts = [], []
    for i, batch in enumerate(batches):
        if batch_limit is not None and i >= batch_limit:
            break
        px = batch["pixel_values"]
        if exact:
            buf = torch.empty(px.shape[0], sum(eng.ffn_dims), device=eng.device, dtype=torch.float32)
            seen += eng.s1_batch(px, img_norms=buf)
            norm_parts.append(buf)
            index_parts.append(batch["index"].to(eng.device, torch.int64))
        else:
            seen += eng.s1_batch(px)
    if exact:
        norms = D.gather_image_norms(torch.cat(norm_parts), group)
        index = D.gather_image_norms(torch.cat(index_parts).view(-1, 1).to(torch.float64), group).view(-1).to(torch.int64)
        norms = norms[torch.argsort(index)]
        acc = torch.zeros(norms.shape[1], device=norms.device, dtype=torch.float32)
        for r in range(norms.shape[0]):
            acc += norms[r]  # fixed global image order, fp32 adds: same bits for any world size
        sums, seen = acc.cpu(), int(norms.shape[0])
    elif group is not None:
        sums, seen = D.reduce_score_sums(eng.s1_score_sums(on_device=True), seen, group)
        sums = sums.cpu()
    else:
        sums = eng.s1_score_sums(on_device=False)
    flat = sums / max(1, seen)
    return [t.clone() for t in eng.split_blocks(flat)]


# ------------------------------------------------------------------------------------------ stage 1: select + gather
@torch.no_grad()
def prune_vit_mlp_width(
    vit_model,
    sparsity: Optional[float] = None,
    strategy: str = "l1",
    min_remaining: int = 256,
    n_to_prune_per_block: Optional[List[int]] = None,
    dataloader=None,
    device: str = "cuda",
    batch_limit: Optional[int] = None,
    progress: bool = False,
    collect_masks: bool = False,
    precomputed_importance: Optional[List[torch.Tensor]] = None,
):
    """Width pruning of the MLP intermediate dimension of every block (src/vit_pruning.py:203-319).

    Mutates `vit_model` in place and returns it (or the dict with masks when collect_masks=True), exactly like
    the reference. The selection runs block by block as in the reference; the kept rows / bias entries / columns of ALL selected
    blocks are then gathered on the GPU by one tssp_ffn_gather_batch launch (bit-exact).
    """
    mlp_pairs = gather_mlp_pairs(vit_model)
    if n_to_prune_per_block is not None:
        if len(n_to_prune_per_block) != len(mlp_pairs):
            raise ValueError("n_to_prune_per_block length must match number of blocks")
    else:
        if sparsity is None:
            raise ValueError("Provide either sparsity or n_to_prune_per_block")
        if not (0.0 <= sparsity < 1.0):
            raise AssertionError("sparsity must be in [0,1)")

    importance_blocks: Optional[List[torch.Tensor]] = None
    if precomputed_importance is not None:
        if len(precomputed_importance) != len(mlp_pairs):
            raise ValueError("precomputed_importance length must match number of blocks")
        importance_blocks = precomputed_importance
    elif strategy == "act_l2" and dataloader is not None:
        print("[S1-LOG] Using activation-based importance (avg L2 over tokens, averaged across calibration samples)")
        importance_blocks = _compute_ffn_activation_importance(vit_model, dataloader, device=device, batch_limit=batch_limit, progress=progress)

    pruned_indices_all: List[List[int]] = []
    prune_masks_all: List[List[int]] = []
    # A cached engine is patched in place only if it matched the module BEFORE this call mutates it; an engine that was
    # already stale (parameters changed since it was built, e.g. optimizer steps) is dropped and rebuilt on next use.
    slot = _engine_in_step(vit_model)
    stale = slot is None and vit_model in _ENGINES
    for inter_dense, out_dense in mlp_pairs:   # refuse what the gather kernel cannot move before anything is mutated
        if inter_dense.weight.is_cuda:
            ops.check_gather_inputs(inter_dense.weight, inter_dense.bias, out_dense.weight, where="prune_vit_mlp_width")
    touched = []
    pending = []  # (block, fc1, fc2, keep_idx) of the blocks selected so far

    def gather_pending():
        """ONE batched gather launch for every selected block, then the rebinding of src/vit_pruning.py:304-311."""
        if not pending:
            return
        with torch.cuda.device(pending[0][1].weight.device):
            outs = ops.ffn_gather_batch([(fc1.weight.detach(), None if fc1.bias is None else fc1.bias.detach(),
                                          fc2.weight.detach(), keep) for _, fc1, fc2, keep in pending])
        for (b, fc1, fc2, _), (new_W_int, new_B_int, new_W_out) in zip(pending, outs):
            hidden = int(fc1.weight.size(1))
            fc1.weight = nn.Parameter(new_W_int)
            if new_B_int is not None:
                fc1.bias = nn.Parameter(new_B_int)
            fc1.out_features = int(new_W_int.size(0))
            fc1.in_features = hidden
            fc2.weight = nn.Parameter(new_W_out)
            fc2.in_features = int(new_W_int.size(0))
            touched.append(b)
        pending.clear()

    try:
        for block_idx, (inter_dense, out_dense) in enumerate(mlp_pairs):
            W_int, B_int, W_out = inter_dense.weight, inter_dense.bias, out_dense.weight
            n_channels = W_int.size(0)
            if not W_int.is_cuda:
                raise L.TsspError("prune_vit_mlp_width: model parameters must live on a CUDA device (no CPU path)")
            if importance_blocks is not None:
                importance = importance_blocks[block_idx].to(W_int.device)
                if importance.numel() != n_channels:
                    raise RuntimeError("precomputed/act_l2 importance size mismatch with intermediate width")
            elif strategy == "l1":
                importance = W_int.abs().sum(dim=1)
            elif strategy == "act_l2":
                raise RuntimeError("act_l2 importance requested but no dataloader/importance available")
            else:
                raise ValueError(f"Unknown strategy {strategy}")

            n_prune = int(n_to_prune_per_block[block_idx]) if n_to_prune_per_block is not None else int(n_channels * sparsity)
            if n_channels - n_prune < min_remaining:
                n_prune = max(0, n_channels - min_remaining)
            print(f"[S1-LOG] block={block_idx}, inter={n_channels}, n_prune={n_prune}, strategy={strategy}")
            if n_prune <= 0:
                continue

            # same torch calls, on the same device, as the reference: the tie order of the unstable sort is theirs
            keep_idx = torch.argsort(importance, descending=True)[: n_channels - n_prune]
            keep_idx, _ = torch.sort(keep_idx)

            if collect_masks:
                prune_mask = torch.ones(n_channels, dtype=torch.int16, device=keep_idx.device)
                prune_mask[keep_idx] = 0  # 1 = pruned, 0 = kept
                prune_masks_all.append(prune_mask.cpu().tolist())
                pruned_indices_all.append(torch.nonzero(prune_mask == 1, as_tuple=False).view(-1).tolist())

            pending.append((block_idx, inter_dense, out_dense, keep_idx))
    except BaseException:
        # the reference mutates block by block, so the blocks selected before a failing one stay pruned
        gather_pending()
        raise
    gather_pending()

    if slot is not None and touched:
        # keep the cached engine in step with the mutated module instead of rebuilding it
        eng: Engine = slot["engine"]
        for b in touched:
            fc1, fc2 = mlp_pairs[b]
            eng.update_ffn(b, fc1.weight.detach(), None if fc1.bias is None else fc1.bias.detach(), fc2.weight.detach())
        slot["sig"] = _signature(vit_model)
    elif stale:
        release_engine(vit_model)

    if collect_masks:
        return {"model": vit_model, "ffn_pruned_indices": pruned_indices_all, "ffn_prune_masks": prune_masks_all}
    return vit_model


# ------------------------------------------------------------------------------------------ evaluation
@torch.no_grad()
def _top1_counts(model, dataloader, device="cuda", max_batches=None, skip_attn: Optional[Sequence[int]] = None):
    model.eval()
    first, batches = _peek(dataloader)
    if first is None or (max_batches is not None and max_batches <= 0):
        return 0, 0
    eng = engine_for(model, device, batch_hint=int(first["pixel_values"].shape[0]))
    correct = torch.zeros(1, device=eng.device, dtype=torch.int64)
    total = 0
    for i, batch in enumerate(batches):
        if max_batches is not None and i >= max_batches:
            break
        total += eng.eval_batch(batch["pixel_values"], batch["labels"], correct, skip_attn)
    return int(correct.item()), total


@torch.no_grad()
def evaluate_top1(model, dataloader, device: str = "cuda", max_batches: Optional[int] = None, progress: bool = False):
    """Top-1 accuracy over at most `max_batches` batches (src/vit_pruning.py:325-373). One device->host read
    at the end instead of one `.item()` per batch."""
    correct, total = _top1_counts(model, dataloader, device, max_batches)
    return correct / max(1, total)


@torch.no_grad()
def measure_latency(model, device: str = "cuda", warmup: int = 3, iters: int = 10, img_size: Optional[int] = 224, batch: int = 1) -> float:
    """Seconds per forward of a random batch (default one image), wall clock between synchronisations, as
    experiments/vit_pruning/auto_2ssp.py:74-99 -- through the engine, so pruned widths and bypassed blocks count.
    img_size=None takes the model's own input resolution."""
    import time
    model.eval()
    eng = engine_for(model, device, batch_hint=max(16, batch))
    size = eng.anatomy.image_size if img_size is None else img_size
    dummy = torch.randn(batch, eng.anatomy.channels, size, size, device=eng.device)
    for _ in range(warmup):
        eng.logits(dummy)
    torch.cuda.synchronize(eng.device)
    start = time.time()
    for _ in range(iters):
        eng.logits(dummy)
    torch.cuda.synchronize(eng.device)
    return (time.time() - start) / iters


# ------------------------------------------------------------------------------------------ stage 2
@torch.no_grad()
def attention_removal_counts(vit_model, dataloader, device="cuda", batch_limit: Optional[int] = 5, *, group=None,
                             shard: str = "candidates", with_scores: bool = False):
    """(baseline_correct, [correct with block i's attention removed], images) over <= batch_limit batches.

    Replaces the B deep copies + B+1 full evaluations of the reference (src/vit_pruning.py:463-497,
    mask_conjunction.py:327-357) by one cached baseline pass and B suffix recomputations per batch.
    With `group` and shard="candidates" every rank passes the SAME data, candidates are dealt across ranks and the
    integer counts summed; with shard="images" every rank passes ITS OWN shard of the data, evaluates all candidates
    on it, and counts and image totals are summed. Both are exact (integers).

    with_scores=True: the baseline pass runs with the scoring fc1 epilogue, so the Stage-1 importances of the same
    images (what `_compute_ffn_activation_importance` would return for this dataloader and batch_limit, bit for bit on
    one GPU) come out of the same sweep; a fourth value, List[B] of CPU fp32 tensors, is returned.
    """
    if shard not in ("candidates", "images"):
        raise ValueError(f"shard must be 'candidates' or 'images', not {shard!r}")
    vit_model.eval()
    kind, blocks = get_blocks(vit_model)
    nb = len(blocks)
    first, batches = _peek(dataloader)
    rank, world = D.rank_world(group) if group is not None else (0, 1)
    if first is None:
        widths = [fc1.out_features for fc1, _ in gather_mlp_pairs(vit_model)]
        if world > 1 and shard == "images":  # an empty shard still takes part in the sums, in the order the other ranks use
            dev = _cuda_device(device)
            scores = None
            if with_scores:
                sums, seen = D.reduce_score_sums(torch.zeros(sum(widths), device=dev, dtype=torch.float32), 0, group)
                scores = [t.clone() for t in torch.split(sums.cpu() / max(1, seen), widths)]
            counts, total = D.sum_image_shard_counts([0] * (nb + 1), 0, group, device=dev)
            return (counts[0], counts[1:], total, scores) if with_scores else (counts[0], counts[1:], total)
        zeros = [torch.zeros(w) for w in widths]  # as Stage 1 on an empty loader (src/vit_pruning.py:197-198)
        return (0, [0] * nb, 0, zeros) if with_scores else (0, [0] * nb, 0)
    eng = engine_for(vit_model, device, batch_hint=int(first["pixel_values"].shape[0]), need_cache=True)
    mine = D.zigzag_candidates(nb, rank, world) if (world > 1 and shard == "candidates") else None
    eng.s2_reset()
    if with_scores:
        eng.s1_reset()
    total = 0
    for i, batch in enumerate(batches):
        if batch_limit is not None and i >= batch_limit:
            break
        total += eng.s2_batch(batch["pixel_values"], batch["labels"], candidates=mine, run_baseline=True, with_scores=with_scores)
    counts = eng.s2_counts()
    scores = None
    if with_scores:
        if world > 1 and shard == "images":  # every rank saw its own images: one all-reduce of the sums, as in Stage 1
            sums, seen = D.reduce_score_sums(eng.s1_score_sums(on_device=True), total, group)
            sums = sums.cpu()
        else:                                # one GPU, or candidate sharding (every rank swept ALL images)
            sums, seen = eng.s1_score_sums(on_device=False), total
        scores = [t.clone() for t in eng.split_blocks(sums / max(1, seen))]
    if world > 1 and shard == "candidates":
        counts = D.merge_candidate_counts(counts, group, device=eng.device)  # disjoint candidate sets: exact
    elif world > 1:
        counts, total = D.sum_image_shard_counts(counts, total, group, device=eng.device)
    if with_scores:
        return counts[0], counts[1:], total, scores
    return counts[0], counts[1:], total


@torch.no_grad()
def prune_vit_attention_blocks(
    vit_model,
    sparsity: float,
    dataloader=None,
    device: str = "cuda",
    batch_limit: int = 5,
    metric_fn=None,
    importance_mode: str = "copy",
    show_progress: bool = True,
    num_to_prune: Optional[int] = None,
    selected_indices: Optional[List[int]] = None,
) -> Dict[str, Any]:
    """Remove the attention submodule of the selected blocks (src/vit_pruning.py:379-520); same selection
    rules, same in-place mutation (bypass modules), same return dict."""
    if not (0.0 <= sparsity < 1.0):
        raise AssertionError("sparsity must be in [0,1)")
    vit_model.eval()
    try:
        _, blocks = get_blocks(vit_model)
        num_blocks = len(blocks)
    except AttributeError:
        num_blocks = 0
    if num_to_prune is None:
        num_to_prune = int(round(num_blocks * sparsity))
    num_to_prune = max(0, min(num_blocks - 1, int(num_to_prune)))
    if num_to_prune == 0:
        print("No attention submodules to prune (num_to_prune=0).")
        return {"model": vit_model, "pruned_indices": [], "original_metrics": None, "final_metrics": None}

    original_metrics = None
    final_metrics = None
    if selected_indices is not None:
        to_prune = sorted(set(i for i in selected_indices if 0 <= i < num_blocks))[:num_to_prune]
    elif dataloader is None or (isinstance(importance_mode, str) and importance_mode.lower() == "heuristic"):
        print("Using heuristic for attention pruning importance (position-based).")
        scores = [(i if i < num_blocks / 2 else num_blocks - i) for i in range(num_blocks)]
        to_prune = sorted(range(num_blocks), key=lambda i: scores[i])[:num_to_prune]
    else:
        print(f"Evaluating {num_blocks} blocks by impact of removing attention (cached-prefix recompute)...")
        base, cand, total = attention_removal_counts(vit_model, dataloader, device, batch_limit)
        original_metrics = base / max(1, total)
        print(f"Baseline accuracy: {original_metrics:.4f}")
        impact_scores = [max(0.0, original_metrics - c / max(1, total)) for c in cand]
        if show_progress:
            for i, imp in enumerate(impact_scores):
                print(f"[Attn] Block {i} impact: {imp:.4f}", flush=True)
        to_prune = sorted(range(num_blocks), key=lambda i: impact_scores[i])[:num_to_prune]  # stable, like the reference
        print(f"Selected blocks to remove attention: {to_prune}")

    slot = _engine_in_step(vit_model)       # signature BEFORE the bypass modules are installed
    stale = slot is None and vit_model in _ENGINES
    for idx in to_prune:
        install_bypass(vit_model, idx)
    if slot is not None:
        kind, blocks = get_blocks(vit_model)
        slot["engine"].set_attention([has_attention(kind, b) for b in blocks])
        slot["sig"] = _signature(vit_model)
    elif stale:
        release_engine(vit_model)

    if dataloader is not None:
        final_metrics = evaluate_top1(vit_model, dataloader, device, max_batches=batch_limit, progress=True)
        print(f"Final accuracy after attention pruning: {final_metrics:.4f}")
        if original_metrics is not None:
            print(f"Accuracy change: {final_metrics - original_metrics:.4f}")
    return {"model": vit_model, "pruned_indices": sorted(list(to_prune)), "original_metrics": original_metrics,
            "final_metrics": final_metrics}


# ------------------------------------------------------------------------------------------ planner
@dataclass
class TwoSSPPlan:
    target_sparsity: float
    num_blocks_total: int
    blocks_to_prune: int
    per_block_neurons_to_prune: int
    stage2_fraction: float
    estimated_total_removed_params: int
    est_error_params: int


@torch.no_grad()
def plan_2ssp_allocation(vit_model, target_sparsity: float, min_remaining: int = 256,
                         forced_blocks: Optional[int] = None) -> TwoSSPPlan:
    """Split one global sparsity target between Stage-2 (K attention removals) and Stage-1 (t neurons per
    block) -- integer host logic of src/vit_pruning.py:586-769, same tie rules and log tags."""
    if not (0.0 < target_sparsity < 1.0):
        raise AssertionError("target_sparsity must be in (0,1)")
    total_params = count_total_params(vit_model)
    block_params = count_block_params(vit_model)
    B = len(block_params)
    P_target = int(round(total_params * target_sparsity))
    hidden, inter_sizes = _get_hidden_and_inter_sizes(vit_model)
    if hidden is None or len(inter_sizes) != B:
        raise RuntimeError("Unable to determine hidden/intermediate sizes for planning.")
    t_max = min((max(0, f - min_remaining) for f in inter_sizes), default=0)
    neuron_cost = 2 * hidden + 1
    denom = B * neuron_cost
    print(f"[PLAN-LOG] B={B}, target_sparsity={target_sparsity}, P_target={P_target}")
    print(f"[PLAN-LOG] hidden={hidden}, inter_sizes={inter_sizes}, min_remaining={min_remaining}")
    print(f"[PLAN-LOG] total_params={total_params}, block_params={block_params}")
    print(f"[PLAN-LOG] t_max_uniform={t_max}, denom=B*(2*hidden+1)={denom}")
    tol = max(1, int(0.02 * P_target))
    attn_counts = _count_attention_params_per_block(vit_model)
    ffn_counts = _count_ffn_params_per_block(vit_model)
    P_attn = sum(attn_counts) / max(1, B)
    W_ffn = sum(ffn_counts) / max(1, B)
    print(f"[PLAN-LOG] attn_params_per_block={attn_counts}")
    print(f"[PLAN-LOG] ffn_params_per_block={ffn_counts}")

    def removed_by(K: int, t: int) -> int:
        return int(round(K * P_attn)) + (t * neuron_cost if t > 0 else 0) * B

    def uniform_t(K: int) -> int:
        rest = max(0, P_target - int(round(K * P_attn)))
        t = int(round(rest / denom)) if denom > 0 else 0
        return max(0, min(t, t_max))

    def prefer(new, cur) -> bool:
        return (new[0] < cur[0] - tol) or (abs(new[0] - cur[0]) <= tol and new[1] > cur[1])

    def scored(K: int, t: int):
        total = removed_by(K, t)
        return (abs(P_target - total), K, t, total)

    if forced_blocks is not None:
        K_values = [max(0, min(B - 1, int(forced_blocks)))]
        print(f"[PLAN-LOG] forced_blocks provided: K_values={K_values}")
    else:
        K_formula = int(round(B * (target_sparsity ** (W_ffn / (1.5 * P_attn))))) if P_attn > 0 else 0
        K_formula = max(0, min(B - 1, K_formula))
        K_values = [k for k in sorted({K_formula + d for d in (-2, -1, 0, 1, 2)}) if 0 <= k <= B - 1]
        print(f"[PLAN-LOG] K_formula={K_formula}, K_candidates={K_values}")

    best = None
    for K in K_values:
        t0 = uniform_t(K)
        for t in (t0, *(max(0, min(t0 + dt, t_max)) for dt in (-1, 1, 2, -2))):
            cand = scored(K, t)
            if best is None or prefer(cand, best):
                best = cand

    if best is not None and forced_blocks is None and best[1] == 0 and P_attn > 0 and P_target >= 0.5 * P_attn:
        K_guess = max(1, int(round(P_target / max(1, P_attn))))
        alt = None
        for K in range(1, min(B - 1, K_guess + 2) + 1):
            cand = scored(K, uniform_t(K))
            if alt is None or prefer(cand, alt):
                alt = cand
        if alt is not None and ((alt[0] < best[0] - tol) or abs(alt[0] - best[0]) <= tol):
            best = alt

    if best is None:
        return TwoSSPPlan(target_sparsity, B, 0, 0, 0.0, 0, P_target)
    err, K, t, total = best
    frac = (K / B) if B > 0 else 0.0
    print(f"[PLAN-LOG] chosen: K={K}, t={t}, stage2_fraction={frac:.6f}")
    print(f"[PLAN-LOG] removal_depth(attn)={int(round(K * P_attn))}, removal_width(ffn)={(t * neuron_cost if t > 0 else 0) * B}, "
          f"total={total}, target={P_target}, err={int(err)}")
    return TwoSSPPlan(target_sparsity, B, K, t, frac, total, int(err))


# ------------------------------------------------------------------------------------------ plugin boundary
class PruningTypes(Enum):
    """pruning_srp-main/mask_conjunction.py:32-36."""
    DEPTH = 0
    WIDTH = 1
    HEAD = 2
    NONE = 3


class PruningInterface:
    """pruning_srp-main/mask_conjunction.py:38-48: what the external framework instantiates and calls."""

    def __init__(self, model, pruning_dataloader):
        self.nn = model
        self.dl = pruning_dataloader
        self.att_prune_type = PruningTypes.DEPTH
        self.mlp_prune_type = PruningTypes.WIDTH


class B200Auto2SSPInterface(PruningInterface):
    """Auto2SSPInterface (pruning_srp-main/mask_conjunction.py:236-362) on the B200 backend.

    fit() -> (att_importance: FloatTensor[B] on CPU, mlp_importance: List[B] of CPU tensors [F]);
    lower importance = pruned earlier. Differences from the reference, all deliberate:
      * a failing backend raises (the reference silently falls back to weight-L1 scores, :286-296);
      * error_policy="heuristic" still maps evaluation errors to the heuristic scores (:330-355);
      * fuse_passes (default on): inside fit() the Stage-2 baseline pass runs with the scoring fc1 epilogue, so the
        Stage-1 importances come out of the same sweep over the calibration images instead of a second one (the
        reference sweeps the same loader twice, :359-362). Same numbers as the separate call (bit for bit on one GPU for
        a loader that yields the same batches twice); the stand-alone methods are unchanged.
    """

    def __init__(self, model, pruning_dataloader, device=None, importance_mode="copy", batch_limit=5, min_remaining=256,
                 error_policy="raise", group=None, s2_shard="candidates", fuse_passes=True):
        super().__init__(model, pruning_dataloader)
        self.fuse_passes = fuse_passes
        self._fusing = False      # True only between the two calls inside fit()
        self._fused_mlp = None
        self.s2_shard = s2_shard  # with `group`: "candidates" (same data on every rank) or "images" (own shard per rank)
        self.device = device or "cuda"
        self.importance_mode = importance_mode
        self.batch_limit = batch_limit
        self.min_remaining = min_remaining
        self.error_policy = error_policy
        self.group = group
        self._get_encoder = get_encoder
        self._gather_mlp_pairs = gather_mlp_pairs
        self._evaluate_top1 = evaluate_top1
        self._compute_ffn_activation_importance = _compute_ffn_activation_importance
        self.last_counts = None

    def _num_blocks(self) -> int:
        _, blocks = get_blocks(self.nn)
        return len(blocks)

    def _compute_mlp_importance(self):
        if self._fusing and self._fused_mlp is not None:
            imps, self._fused_mlp = self._fused_mlp, None
            return imps
        if self.dl is not None:
            imps = _compute_ffn_activation_importance(self.nn, self.dl, device=self.device, batch_limit=self.batch_limit,
                                                      progress=False, group=self.group)
            return [t.detach().to("cpu") for t in imps]
        return [fc1.weight.abs().sum(dim=1).detach().to("cpu") for fc1, _ in gather_mlp_pairs(self.nn)]

    def _compute_att_depth_importance(self):
        B = self._num_blocks()
        heuristic = [(i if i < B / 2 else B - i) for i in range(B)]
        if self.importance_mode.lower() == "heuristic" or self.dl is None:
            return torch.tensor(heuristic, dtype=torch.float32)
        try:
            if self._fusing:
                base, cand, total, scores = attention_removal_counts(self.nn, self.dl, self.device, self.batch_limit, group=self.group,
                                                                     shard=self.s2_shard, with_scores=True)
                self._fused_mlp = [t.detach().to("cpu") for t in scores]
            else:
                base, cand, total = attention_removal_counts(self.nn, self.dl, self.device, self.batch_limit, group=self.group,
                                                             shard=self.s2_shard)
        except Exception:
            if getattr(self, "error_policy", "raise") == "raise":
                raise
            return torch.tensor(heuristic, dtype=torch.float32)
        self.last_counts = (base, cand, total)
        baseline = base / max(1, total)
        return torch.tensor([max(0.0, baseline - c / max(1, total)) for c in cand], dtype=torch.float32)

    def fit(self):
        fuse = bool(self.fuse_passes) and self.dl is not None and str(self.importance_mode).lower() != "heuristic"
        self._fusing, self._fused_mlp = fuse, None
        try:
            self.att_importance = self._compute_att_depth_importance()
            self.mlp_importance = self._compute_mlp_importance()
        finally:
            self._fusing, self._fused_mlp = False, None
        return self.att_importance, self.mlp_importance


# ------------------------------------------------------------------------------------------ wire formats
_FLOAT_REPR = float.__repr__


def _json_float(v: float) -> str:
    if v != v:
        return "NaN"
    if v in (float("inf"), float("-inf")):
        return "Infinity" if v > 0 else "-Infinity"
    return _FLOAT_REPR(v)


def _json_indent2(obj, ensure_ascii: bool = True, level: int = 0) -> str:
    """The bytes `json.dumps(obj, indent=2, ensure_ascii=...)` produces, built with joins over flat int / float
    containers (the pure-Python encoder json falls back to when indent is set spends 50 ms on a ViT-B score file)."""
    pad, pad1 = "  " * level, "  " * (level + 1)
    if isinstance(obj, dict):
        if not obj:
            return "{}"
        keys = [k if isinstance(k, str) else (json.dumps(k) if not isinstance(k, (int, float)) or isinstance(k, bool) else str(k)) for k in obj]
        if all(type(v) is float for v in obj.values()):
            vals = [_json_float(v) for v in obj.values()]
        else:
            vals = [_json_indent2(v, ensure_ascii, level + 1) for v in obj.values()]
        sep = ",\n" + pad1
        return "{\n" + pad1 + sep.join([json.dumps(k, ensure_ascii=ensure_ascii) + ": " + v for k, v in zip(keys, vals)]) + "\n" + pad + "}"
    if isinstance(obj, (list, tuple)):
        if not obj:
            return "[]"
        sep = ",\n" + pad1
        if all(type(v) is int for v in obj):
            return "[\n" + pad1 + sep.join(map(str, obj)) + "\n" + pad + "]"
        if all(type(v) is float for v in obj):
            return "[\n" + pad1 + sep.join(map(_json_float, obj)) + "\n" + pad + "]"
        return "[\n" + pad1 + sep.join([_json_indent2(v, ensure_ascii, level + 1) for v in obj]) + "\n" + pad + "]"
    if type(obj) is float:
        return _json_float(obj)
    return json.dumps(obj, ensure_ascii=ensure_ascii)


_KEY_PREFIXES: Dict[tuple, List[str]] = {}


def _ffn_scores_text_py(mlp_importance: Sequence[torch.Tensor]) -> str:
    """Pure-Python form of the score file text (any dtype; also what the C formatter is tested against)."""
    parts = []
    for b, imp in enumerate(mlp_importance):
        t64 = imp.detach().cpu().flatten().to(torch.float64)  # float(v) of the reference: the exact double
        vals = t64.tolist()
        key = (b, len(vals))
        prefix = _KEY_PREFIXES.get(key)
        if prefix is None:
            if len(_KEY_PREFIXES) > 256:
                _KEY_PREFIXES.clear()
            prefix = _KEY_PREFIXES[key] = [f'    "{b}:{j}": ' for j in range(len(vals))]
        reprs = map(_FLOAT_REPR, vals) if bool(torch.isfinite(t64).all()) else map(_json_float, vals)
        if vals:
            parts.append(",\n".join(map(str.__add__, prefix, reprs)))
    return '{\n  "ffn": {\n' + ",\n".join(parts) + "\n  }\n}" if parts else '{\n  "ffn": {}\n}'


def _ffn_scores_text(mlp_importance: Sequence[torch.Tensor]) -> bytes:
    """The bytes of json.dumps({"ffn": {"<block>:<neuron>": float(score)}}, indent=2). fp32 / fp16 / bf16 scores (what this
    path and the reference produce) go through tssp_format_ffn_scores -- shortest round-trip digits laid out by CPython's
    repr rule, 3 ms for a ViT-B file against 10-20 ms of Python string work; other dtypes take the Python form."""
    imps = [imp.detach().cpu().flatten() for imp in mlp_importance]
    if imps and all(t.dtype in (torch.float32, torch.float16, torch.bfloat16) for t in imps):
        import ctypes as C
        try:
            lib = L.load()
        except L.TsspError:
            lib = None
        if lib is not None:
            flat = torch.cat([t.to(torch.float32) for t in imps]).contiguous()
            widths = (C.c_int32 * len(imps))(*[int(t.numel()) for t in imps])
            cap = 64 * int(flat.numel()) + 64
            buf = C.create_string_buffer(cap)
            n = lib.tssp_format_ffn_scores(C.c_void_p(flat.data_ptr()), widths, len(imps), buf, cap)
            if n < 0 or n > cap:
                L.check(1)
            return buf.raw[:n]
    return _ffn_scores_text_py(mlp_importance).encode("utf-8")


def save_ffn_importances(mlp_importance: Sequence[torch.Tensor], path: str) -> str:
    """{"ffn": {"<block>:<neuron>": score}} in (block, neuron) order, indent=2
    (experiments/vit_pruning/auto_2ssp.py:769-786; manual-experiments/2ssp_vit_b16_ffn_importances.json): the bytes of
    json.dump({"ffn": {...}}, f, ensure_ascii=False, indent=2). (Writing from a worker thread during select + gather was
    measured SLOWER: the two Python threads fight over the GIL and the flow has no GPU time to hide behind.)"""
    text = _ffn_scores_text(list(mlp_importance))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "wb") as f:
        f.write(text)
    return path


def save_ffn_masks(masks: List[List[int]], indices: List[List[int]], path: str, *, min_remaining: int,
                   block_inter_sizes: Optional[List[int]] = None, s1_sparsity: Optional[float] = None,
                   strategy: str = "act_l2") -> str:
    """experiments/vit_pruning/auto_2ssp.py:789-806."""
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w", encoding="utf-8") as f:
        f.write(_json_indent2({"format_version": 1, "stage": "s1", "strategy": strategy, "min_remaining": min_remaining,
                               "s1_sparsity": s1_sparsity, "block_inter_sizes": block_inter_sizes, "masks": masks, "indices": indices}))
    return path


def save_attention_indices(indices: List[int], path: str) -> str:
    """experiments/vit_pruning/auto_2ssp.py:808-817."""
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w", encoding="utf-8") as f:
        json.dump({"format_version": 1, "stage": "s2", "indices": list(indices)}, f, indent=2)
    return path


def save_framework_export(prefix: str, model, mlp_importance: Optional[Sequence[torch.Tensor]], att_importance=None,
                          ffn_masks: Optional[List[List[int]]] = None,
                          pruned_attn_block_indices: Optional[Sequence[int]] = None) -> Dict[str, str]:
    """<prefix>_scores.json {"ffn","heads","qkv_dim"} and <prefix>_masks.json, the layout of
    adaptation-for-Pures-framework/auto_2ssp.py:71-185: FFN scores per "<layer>:<neuron>"; the per-block
    attention importance broadcast to every head / qkv dim of the block; masks as one 0/1 list per layer
    (1 = pruned), heads and qkv dims fully masked for blocks whose attention was removed."""
    _, blocks = get_blocks(model)
    B = len(blocks)
    cfg = getattr(model, "config", None)
    hidden = getattr(cfg, "hidden_size", None) or 768
    num_heads = getattr(cfg, "num_attention_heads", None) or 12
    imps = list(mlp_importance or [])
    ffn_scores = {f"{l}:{i}": float(v) for l, vec in enumerate(imps) for i, v in enumerate(vec.detach().cpu().tolist())}
    if att_importance is not None:
        att_vals = [float(v) for v in att_importance.detach().cpu().tolist()]
        att_vals = (att_vals + [0.0] * B)[:B]
    else:
        att_vals = [0.0] * B
    head_scores = {f"{l}:{h}": att_vals[l] for l in range(B) for h in range(num_heads)}
    qkv_scores = {f"{l}:{d}": att_vals[l] for l in range(B) for d in range(hidden)}
    if ffn_masks is not None and len(ffn_masks) == B:
        ffn_mask = {str(l): m for l, m in enumerate(ffn_masks)}
    else:
        ffn_mask = {str(l): [0] * int(len(imps[l]) if l < len(imps) else hidden * 4) for l in range(B)}
    gone = set(pruned_attn_block_indices or [])
    head_mask = {str(l): [1 if l in gone else 0] * num_heads for l in range(B)}
    qkv_mask = {str(l): [1 if l in gone else 0] * hidden for l in range(B)}
    d = os.path.dirname(prefix)
    os.makedirs(d if d else ".", exist_ok=True)
    out = {"scores": prefix + "_scores.json", "masks": prefix + "_masks.json"}
    with open(out["scores"], "w") as f:
        f.write(_json_indent2({"ffn": ffn_scores, "heads": head_scores, "qkv_dim": qkv_scores}))
    with open(out["masks"], "w") as f:
        f.write(_json_indent2({"ffn": ffn_mask, "heads": head_mask, "qkv_dim": qkv_mask}))
    return out


# ------------------------------------------------------------------------------------------ external masks -> gather
_IJ_KEY = re.compile(r"^(\d+):(\d+)$")


def load_ffn_mask(path: str) -> Dict[int, Dict[int, int]]:
    """Mask JSON -> {block: {neuron: 0/1}} (experiments/vit_pruning/apply_mask_prune.py:200-256): every nested dict
    whose keys all look like "<block>:<neuron>" with numeric values is a leaf; leaves are merged; bit = round(value) != 0."""
    with open(path, "r", encoding="utf-8") as f:
        data = json.load(f)
    leaves: List[Dict[str, Any]] = []

    def walk(obj):
        if isinstance(obj, dict):
            if obj and all(isinstance(k, str) and _IJ_KEY.match(k) and isinstance(v, (int, float)) for k, v in obj.items()):
                leaves.append(obj)
                return
            for v in obj.values():
                walk(v)
        elif isinstance(obj, list):
            for v in obj:
                walk(v)

    walk(data)
    if not leaves:
        raise RuntimeError(f"Mask file has no ij-leaf dicts: {path}")
    blocks: Dict[int, Dict[int, int]] = {}
    for leaf in leaves:
        for k, v in leaf.items():
            m = _IJ_KEY.match(k)
            blocks.setdefault(int(m.group(1)), {})[int(m.group(2))] = 1 if int(round(float(v))) != 0 else 0
    return blocks


def mask_to_importance(blocks_mask: Dict[int, Dict[int, int]], inter_sizes: Sequence[int]):
    """(+1 keep / -1 prune importance per block, number of ones per block) -- apply_mask_prune.py:259-280; neurons
    that the mask does not mention are kept."""
    imp, n_prune = [], []
    for i, width in enumerate(inter_sizes):
        vec = torch.ones(width, dtype=torch.float32)
        ones = [j for j, bit in blocks_mask.get(i, {}).items() if bit == 1 and 0 <= j < width]
        if ones:
            vec[torch.tensor(ones, dtype=torch.int64)] = -1.0
        imp.append(vec)
        n_prune.append(len(ones))
    return imp, n_prune


@torch.no_grad()
def apply_ffn_mask(vit_model, mask, min_remaining: int = 256, device: str = "cuda"):
    """External 0/1 mask (path or {block: {neuron: bit}}) -> Stage-1 gather, the flow of apply_mask_prune.py:366-392:
    +-1 importances, per-block counts clamped to min_remaining, prune_vit_mlp_width(precomputed_importance=...)."""
    blocks_mask = load_ffn_mask(mask) if isinstance(mask, (str, os.PathLike)) else mask
    _, inter_sizes = _get_hidden_and_inter_sizes(vit_model)
    imp, n_prune = mask_to_importance(blocks_mask, inter_sizes)
    for i, (width, k) in enumerate(zip(inter_sizes, n_prune)):
        if width - k < min_remaining:
            adj = max(0, width - min_remaining)
            if k > adj:
                print(f"[WARN] Block {i}: requested prune {k} exceeds min_remaining constraint ({min_remaining}). Adjusting to {adj}.")
                n_prune[i] = adj
    return prune_vit_mlp_width(vit_model, n_to_prune_per_block=n_prune, min_remaining=min_remaining, strategy="l1", dataloader=None,
                               device=device, progress=False, collect_masks=True, precomputed_importance=imp)


# ------------------------------------------------------------------------------------------ iterative Stage 2
@torch.no_grad()
def attention_removal_iterative(vit_model, dataloader, num_to_prune: int, device="cuda", batch_limit: Optional[int] = 5):
    """Paper-faithful greedy Stage 2 (the LLM original, src/utilities.py:446-505): remove the attention whose removal
    hurts least, then re-evaluate the remaining blocks WITH it removed, `num_to_prune` times. The metric is top-1
    accuracy (maximised; the first best block wins ties, like the strict `<` of the original on perplexity).

    Does not mutate `vit_model`; returns (removal_order, top1_after_each_removal). Every round is one cached baseline
    pass plus one suffix recomputation per remaining block inside the engine.
    """
    vit_model.eval()
    kind, blocks = get_blocks(vit_model)
    nb = len(blocks)
    present0 = [has_attention(kind, b) for b in blocks]
    batches = list(dataloader) if batch_limit is None else [b for i, b in zip(range(batch_limit), dataloader)]
    if not batches:
        return [], []
    eng = engine_for(vit_model, device, batch_hint=int(batches[0]["pixel_values"].shape[0]), need_cache=True)
    present = list(present0)
    order: List[int] = []
    accs: List[float] = []
    try:
        for _ in range(max(0, min(int(num_to_prune), sum(present0) - 1))):
            cands = [i for i in range(nb) if present[i]]
            eng.set_attention(present)
            eng.s2_reset()
            total = 0
            for batch in batches:
                total += eng.s2_batch(batch["pixel_values"], batch["labels"], candidates=cands, run_baseline=False)
            counts = eng.s2_counts()[1:]
            best = max(cands, key=lambda i: (counts[i], -i))
            present[best] = False
            order.append(best)
            accs.append(counts[best] / max(1, total))
    finally:
        eng.set_attention(present0)
    return order, accs
