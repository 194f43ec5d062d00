"""Seeded timm-shaped CLIP image towers (OpenAI / LAION ViT-B/32, B/16, L/14, L/14@336 at test and full size) for the CLIP
tests and tools/clip_bench.py (TEST / MEASUREMENT INFRASTRUCTURE).

timm is not installed here, so `TimmLikeClipViT` restates the parts of timm's `VisionTransformer` with `pre_norm=True`
that the engine reads, with timm's attribute names: `norm_pre` (a LayerNorm over every token after `_pos_embed`, before
block 0), a bias-free `patch_embed.proj` (timm passes `bias=not pre_norm`), `blocks[i].mlp.act` = `QuickGELU`
(`act_layer='quick_gelu'` of the OpenAI weights: x * sigmoid(1.702 x)), LayerNorm eps 1e-5 throughout, token pooling and a
Linear head with a zero bias (timm's `_convert_openai_clip` maps `proj` to `head` with a zero bias). Values are portable
(bit-identical on every CPU, see oracle.synth._portable_normal). Kept next to the tests so that oracle/ and its golden
vectors stay as they are.
"""
from __future__ import annotations

import os
import sys

import torch

from oracle.synth import _portable_normal, _TimmLikeBlock

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import layerscale_synth as LS  # noqa: E402

CLIP_SHAPES = {
    # name: (image, patch, dim, depth, heads, hidden, classes)
    "tiny": (48, 8, 128, 3, 2, 512, 10),          # T = 37
    "tiny192": (48, 8, 192, 3, 3, 768, 10),       # T = 37, the 192-wide LayerNorm / GEMM forms
    "b32": (224, 32, 768, 12, 12, 3072, 1000),    # T = 50, K = 3072 patch GEMM
    "b16": (224, 16, 768, 12, 12, 3072, 1000),    # T = 197
    "l14": (224, 14, 1024, 24, 16, 4096, 1000),   # T = 257
    "l14_336": (336, 14, 1024, 24, 16, 4096, 1000),  # T = 577
}
EPS = 1e-5


class QuickGELU(torch.nn.Module):
    """timm.layers.QuickGELU (and open_clip's): x * sigmoid(1.702 x)."""

    def forward(self, x):
        return x * torch.sigmoid(1.702 * x)


def _init(model, dim, seed):
    """Matrices scale with 1 / sqrt(width) as in layerscale_synth; fc1 biases centred at -1 so that a real share of the
    pre-activations falls in [-4, 0], where QuickGELU and erf GELU differ most; the head bias stays zero."""
    g = torch.Generator().manual_seed(seed)
    w_std = 0.05 * (128 / dim) ** 0.5
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("gamma"):
                p.copy_(0.5 + _portable_normal(p.shape, g) * 0.1)
            elif name == "head.bias":
                p.zero_()
            elif name.endswith("mlp.fc1.bias"):
                p.copy_(_portable_normal(p.shape, g) - 1.0)
            elif p.dim() >= 2:
                p.copy_(_portable_normal(p.shape, g) * w_std)
            elif p.dim() == 1 and p.numel() > 1:
                p.add_(_portable_normal(p.shape, g) * 0.02)


class TimmLikeClipViT(torch.nn.Module):
    """act: "quick_gelu" or "gelu" (erf, nn.GELU()); pre_norm=False: `norm_pre` is Identity and the patch projection has a
    bias, as timm builds a tower without pre_norm."""

    def __init__(self, dim=128, heads=2, hidden=512, depth=3, image=48, patch=8, classes=10, act="quick_gelu", pre_norm=True,
                 seed=3):
        super().__init__()
        self.patch_embed = torch.nn.Module()
        self.patch_embed.proj = torch.nn.Conv2d(3, dim, patch, patch, bias=not pre_norm)
        self.cls_token = torch.nn.Parameter(torch.zeros(1, 1, dim))
        self.num_prefix_tokens = 1
        self.global_pool = "token"
        self.pos_embed = torch.nn.Parameter(torch.zeros(1, (image // patch) ** 2 + 1, dim))
        self.norm_pre = torch.nn.LayerNorm(dim, eps=EPS) if pre_norm else torch.nn.Identity()
        self.blocks = torch.nn.ModuleList([_TimmLikeBlock(dim, heads, hidden) for _ in range(depth)])
        for b in self.blocks:
            b.norm1.eps = b.norm2.eps = EPS
            b.mlp.act = QuickGELU() if act == "quick_gelu" else torch.nn.GELU()
        self.norm = torch.nn.LayerNorm(dim, eps=EPS)
        self.head = torch.nn.Linear(dim, classes)
        _init(self, dim, seed)
        self.eval()

    def forward(self, x):
        t = self.patch_embed.proj(x).flatten(2).transpose(1, 2)
        t = torch.cat([self.cls_token.expand(t.shape[0], -1, -1), t], dim=1) + self.pos_embed
        t = self.norm_pre(t)
        for b in self.blocks:
            t = b(t)
        return self.head(self.norm(t)[:, 0])


class ClipLayerScaleViT(LS.TimmLikeLayerScaleViT):
    """The combined layout: LayerScale and register tokens (layerscale_synth) with `norm_pre` and QuickGELU."""

    def __init__(self, seed=3):
        super().__init__(reg_tokens=4, no_embed_class=True, seed=seed)   # the tiny_reg4 shape: D = 128, T = 41
        self.norm_pre = torch.nn.LayerNorm(128, eps=1e-6)                 # eps of the stand-in's other norms
        for b in self.blocks:
            b.mlp.act = QuickGELU()
        _init(self, 128, seed)
        self.eval()

    def forward(self, x):
        t = self.norm_pre(self._pos_embed(self.patch_embed(x)))
        for b in self.blocks:
            t = b(t)
        return self.head(self.norm(t)[:, 0])


def make_clip(name: str, seed: int = 3, act: str = "quick_gelu", pre_norm: bool = True) -> TimmLikeClipViT:
    image, patch, dim, depth, heads, hidden, classes = CLIP_SHAPES[name]
    return TimmLikeClipViT(dim, heads, hidden, depth, image, patch, classes, act, pre_norm, seed)


def image_size(name: str) -> int:
    return CLIP_SHAPES[name][0]
