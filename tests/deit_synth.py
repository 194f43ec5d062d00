"""Seeded synthetic DeiT models for the DeiT tests and tools/deit_bench.py (TEST / MEASUREMENT INFRASTRUCTURE).

Built like oracle/synth.py's `make_vit` (random-init HF module under `torch.manual_seed(seed)`, then portable values
from `torch.Generator().manual_seed(1000003 + seed)`), so the bits are the same on every CPU. Kept next to the tests so
that oracle/ and the golden vectors pinned to it stay as they are.
"""
from __future__ import annotations

import torch

from oracle.synth import _PatchEmbed, _portable_normal, _TimmLikeBlock

DEIT_SHAPES = {
    # name: (image, patch, hidden, layers, heads, ffn, labels) in the layout of oracle.synth.SHAPES
    "tiny": (48, 8, 192, 3, 3, 768, 10),            # T = 38, D = 192: the DeiT-Ti width at test size
    "ti": (224, 16, 192, 12, 3, 768, 1000),         # DeiT-Ti/16, T = 198
    "small": (224, 16, 384, 12, 6, 1536, 1000),     # DeiT-S/16
    "base": (224, 16, 768, 12, 12, 3072, 1000),     # DeiT-B/16
    "base384": (384, 16, 768, 12, 12, 3072, 1000),  # DeiT-B/16 at 384^2, T = 578
}

HEADS = ("teacher", "cls", None)


def make_deit(shape: str = "tiny", seed: int = 0, head: str | None = "teacher"):
    """Random-init HF DeiT of the named shape. head="teacher": DeiTForImageClassificationWithTeacher (averaged CLS and
    distillation heads); "cls": DeiTForImageClassification (CLS head only); None: DeiTModel (no head)."""
    from transformers import DeiTConfig, DeiTForImageClassification, DeiTForImageClassificationWithTeacher, DeiTModel
    if head not in HEADS:
        raise ValueError(f"head={head!r} is not one of {HEADS}")
    image, patch, hidden, layers, heads, ffn, labels = DEIT_SHAPES[shape]
    cfg = DeiTConfig(image_size=image, patch_size=patch, hidden_size=hidden, num_hidden_layers=layers,
                     num_attention_heads=heads, intermediate_size=ffn, num_labels=labels)
    torch.manual_seed(seed)
    cls = {"teacher": DeiTForImageClassificationWithTeacher, "cls": DeiTForImageClassification, None: DeiTModel}[head]
    model = cls(cfg)
    gen = torch.Generator().manual_seed(1000003 + seed)
    with torch.no_grad():
        for pname, prm in sorted(model.named_parameters()):
            if "layernorm" in pname.lower():
                prm.copy_(_portable_normal(prm.shape, gen) * (0.1 if pname.endswith("weight") else 0.05) + (1.0 if pname.endswith("weight") else 0.0))
            else:                              # matrices, tokens, position table and biases
                prm.copy_(_portable_normal(prm.shape, gen) * 0.02)
    model.eval()
    return model


class TimmLikeDistilledViT(torch.nn.Module):
    """Stand-in with the attribute layout of timm's VisionTransformerDistilled (timm is not installed here): a
    `dist_token` after `cls_token`, a `pos_embed` of G^2 + 2 rows and a `head_dist`; in eval the output is the mean of
    head(x[:, 0]) and head_dist(x[:, 1])."""

    def __init__(self, dim=192, heads=3, hidden=384, depth=2, image=48, patch=8, classes=10, seed=3):
        super().__init__()
        self.patch_embed = _PatchEmbed(dim, patch)
        self.cls_token = torch.nn.Parameter(torch.zeros(1, 1, dim))
        self.dist_token = torch.nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = torch.nn.Parameter(torch.zeros(1, (image // patch) ** 2 + 2, dim))
        self.blocks = torch.nn.ModuleList([_TimmLikeBlock(dim, heads, hidden) for _ in range(depth)])
        self.norm = torch.nn.LayerNorm(dim, eps=1e-6)
        self.head = torch.nn.Linear(dim, classes)
        self.head_dist = torch.nn.Linear(dim, classes)
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            for p in self.parameters():
                if p.dim() >= 2:
                    p.copy_(_portable_normal(p.shape, g) * 0.05)
                elif p.dim() == 1 and p.numel() > 1:
                    p.add_(_portable_normal(p.shape, g) * 0.02)
        self.eval()

    def forward(self, x):
        t = self.patch_embed(x)
        n = t.shape[0]
        t = torch.cat([self.cls_token.expand(n, -1, -1), self.dist_token.expand(n, -1, -1), t], dim=1) + self.pos_embed
        for b in self.blocks:
            t = b(t)
        t = self.norm(t)
        return (self.head(t[:, 0]) + self.head_dist(t[:, 1])) / 2
