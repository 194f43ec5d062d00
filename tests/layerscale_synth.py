"""Seeded timm-shaped LayerScale ViTs (DeiT-III, DINOv2 with and without register tokens) for the LayerScale tests and
tools/layerscale_bench.py (TEST / MEASUREMENT INFRASTRUCTURE).

timm is not installed here, so `TimmLikeLayerScaleViT` restates the parts of timm's `VisionTransformer` the engine
reads, with timm's attribute names: `blocks[i].ls1.gamma` / `.ls2.gamma` (timm `LayerScale`: x * gamma, applied to the
attention output after `proj` and to the MLP output after `fc2`, before the residual add), `reg_token` [1, R, D] after
`cls_token`, `no_embed_class`, `global_pool = 'token'` and `num_prefix_tokens`. Values are portable (bit-identical on
every CPU, see oracle.synth._portable_normal). Kept next to the tests so that oracle/ and its golden vectors stay as
they are.
"""
from __future__ import annotations

import torch

from oracle.synth import _PatchEmbed, _portable_normal, _TimmLikeBlock

LS_SHAPES = {
    # name: (image, patch, dim, depth, heads, hidden, classes, reg_tokens, no_embed_class)
    "tiny_reg4": (84, 14, 128, 3, 2, 256, 10, 4, True),      # T = 36 + 1 + 4 = 41, DINOv2-reg layout at test size
    "tiny_p14": (84, 14, 128, 3, 2, 256, 10, 0, False),      # T = 37, DINOv2 layout at test size
    "deit3_tiny": (48, 8, 192, 3, 3, 768, 10, 0, True),      # T = 37, DeiT-III layout at the DeiT-Ti width
    "deit3_small": (224, 16, 384, 12, 6, 1536, 1000, 0, True),
    "deit3_base": (224, 16, 768, 12, 12, 3072, 1000, 0, True),   # T = 197
    "dinov2_small": (224, 14, 384, 12, 6, 1536, 1000, 0, False),  # T = 257
    "dinov2_base": (224, 14, 768, 12, 12, 3072, 1000, 0, False),
    "dinov2_small_reg4": (224, 14, 384, 12, 6, 1536, 1000, 4, True),  # T = 261
    "dinov2_base_reg4": (224, 14, 768, 12, 12, 3072, 1000, 4, True),
}


class LayerScale(torch.nn.Module):
    """timm.layers.LayerScale: x * gamma."""

    def __init__(self, dim, init_values):
        super().__init__()
        self.gamma = torch.nn.Parameter(init_values * torch.ones(dim))

    def forward(self, x):
        return x * self.gamma


class LayerScaleBlock(_TimmLikeBlock):
    """timm Block with LayerScale: x = x + ls1(attn(norm1(x))); x = x + ls2(mlp(norm2(x)))."""

    def __init__(self, dim, heads, hidden, init_values):
        super().__init__(dim, heads, hidden)
        self.ls1 = LayerScale(dim, init_values) if init_values is not None else torch.nn.Identity()
        self.ls2 = LayerScale(dim, init_values) if init_values is not None else torch.nn.Identity()

    def forward(self, x):
        x = x + self.ls1(self.attn(self.norm1(x)))
        return x + self.ls2(self.mlp(self.norm2(x)))


class TimmLikeLayerScaleViT(torch.nn.Module):
    """classes = 0: no head (`head = Identity`, the DINOv2 backbone as published); the forward then returns the
    normalised CLS features. init_values = None: no LayerScale (`ls1` / `ls2` are Identity)."""

    def __init__(self, dim=128, heads=2, hidden=256, depth=3, image=84, patch=14, classes=10, reg_tokens=0,
                 no_embed_class=False, init_values=0.5, seed=3):
        super().__init__()
        self.patch_embed = _PatchEmbed(dim, patch)
        self.cls_token = torch.nn.Parameter(torch.zeros(1, 1, dim))
        self.reg_token = torch.nn.Parameter(torch.zeros(1, reg_tokens, dim)) if reg_tokens else None
        self.no_embed_class = no_embed_class
        self.num_prefix_tokens = 1 + reg_tokens
        self.global_pool = "token"
        grid = (image // patch) ** 2
        self.pos_embed = torch.nn.Parameter(torch.zeros(1, grid + (0 if no_embed_class else self.num_prefix_tokens), dim))
        self.blocks = torch.nn.ModuleList([LayerScaleBlock(dim, heads, hidden, init_values) for _ in range(depth)])
        self.norm = torch.nn.LayerNorm(dim, eps=1e-6)
        self.head = torch.nn.Linear(dim, classes) if classes > 0 else torch.nn.Identity()
        g = torch.Generator().manual_seed(seed)
        # matrices: 0.05 at the test width 128, scaled by 1 / sqrt(dim) so that every width keeps the activation scale of
        # the test models (0.0204 at 768, about timm's init std of 0.02); a fixed 0.05 at 768 lets the residual stream and
        # the logits grow with depth far beyond those of a trained model
        w_std = 0.05 * (128 / dim) ** 0.5
        with torch.no_grad():
            for name, p in self.named_parameters():
                if name.endswith("gamma"):   # around 0.5 rather than timm's 1e-5, so that the scaled branches matter
                    p.copy_(0.5 + _portable_normal(p.shape, g) * 0.1)
                elif p.dim() >= 2:
                    p.copy_(_portable_normal(p.shape, g) * w_std)
                elif p.dim() == 1 and p.numel() > 1:
                    p.add_(_portable_normal(p.shape, g) * 0.02)
        self.eval()

    def _pos_embed(self, x):
        # timm VisionTransformer._pos_embed (dynamic_img_size=False): without no_embed_class the table covers the prefix
        # tokens and is added after they are concatenated; with it, it covers the patches only and is added before
        n = x.shape[0]
        prefix = [self.cls_token.expand(n, -1, -1)]
        if self.reg_token is not None:
            prefix.append(self.reg_token.expand(n, -1, -1))
        if self.no_embed_class:
            return torch.cat(prefix + [x + self.pos_embed], dim=1)
        return torch.cat(prefix + [x], dim=1) + self.pos_embed

    def forward(self, x):
        t = self._pos_embed(self.patch_embed(x))
        for b in self.blocks:
            t = b(t)
        return self.head(self.norm(t)[:, 0])


def make_ls(name: str, seed: int = 3, classes: int | None = None, init_values: float | None = 0.5) -> TimmLikeLayerScaleViT:
    image, patch, dim, depth, heads, hidden, n_cls, reg, nec = LS_SHAPES[name]
    return TimmLikeLayerScaleViT(dim, heads, hidden, depth, image, patch, n_cls if classes is None else classes, reg, nec,
                                 init_values, seed)


def image_size(name: str) -> int:
    return LS_SHAPES[name][0]
