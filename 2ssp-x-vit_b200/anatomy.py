"""Model anatomy: which module layouts the drop-in accepts and where their parameters live.

Mirrors the reference's attribute walking (src/vit_pruning.py:28-75 `_get_encoder`, `_gather_mlp_pairs`,
`_get_hidden_and_inter_sizes`): HF `ViTModel` / `ViTForImageClassification`
(`.vit.encoder.layer[i].{attention,intermediate,output}`), HF `DeiTModel` / `DeiTForImageClassification` /
`DeiTForImageClassificationWithTeacher` (`.deit`, the same layer layout; the reference reaches it through
`model.base_model`) and timm-shaped `VisionTransformer` (`.blocks[i].{norm1,attn,norm2,mlp.fc1,mlp.fc2}`), distilled
ones (`dist_token`, `head_dist`) included, and those with LayerScale (`.blocks[i].ls1.gamma`, `.ls2.gamma`), register
tokens (`reg_token`) and class-free position tables (`no_embed_class`): DeiT-III and DINOv2, and those with a pre-norm
(`norm_pre`, timm `pre_norm=True`) and QuickGELU (`blocks[i].mlp.act`): the CLIP image towers.

The reference walks any timm `VisionTransformer`, so every timm-layout module the engine would not compute exactly is
refused here by name (`_refuse_timm_extras`, `_ffn_act`) instead of being run without it. HF `Dinov2*` classes fail the
reference's walk (`layer[i].intermediate`) and fail here the same way.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn


def get_encoder(vit_model):
    if hasattr(vit_model, "vit"):
        base = vit_model.vit
    elif hasattr(vit_model, "base_model"):
        base = vit_model.base_model
    else:
        base = vit_model
    return base.encoder if hasattr(base, "encoder") else base


def get_blocks(vit_model) -> Tuple[str, nn.ModuleList]:
    enc = get_encoder(vit_model)
    if hasattr(enc, "layer"):
        return "hf", enc.layer
    if hasattr(enc, "blocks"):
        return "timm", enc.blocks
    raise AttributeError("Unsupported ViT model structure: expected encoder.layer or blocks")


def gather_mlp_pairs(vit_model) -> List[Tuple[nn.Linear, nn.Linear]]:
    kind, blocks = get_blocks(vit_model)
    if kind == "hf":
        return [(b.intermediate.dense, b.output.dense) for b in blocks]
    return [(b.mlp.fc1, b.mlp.fc2) for b in blocks]


def attention_module(kind: str, block):
    return getattr(block, "attention" if kind == "hf" else "attn", None)


class AttentionBypass(nn.Module):
    """Parameter-free replacement of an attention submodule: returns zeros, so the residual add leaves the
    hidden states unchanged (src/vit_pruning.py:416-429). HF ViTLayer of transformers < 5 indexes the
    attention output with [0]; >= 5 adds it directly, hence `as_tuple`."""

    is_tssp_bypass = True

    def __init__(self, as_tuple: bool):
        super().__init__()
        self.as_tuple = as_tuple

    def forward(self, hidden_states, *args, **kwargs):
        zeros = torch.zeros_like(hidden_states)
        return (zeros,) if self.as_tuple else zeros


def hf_attention_returns_tuple() -> bool:
    try:
        import transformers
        return int(transformers.__version__.split(".")[0]) < 5
    except Exception:
        return True


def has_attention(kind: str, block) -> bool:
    """False if the block's attention has been replaced by a parameter-free bypass (ours or the reference's)."""
    m = attention_module(kind, block)
    if m is None:
        return False
    return any(True for _ in m.parameters())


def install_bypass(vit_model, index: int) -> None:
    kind, blocks = get_blocks(vit_model)
    if kind == "hf" and hasattr(blocks[index], "attention"):
        blocks[index].attention = AttentionBypass(as_tuple=hf_attention_returns_tuple())
    elif kind == "timm" and hasattr(blocks[index], "attn"):
        blocks[index].attn = AttentionBypass(as_tuple=False)


@dataclass
class Anatomy:
    """Everything tssp_create / tssp_load_weights need, as found on the module."""
    kind: str
    n_blocks: int
    hidden: int
    heads: int
    image_size: int
    patch_size: int
    channels: int
    n_classes: int
    head_hidden: int
    ln_eps: float
    ffn_dims: List[int]
    attn_present: List[bool]
    score_point: int                      # 0 post-GELU (HF hook point), 1 pre-GELU (timm hook point)
    prefix_tokens: int = 1                # tokens ahead of the patches: 1 (CLS), 2 (CLS, distillation token: DeiT) or 1 + R
    dist_head: bool = False               # logits = (head(row 0) + dist_head(row 1)) / 2 (globals_ "head_dist_w/_b")
    dist_token: bool = False              # row 1 is a distillation token (globals_ "dist")
    register_tokens: int = 0              # R timm register tokens after CLS (globals_ "reg", [R, D])
    pos_covers_prefix: bool = True        # False: timm no_embed_class, the position table has G^2 rows (patches only)
    layer_scale: bool = False             # blocks carry "ls1" / "ls2" gammas [D] (timm LayerScale)
    pre_norm: bool = False                # LayerNorm over every token before block 0 (globals_ "norm_pre_w" / "norm_pre_b")
    ffn_act: str = "gelu"                 # MLP activation of every block: "gelu" (erf) or "quick_gelu" (x * sigmoid(1.702 x))
    globals_: Dict[str, Optional[torch.Tensor]] = field(default_factory=dict)
    blocks: List[Dict[str, Optional[torch.Tensor]]] = field(default_factory=list)


def _p(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.detach()


def _head(module) -> Tuple[int, int, Optional[torch.Tensor], Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(n_classes, head_hidden, head0_w, head_w, head_b) for nn.Linear or Sequential(Linear, GELU, Linear)."""
    if module is None or isinstance(module, nn.Identity):
        return 0, 0, None, None, None
    if isinstance(module, nn.Linear):
        return module.out_features, 0, None, _p(module.weight), _p(module.bias)
    if isinstance(module, nn.Sequential) and len(module) == 3 and isinstance(module[0], nn.Linear) \
            and isinstance(module[1], nn.GELU) and isinstance(module[2], nn.Linear):
        if module[0].bias is not None:
            raise AttributeError("Sequential head with a biased first Linear is not supported")
        return module[2].out_features, module[0].out_features, _p(module[0].weight), _p(module[2].weight), _p(module[2].bias)
    raise AttributeError(f"Unsupported classification head: {type(module).__name__}")


def _dist_head(main: Tuple, module) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(weight, bias) of a distillation head averaged with the main head `main` (a `_head` tuple), or (None, None)."""
    if module is None or isinstance(module, nn.Identity):
        if main[0] > 0:
            raise AttributeError("a classification head without its distillation head is not supported")
        return None, None
    if main[1] > 0:
        raise AttributeError("a distillation head combined with a Sequential classification head is not supported")
    if not isinstance(module, nn.Linear):
        raise AttributeError(f"Unsupported distillation head: {type(module).__name__}")
    if module.out_features != main[0]:
        raise AttributeError(f"distillation head has {module.out_features} outputs, the classification head {main[0]}")
    return _p(module.weight), _p(module.bias)


def _is_identity(m) -> bool:
    return m is None or isinstance(m, nn.Identity)


def _refuse_timm_extras(root, blocks) -> None:
    """AttributeError naming every timm VisionTransformer feature the engine does not compute: a model that has one is
    refused rather than run without it."""
    if not _is_identity(getattr(root, "fc_norm", None)):
        raise AttributeError(f"fc_norm ({type(root.fc_norm).__name__}) is not supported: only Identity")
    if not _is_identity(getattr(getattr(root, "patch_embed", None), "norm", None)):
        raise AttributeError("patch_embed.norm is not supported: only Identity")
    pool = getattr(root, "global_pool", "token")
    if pool != "token":
        raise AttributeError(f"global_pool={pool!r} is not supported: the classifier reads the CLS token ('token') only")
    if getattr(root, "attn_pool", None) is not None:
        raise AttributeError("attn_pool is not supported: the classifier reads the CLS token only")
    if getattr(root, "cls_token", None) is None:
        raise AttributeError("cls_token is missing: models without a class token are not supported")
    if getattr(root, "dynamic_img_size", False):
        raise AttributeError("dynamic_img_size=True is not supported: the engine runs one fixed image size")
    if getattr(root, "dist_token", None) is not None and getattr(root, "reg_token", None) is not None:
        raise AttributeError("dist_token together with reg_token is not supported")
    for i, b in enumerate(blocks):
        for owner, name in (("attn", "q_norm"), ("attn", "k_norm"), ("attn", "norm"), ("mlp", "norm")):
            m = getattr(getattr(b, owner, None), name, None)
            if not _is_identity(m):
                raise AttributeError(f"blocks[{i}].{owner}.{name} ({type(m).__name__}) is not supported: only Identity")


def _norm_pre(root, hidden: int) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(weight, bias) of timm's `norm_pre` LayerNorm (pre_norm=True: CLIP towers), or (None, None) when it is Identity. A
    non-affine LayerNorm is taken as ones / zeros. The engine carries one LayerNorm eps, that of `norm`."""
    m = getattr(root, "norm_pre", None)
    if _is_identity(m):
        return None, None
    if not isinstance(m, nn.LayerNorm) or tuple(m.normalized_shape) != (hidden,):  # timm's LayerNorm subclasses nn.LayerNorm
        raise AttributeError(f"norm_pre ({type(m).__name__}) is not supported: only Identity or nn.LayerNorm({hidden})")
    if float(m.eps) != float(root.norm.eps):
        raise AttributeError(f"norm_pre.eps={m.eps} differs from norm.eps={root.norm.eps}: the engine applies one LayerNorm eps")
    w = _p(m.weight) if m.weight is not None else torch.ones(hidden)
    b = _p(m.bias) if m.bias is not None else torch.zeros(hidden)
    return w, b


def _act_kind(act) -> Optional[str]:
    """'gelu' (erf), 'quick_gelu', or None for any other module. timm cannot be imported here, so its activation classes
    are matched by name: timm.layers.GELU wraps F.gelu (erf), QuickGELU is x * sigmoid(1.702 x)."""
    if isinstance(act, nn.GELU):
        return "gelu" if act.approximate == "none" else None
    name = type(act).__name__
    return {"GELU": "gelu", "QuickGELU": "quick_gelu"}.get(name)


def ffn_act_signature(vit_model) -> tuple:
    """Per block: the class of `mlp.act` and its `approximate` setting (timm layout; () for HF models, whose activation
    is a config string). Parameter-free, so the parameter signature of a cached engine does not see a swapped module."""
    try:
        kind, blocks = get_blocks(vit_model)
    except AttributeError:
        return ()
    if kind != "timm":
        return ()
    acts = [getattr(getattr(b, "mlp", None), "act", None) for b in blocks]
    return tuple((type(a), getattr(a, "approximate", None)) for a in acts)


def _ffn_act(blocks) -> str:
    """The one MLP activation of every block: AttributeError naming the block for any other module or a mix of kinds."""
    kinds = []
    for i, b in enumerate(blocks):
        act = getattr(b.mlp, "act", None)
        kind = _act_kind(act)
        if kind is None:
            what = type(act).__name__ + (f", approximate={act.approximate!r}" if isinstance(act, nn.GELU) else "")
            raise AttributeError(f"blocks[{i}].mlp.act ({what}) is not supported: only erf GELU or QuickGELU")
        if kinds and kind != kinds[0]:
            raise AttributeError(f"blocks[{i}].mlp.act ({type(act).__name__}) differs from blocks[0].mlp.act "
                                 f"({type(blocks[0].mlp.act).__name__}): every block must use the same activation")
        kinds.append(kind)
    return kinds[0]


def _layer_scale(block, name: str, index: int) -> Optional[torch.Tensor]:
    """gamma of timm's LayerScale `block.<name>` (x * gamma), or None when the module is Identity / absent."""
    m = getattr(block, name, None)
    if _is_identity(m):
        return None
    gamma = getattr(m, "gamma", None)
    if not isinstance(gamma, torch.Tensor):
        raise AttributeError(f"blocks[{index}].{name} ({type(m).__name__}) has no gamma: only timm LayerScale is supported")
    return _p(gamma).reshape(-1)


def _hf_root(vit_model):
    for name in ("vit", "deit"):
        if hasattr(vit_model, name):
            return getattr(vit_model, name)
    return vit_model


def describe(vit_model) -> Anatomy:
    kind, blocks = get_blocks(vit_model)
    pairs = gather_mlp_pairs(vit_model)
    hidden = pairs[0][0].weight.size(1)
    prefix = 1
    hdw = hdb = None
    dist = False
    n_reg, pos_covers_prefix, layer_scale = 0, True, False
    ffn_act = "gelu"
    if kind == "hf":
        vit = _hf_root(vit_model)
        emb = vit.embeddings
        conv = emb.patch_embeddings.projection
        final_ln = vit.layernorm
        if getattr(emb, "distillation_token", None) is not None:  # DeiTEmbeddings: [CLS, distillation, patches]
            prefix = 2
        if hasattr(vit_model, "cls_classifier"):                  # DeiTForImageClassificationWithTeacher: averaged heads
            head = _head(vit_model.cls_classifier)
            hdw, hdb = _dist_head(head, getattr(vit_model, "distillation_classifier", None))
            dist = hdw is not None
        else:
            head = _head(getattr(vit_model, "classifier", None))
        n_classes, head_hidden, h0, hw, hb = head
        cfg = vit_model.config
        heads = int(cfg.num_attention_heads)
        act = getattr(cfg, "hidden_act", "gelu")
        if act != "gelu":
            raise AttributeError(f"hidden_act={act!r} unsupported (erf GELU only)")
        g = {
            "patch_w": _p(conv.weight), "patch_b": _p(conv.bias), "cls": _p(emb.cls_token), "pos": _p(emb.position_embeddings),
            "final_ln_w": _p(final_ln.weight), "final_ln_b": _p(final_ln.bias), "head0_w": h0, "head_w": hw, "head_b": hb,
            "dist": _p(getattr(emb, "distillation_token", None)), "head_dist_w": hdw, "head_dist_b": hdb,
        }
        blks = []
        for b in blocks:
            present = has_attention(kind, b)
            d: Dict[str, Optional[torch.Tensor]] = {
                "ln2_w": _p(b.layernorm_after.weight), "ln2_b": _p(b.layernorm_after.bias),
                "fc1_w": _p(b.intermediate.dense.weight), "fc1_b": _p(b.intermediate.dense.bias),
                "fc2_w": _p(b.output.dense.weight), "fc2_b": _p(b.output.dense.bias),
            }
            if present:
                sa = b.attention.attention
                d.update({
                    "ln1_w": _p(b.layernorm_before.weight), "ln1_b": _p(b.layernorm_before.bias),
                    "q_w": _p(sa.query.weight), "q_b": _p(sa.query.bias), "k_w": _p(sa.key.weight), "k_b": _p(sa.key.bias),
                    "v_w": _p(sa.value.weight), "v_b": _p(sa.value.bias),
                    "proj_w": _p(b.attention.output.dense.weight), "proj_b": _p(b.attention.output.dense.bias),
                })
            blks.append(d)
        eps = float(final_ln.eps)
        score_point = 0
    else:
        root = vit_model
        _refuse_timm_extras(root, blocks)
        ffn_act = _ffn_act(blocks)
        npw, npb = _norm_pre(root, hidden)
        conv = root.patch_embed.proj
        final_ln = root.norm
        head = _head(getattr(root, "head", None))
        if getattr(root, "dist_token", None) is not None:  # timm VisionTransformerDistilled: eval output averages both heads
            prefix = 2
            hdw, hdb = _dist_head(head, getattr(root, "head_dist", None))
            dist = hdw is not None
        reg = getattr(root, "reg_token", None)
        if reg is not None:  # timm _pos_embed: [CLS, reg_token rows, patches]
            n_reg = int(reg.shape[1])
            prefix += n_reg
        pos_covers_prefix = not bool(getattr(root, "no_embed_class", False))
        n_classes, head_hidden, h0, hw, hb = head
        first_attn = next((b.attn for b in blocks if has_attention(kind, b)), None)
        heads = int(first_attn.num_heads) if first_attn is not None else hidden // 64
        g = {
            "patch_w": _p(conv.weight), "patch_b": _p(conv.bias), "cls": _p(root.cls_token), "pos": _p(root.pos_embed),
            "final_ln_w": _p(final_ln.weight), "final_ln_b": _p(final_ln.bias), "head0_w": h0, "head_w": hw, "head_b": hb,
            "dist": _p(getattr(root, "dist_token", None)), "head_dist_w": hdw, "head_dist_b": hdb,
            "reg": None if reg is None else _p(reg).reshape(n_reg, hidden),
            "norm_pre_w": npw, "norm_pre_b": npb,
        }
        gammas = [(_layer_scale(b, "ls1", i), _layer_scale(b, "ls2", i)) for i, b in enumerate(blocks)]
        layer_scale = any(g is not None for pair in gammas for g in pair)
        blks = []
        for b, (ls1, ls2) in zip(blocks, gammas):
            present = has_attention(kind, b)
            d = {
                "ln2_w": _p(b.norm2.weight), "ln2_b": _p(b.norm2.bias),
                "fc1_w": _p(b.mlp.fc1.weight), "fc1_b": _p(b.mlp.fc1.bias),
                "fc2_w": _p(b.mlp.fc2.weight), "fc2_b": _p(b.mlp.fc2.bias),
            }
            if present:
                qkv_w, qkv_b = _p(b.attn.qkv.weight), _p(b.attn.qkv.bias)
                D = hidden
                d.update({
                    "ln1_w": _p(b.norm1.weight), "ln1_b": _p(b.norm1.bias),
                    "q_w": qkv_w[0:D], "k_w": qkv_w[D:2 * D], "v_w": qkv_w[2 * D:3 * D],
                    "q_b": None if qkv_b is None else qkv_b[0:D], "k_b": None if qkv_b is None else qkv_b[D:2 * D],
                    "v_b": None if qkv_b is None else qkv_b[2 * D:3 * D],
                    "proj_w": _p(b.attn.proj.weight), "proj_b": _p(b.attn.proj.bias),
                })
            if layer_scale:  # a block without its own LayerScale scales by exactly 1
                d["ls1"] = (ls1 if ls1 is not None else torch.ones(hidden)) if present else None
                d["ls2"] = ls2 if ls2 is not None else torch.ones(hidden)
            blks.append(d)
        eps = float(final_ln.eps)
        score_point = 1
    dist_tok = g.get("dist") is not None
    pw = g["patch_w"]
    channels, patch = int(pw.shape[1]), int(pw.shape[2])
    n_tokens = int(g["pos"].reshape(-1, hidden).shape[0])
    covered = prefix if pos_covers_prefix else 0  # no_embed_class: the table holds the patches' rows only
    grid = int(round(max(0, n_tokens - covered) ** 0.5))
    if grid * grid + covered != n_tokens:
        what = "CLS" if prefix == 1 else ("CLS and distillation token" if dist_tok else f"CLS and {n_reg} register tokens")
        if not pos_covers_prefix:
            what = f"nothing (no_embed_class; {what} get no position)"
        raise AttributeError(f"position table with {n_tokens} rows fits neither layout: not a square grid plus {what} "
                             f"({prefix} prefix token{'s' if prefix > 1 else ''})")
    return Anatomy(
        kind=kind, n_blocks=len(blocks), hidden=int(hidden), heads=heads, image_size=grid * patch, patch_size=patch,
        channels=channels, n_classes=int(n_classes), head_hidden=int(head_hidden), ln_eps=eps,
        ffn_dims=[int(p[0].weight.size(0)) for p in pairs], attn_present=[has_attention(kind, b) for b in blocks],
        score_point=score_point, prefix_tokens=prefix, dist_head=dist, dist_token=dist_tok, register_tokens=n_reg,
        pos_covers_prefix=pos_covers_prefix, layer_scale=layer_scale, pre_norm=g.get("norm_pre_w") is not None,
        ffn_act=ffn_act, globals_=g, blocks=blks,
    )
