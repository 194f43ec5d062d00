"""LayerScale ViTs (timm DeiT-III and DINOv2: ls1 / ls2 gammas, patch 14, register tokens, class-free position tables)
through the engine and the drop-in API. GPU tests are marked `gpu`; the anatomy, refusal, configuration and planner
checks at the top run without one.

Parity is against the stand-in's own fp32 forward and the oracle's functions, which run on it unchanged (timm hook point:
`mlp.fc1`, pre-GELU). Tolerances are those of tests/test_gpu_parity.py.
"""
import copy
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import synth
from oracle import twossp_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import layerscale_synth as LS  # noqa: E402

SCORE_RTOL = 1e-2
LOGIT_MAX_ABS = 3e-2
LOGIT_MEAN_ABS = 5e-3
DELTA = 2


def _rel(got, want):
    return max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, want))


@torch.no_grad()
def _fp32_logits(model, px, batch=16):
    model = copy.deepcopy(model).float().cpu().eval()
    return torch.cat([model(px[s:s + batch]).float() for s in range(0, px.shape[0], batch)])


# ----------------------------------------------------------------------------------------------- no GPU needed
@pytest.mark.parametrize("name,T", [("tiny_reg4", 41), ("tiny_p14", 37), ("deit3_tiny", 37), ("deit3_base", 197),
                                    ("dinov2_small", 257), ("dinov2_base", 257), ("dinov2_small_reg4", 261),
                                    ("dinov2_base_reg4", 261)])
def test_anatomy_of_layerscale_layouts(name, T):
    from twossp_b200.anatomy import describe
    image, patch, dim, depth, heads, hidden, classes, reg, nec = LS.LS_SHAPES[name]
    a = describe(LS.make_ls(name))
    assert (a.kind, a.hidden, a.heads, a.image_size, a.patch_size, a.n_blocks, a.score_point) == \
        ("timm", dim, heads, image, patch, depth, 1)
    assert (a.prefix_tokens, a.register_tokens, a.dist_token, a.dist_head) == (1 + reg, reg, False, False)
    assert a.pos_covers_prefix == (not nec) and a.layer_scale
    assert (image // patch) ** 2 + a.prefix_tokens == T
    assert all(b["ls1"].shape == (dim,) and b["ls2"].shape == (dim,) for b in a.blocks)
    assert (a.globals_["reg"] is None) == (reg == 0)


def test_anatomy_without_layerscale_and_headless():
    from twossp_b200.anatomy import describe
    a = describe(LS.make_ls("tiny_reg4", init_values=None))
    assert not a.layer_scale and "ls1" not in a.blocks[0] and a.register_tokens == 4
    a = describe(LS.make_ls("dinov2_small", classes=0))
    assert a.n_classes == 0 and a.layer_scale


def _refusal(mutate, match):
    from twossp_b200.anatomy import describe
    m = LS.make_ls("tiny_reg4")
    mutate(m)
    with pytest.raises(AttributeError, match=match):
        describe(m)


@pytest.mark.parametrize("what,mutate,match", [
    ("norm_pre", lambda m: setattr(m, "norm_pre", torch.nn.LayerNorm(128)), "norm_pre"),
    ("fc_norm", lambda m: setattr(m, "fc_norm", torch.nn.LayerNorm(128)), "fc_norm"),
    ("q_norm", lambda m: setattr(m.blocks[1].attn, "q_norm", torch.nn.LayerNorm(64)), r"blocks\[1\]\.attn\.q_norm"),
    ("k_norm", lambda m: setattr(m.blocks[0].attn, "k_norm", torch.nn.LayerNorm(64)), r"blocks\[0\]\.attn\.k_norm"),
    ("attn_norm", lambda m: setattr(m.blocks[2].attn, "norm", torch.nn.LayerNorm(128)), r"blocks\[2\]\.attn\.norm"),
    ("mlp_norm", lambda m: setattr(m.blocks[0].mlp, "norm", torch.nn.LayerNorm(256)), r"blocks\[0\]\.mlp\.norm"),
    ("global_pool", lambda m: setattr(m, "global_pool", "avg"), "global_pool"),
    ("attn_pool", lambda m: setattr(m, "attn_pool", torch.nn.Linear(128, 128)), "attn_pool"),
    ("cls_token", lambda m: setattr(m, "cls_token", None), "cls_token"),
    ("dynamic_img_size", lambda m: setattr(m, "dynamic_img_size", True), "dynamic_img_size"),
    ("dist_and_reg", lambda m: setattr(m, "dist_token", torch.nn.Parameter(torch.zeros(1, 1, 128))), "dist_token together with reg_token"),
    ("not_layerscale", lambda m: setattr(m.blocks[0], "ls1", torch.nn.Dropout()), r"blocks\[0\]\.ls1"),
    ("pos_rows", lambda m: setattr(m, "pos_embed", torch.nn.Parameter(torch.zeros(1, 41, 128))), "fits neither layout"),
])
def test_refusals_name_the_attribute(what, mutate, match):
    _refusal(mutate, match)


def test_hf_dinov2_is_outside_the_walk():
    transformers = pytest.importorskip("transformers")
    if not hasattr(transformers, "Dinov2Model"):
        pytest.skip("transformers has no Dinov2Model")
    from twossp_b200.anatomy import describe
    cfg = transformers.Dinov2Config(hidden_size=128, num_hidden_layers=1, num_attention_heads=2, intermediate_size=256,
                                    image_size=56, patch_size=14)
    with pytest.raises(AttributeError):
        describe(transformers.Dinov2Model(cfg))   # layer[i] has no .intermediate: the reference's walk fails the same way


def _config(L, hidden=128, image=84, patch=14):
    cfg = L.TsspConfig()
    cfg.n_blocks, cfg.hidden, cfg.heads = 2, hidden, hidden // 64
    cfg.image_size, cfg.patch_size, cfg.channels = image, patch, 3
    cfg.n_classes, cfg.head_hidden, cfg.max_images = 10, 0, 4
    cfg.score_point, cfg.cache_blocks, cfg.ln_eps = 1, 0, 1e-6
    for i in range(2):
        cfg.ffn_dims[i] = 256
        cfg.attn_present[i] = 1
    return cfg


def test_create_layout_validates_before_touching_a_device():
    import __graft_entry__ as g
    g.build()
    from twossp_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()

    def err(cfg, *layout):   # (dist_token, register_tokens, pos_patches_only, layer_scale)
        cfg.dist_token, cfg.register_tokens, cfg.pos_patches_only, cfg.layer_scale = layout
        assert lib.tssp_create(C.byref(cfg), 4096, C.byref(h)) != 0   # device 4096 exists nowhere
        return lib.tssp_last_error().decode()

    msg = err(_config(L), 0, 8, 1, 1)
    assert "register_tokens=8" in msg and "[0,7]" in msg, msg
    msg = err(_config(L), 1, 4, 1, 1)
    assert "distillation token and register tokens" in msg, msg
    msg = err(_config(L, hidden=768, image=518, patch=14), 0, 0, 0, 1)   # DINOv2 at its native size
    assert "T=1370" in msg and "[32,1025]" in msg, msg
    msg = err(_config(L, hidden=768, image=518, patch=14), 0, 4, 1, 1)   # ... with four registers
    assert "T=1374" in msg and "[32,1025]" in msg, msg
    # valid layouts pass validation and fail on the device: patch 14 (K = 588), T = 41 / 257 / 261, patch 8 with LayerScale
    for layout, image, patch in (((0, 4, 1, 1), 84, 14), ((0, 0, 0, 1), 224, 14), ((0, 4, 1, 1), 224, 14), ((0, 0, 1, 1), 48, 8)):
        msg = err(_config(L, image=image, patch=patch), *layout)
        assert "device" in msg.lower() and "config" not in msg and "layout" not in msg, msg


@pytest.fixture(scope="module")
def ls_planner_models():
    return {name: LS.make_ls(name) for name in ("deit3_small", "deit3_base", "dinov2_small", "dinov2_base")}


@pytest.mark.parametrize("name", ["deit3_small", "deit3_base", "dinov2_small", "dinov2_base"])
@pytest.mark.parametrize("target", [0.25, 0.375, 0.5])
def test_planner_matches_oracle_on_layerscale_models(ls_planner_models, name, target):
    from twossp_b200 import api
    m = ls_planner_models[name]
    got = api.plan_2ssp_allocation(m, target)
    want = O.plan(m, target)
    assert (got.blocks_to_prune, got.per_block_neurons_to_prune, got.estimated_total_removed_params, got.est_error_params) == \
        (want.blocks_to_prune, want.per_block_neurons_to_prune, want.estimated_total_removed_params, want.est_error_params)
    assert got.stage2_fraction == want.stage2_fraction


# ----------------------------------------------------------------------------------------------- GPU fixtures
@pytest.fixture(scope="module")
def cuda_ready():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    torch.cuda.set_device(0)


@pytest.fixture(scope="module")
def lib(cuda_ready):
    from twossp_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ops(cuda_ready):
    from twossp_b200 import ops as o
    return o


@pytest.fixture(scope="module")
def api(cuda_ready):
    from twossp_b200 import api as a
    return a


@pytest.fixture(params=[1, 2], ids=["cta1", "pair"])
def gemm_form(request, lib):
    lib.check(lib.load().tssp_set_gemm_form(request.param))
    yield request.param
    lib.check(lib.load().tssp_set_gemm_form(0))


TINY = ("tiny_reg4", "tiny_p14", "deit3_tiny")


@pytest.fixture(scope="module", params=TINY)
def tiny(request):
    """(name, model on CPU, 24 pixels, fp32 logits of the module, self-labels)"""
    model = LS.make_ls(request.param)
    px = synth.make_pixels(24, LS.image_size(request.param), seed=1234)
    logits = _fp32_logits(model, px)
    return request.param, model, px, logits, logits.argmax(-1)


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("prefix", [1, 5])
@pytest.mark.parametrize("n,H,P", [(2, 84, 14), (3, 224, 14), (2, 45, 5)])
def test_im2col_patch14_is_bit_exact_and_zero_padded(ops, prefix, n, H, P):
    px = torch.randn(n, 3, H, H, device="cuda")
    G, K = H // P, 3 * P * P
    Kp = (K + 7) // 8 * 8
    out = ops.im2col(px, P, prefix=prefix)
    assert out.shape == (n * (G * G + prefix), Kp)
    ref = torch.nn.functional.unfold(px, P, stride=P).transpose(1, 2)            # [n, G^2, C*P*P] in (c, ky, kx) order
    ref = torch.cat([torch.zeros(n, prefix, K, device="cuda"), ref], dim=1).bfloat16().reshape(-1, K)
    assert torch.equal(out[:, :K].view(torch.int16), ref.view(torch.int16))
    assert not out[:, K:].view(torch.int16).any()


@pytest.mark.gpu
@pytest.mark.parametrize("M", [261 * 16, 41 * 9])
def test_patch_gemm_at_k592_matches_torch(ops, lib, gemm_form, M):
    # the patch-embedding GEMM of P = 14: K = 588 padded to 592, ten 64-deep k-slabs with TMA zero fill past 592
    K, Kp, N = 588, 592, 384
    g = torch.Generator().manual_seed(M)
    a = torch.zeros(M, Kp, dtype=torch.bfloat16)
    a[:, :K] = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    w = torch.zeros(N, Kp, dtype=torch.bfloat16)
    w[:, :K] = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    base = torch.randn(M, N, generator=g)
    out = base.clone().cuda()
    ops.gemm(lib.EPI_F32, a.cuda(), w.cuda(), out, None, reduce_add=True)
    ref = a.double() @ w.double().t() + base.double()
    assert (out.cpu().double() - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", [(257 * 16, 768, 768), (257 * 16, 768, 3072), (261 * 9, 384, 384), (41 * 9, 128, 256),
                                   (37 * 5, 192, 768)])
@pytest.mark.parametrize("reduce_add", [False, True])
def test_gemm_scaled_epilogue_matches_torch(ops, lib, gemm_form, M, N, K, reduce_add):
    # proj / fc2 of LayerScale blocks: x (+)= gamma * (a w^T + b), every fp32 tile width (256, 192 at N = 384 / 192,
    # 128 at N = 128) and rows that are not a multiple of 128
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    gamma = (0.5 + torch.randn(N, generator=g) * 0.1).cuda()
    base = torch.randn(M, N, generator=g).cuda()
    out = base.clone() if reduce_add else torch.full((M, N), float("nan"), device="cuda")
    ops.gemm_scaled(a, w, out, bias, gamma, reduce_add=reduce_add)
    ref = gamma.double() * (a.double() @ w.double().t() + bias.double()) + (base.double() if reduce_add else 0)
    assert torch.isfinite(out).all()
    assert (out.double() - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())
    # the same accumulator through the unscaled epilogue, then gamma * (.) in fp32: the scaled one's bits
    plain = torch.full((M, N), float("nan"), device="cuda")
    ops.gemm(lib.EPI_F32, a, w, plain, bias)
    want = gamma * plain + (base if reduce_add else 0)
    assert torch.equal(out, want)


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,heads", [(4, 257, 6), (3, 261, 12), (2, 261, 6), (5, 41, 2), (5, 37, 3)])
def test_attention_at_layerscale_shapes(ops, n, T, heads):
    D = heads * 64
    g = torch.Generator(device="cuda").manual_seed(T * 7 + heads)
    qkv = torch.randn(n * T, 3 * D, device="cuda", generator=g).bfloat16()
    ctx = ops.attention(qkv, n, T, heads)
    q, k, v = qkv.float().view(n, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(n * T, D)
    assert torch.isfinite(ctx.float()).all()
    assert ((ctx.float() - ref).abs() <= ref.abs() * 2 ** -7 + 6e-3).all()


# ----------------------------------------------------------------------------------------------- exactness
def _bits(api, model, px, labels):
    """(score sums, logits, Stage-2 counts) of the engine on `model` (moved to the GPU)."""
    gm = copy.deepcopy(model).cuda()
    batches = [{"pixel_values": px[:12], "labels": labels[:12]}, {"pixel_values": px[12:], "labels": labels[12:]}]
    scores = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    logits = api.engine_for(gm, "cuda", batch_hint=24).logits(px).cpu()
    counts = api.attention_removal_counts(gm, batches, "cuda", None)
    api.release_engine(gm)
    return scores, logits, counts


def _same(x, y):
    assert all(torch.equal(a, b) for a, b in zip(x[0], y[0]))
    assert torch.equal(x[1], y[1]) and x[2] == y[2]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_reg4", "deit3_tiny"])
def test_unit_gammas_give_the_bits_of_the_model_without_layerscale(api, name):
    ls = LS.make_ls(name)
    with torch.no_grad():
        for b in ls.blocks:
            b.ls1.gamma.fill_(1.0)
            b.ls2.gamma.fill_(1.0)
    plain = copy.deepcopy(ls)
    for b in plain.blocks:
        b.ls1, b.ls2 = torch.nn.Identity(), torch.nn.Identity()
    px = synth.make_pixels(24, LS.image_size(name), seed=7)
    labels = _fp32_logits(plain, px).argmax(-1)
    _same(_bits(api, ls, px, labels), _bits(api, plain, px, labels))


@pytest.mark.gpu
def test_class_free_position_table_gives_the_bits_of_the_embedded_one(api):
    # the reg4 layout with a table over all 41 rows, and the same model rewritten as no_embed_class:
    # tokens' = tokens + pos[:5], pos' = pos[5:]
    full = LS.TimmLikeLayerScaleViT(reg_tokens=4, no_embed_class=False, seed=5)
    free = LS.TimmLikeLayerScaleViT(reg_tokens=4, no_embed_class=True, seed=5)
    free.load_state_dict({k: v for k, v in full.state_dict().items() if k not in ("pos_embed", "cls_token", "reg_token")}, strict=False)
    with torch.no_grad():
        free.cls_token.copy_(full.cls_token + full.pos_embed[:, :1])
        free.reg_token.copy_(full.reg_token + full.pos_embed[:, 1:5])
        free.pos_embed.copy_(full.pos_embed[:, 5:])
    px = synth.make_pixels(24, 84, seed=8)
    labels = _fp32_logits(full, px).argmax(-1)
    _same(_bits(api, free, px, labels), _bits(api, full, px, labels))


# ----------------------------------------------------------------------------------------------- tiny stand-ins
@pytest.mark.gpu
def test_tiny_logits_scores_and_stage2_counts(api, tiny):
    name, model, px, ref, labels = tiny
    gm = copy.deepcopy(model).cuda()
    logits = api.engine_for(gm, "cuda", batch_hint=24).logits(px).cpu()
    err = (logits - ref).abs()
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (name, err.max().item(), err.mean().item())
    batches = [{"pixel_values": px[:12], "labels": labels[:12]}, {"pixel_values": px[12:], "labels": labels[12:]}]
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    want = O.s1_scores(model, batches, "cpu", None, autocast=False)
    assert _rel(got, want) <= SCORE_RTOL
    base, cand, total = api.attention_removal_counts(gm, batches, "cuda", None)
    rb, rc, rt = O.s2_candidate_scores(model, batches, "cpu", None, autocast=False)
    tol = max(DELTA, int(0.01 * total))
    assert total == rt == 24 and abs(base - rb) <= tol and all(abs(a - b) <= tol for a, b in zip(cand, rc)), (base, cand, rb, rc)
    api.release_engine(gm)


@pytest.mark.gpu
def test_headless_backbone_scores(api):
    model = LS.make_ls("tiny_reg4", classes=0)
    px = synth.make_pixels(16, 84, seed=3)
    batches = [{"pixel_values": px[:8]}, {"pixel_values": px[8:]}]
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert _rel(got, O.s1_scores(model, batches, "cpu", None, autocast=False)) <= SCORE_RTOL
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_captured_chains_equal_eager_launches(api, lib, tiny):
    name, model, px, _, labels = tiny
    out = {}
    for graphs in (0, 1):
        lib.check(lib.load().tssp_set_graphs(graphs))
        try:
            out[graphs] = _bits(api, model, px, labels)
        finally:
            lib.check(lib.load().tssp_set_graphs(1))
    _same(out[0], out[1])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_reg4", "tiny_p14"])
def test_tiny_first_host_batch_split_gives_the_same_bits(api, lib, name):
    # T = 41 / 37 (odd): gcd(T, 32) = 1, so the parts are multiples of 32 images and keep their 32-row sub-tile offsets
    n = 160
    model = LS.make_ls(name).cuda()
    px = synth.make_pixels(n, 84, seed=11)
    eng = api.engine_for(model, "cuda", batch_hint=n)
    out = {}
    for where in ("device", "host"):
        eng.s1_reset()
        src = px.cuda() if where == "device" else px.pin_memory()
        norms = torch.zeros(n, sum(eng.ffn_dims), device="cuda")
        eng.s1_batch(src, img_norms=norms)
        eng.s1_batch(src[: n // 2])
        out[where] = (norms.cpu(), eng.s1_score_sums().clone())
    assert float(out["device"][0].abs().min()) > 0
    assert torch.equal(out["device"][0], out["host"][0]) and torch.equal(out["device"][1], out["host"][1])
    api.release_engine(model)


@pytest.mark.gpu
def test_tiny_fit_and_both_prune_functions(api, tiny, capsys):
    name, model, px, _, labels = tiny
    batches = synth.make_batches(px, labels, 8)
    gm = copy.deepcopy(model).cuda()
    width = gm.blocks[0].mlp.fc1.out_features
    att, mlp = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None).fit()
    separate = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert all(torch.equal(a, b) for a, b in zip(mlp, separate))
    ref_scores = O.s1_scores(model, batches, "cpu", None, autocast=False)
    assert _rel(mlp, ref_scores) <= SCORE_RTOL
    t = width // 2 - 3   # leaves an odd width
    res = api.prune_vit_mlp_width(gm, strategy="act_l2", dataloader=batches, device="cuda", batch_limit=None,
                                  n_to_prune_per_block=[t] * 3, collect_masks=True, min_remaining=8)
    got = np.asarray(res["ffn_prune_masks"], dtype=np.uint8)
    listed = []
    for b, rs in enumerate(ref_scores):
        rs = rs.numpy()
        want = np.zeros_like(got[b])
        want[np.argsort(rs, kind="stable")[:t]] = 1
        cut = np.sort(rs)[t - 1: t + 1].mean()
        for j in np.nonzero(got[b] != want)[0]:
            gap = abs(rs[j] - cut) / cut
            listed.append((b, int(j), float(gap)))
            assert gap <= SCORE_RTOL, f"block {b} neuron {j} flipped with relative gap {gap:.3e} to the cut"
    with capsys.disabled():
        print(f"\n[{name}] mask disagreements vs oracle (block, neuron, rel. gap to cut): {len(listed)} of {got.size}: {listed}")
    assert [fc1.out_features for fc1, _ in api._gather_mlp_pairs(gm)] == [width - t] * 3
    res = api.prune_vit_attention_blocks(gm, 0.0, dataloader=batches, device="cuda", batch_limit=None, importance_mode="copy",
                                         show_progress=False, num_to_prune=1)
    assert len(res["pruned_indices"]) == 1 and res["final_metrics"] is not None
    # the mutated module (odd widths, a bypassed attention whose ls1 now scales zeros) against the engine
    el = api.engine_for(gm, "cuda", batch_hint=8).logits(px).cpu()
    err = (el - _fp32_logits(gm, px)).abs()
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (err.max().item(), err.mean().item())
    api.release_engine(gm)


# ----------------------------------------------------------------------------------------------- full size
@pytest.fixture
def fp32_cuda_reference():
    """The module's own forward on the GPU in true fp32 (no TF32 in the patch convolution or the matmuls)."""
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["deit3_base", "dinov2_base_reg4"])
def test_full_size_against_fp32_module(api, fp32_cuda_reference, name, capsys):
    # 256 images through the engine and through the fp32 module on the same device
    model = LS.make_ls(name).cuda()
    image = LS.image_size(name)
    px = synth.make_pixels(256, image, seed=21).cuda()
    with torch.no_grad():
        ref = torch.cat([model(px[s:s + 64]).float() for s in range(0, 256, 64)])
    labels = ref.argmax(-1)
    batches = [{"pixel_values": px[s:s + 128], "labels": labels[s:s + 128]} for s in (0, 128)]
    logits = api.engine_for(model, "cuda", batch_hint=128).logits(px)
    err = (logits - ref).abs()
    got = api._compute_ffn_activation_importance(model, batches, device="cuda")
    want = O.s1_scores(model, batches, "cuda", None, autocast=False)
    rel = _rel([g.cpu() for g in got], [w.cpu() for w in want])
    plan = api.plan_2ssp_allocation(model, 0.375)
    t = plan.per_block_neurons_to_prune
    flips = 0
    for g_, w_ in zip(got, want):
        mg = torch.zeros_like(g_, dtype=torch.bool)
        mg[torch.argsort(g_.cpu(), stable=True)[:t].to(mg.device)] = True
        mw = torch.zeros_like(w_, dtype=torch.bool)
        mw[torch.argsort(w_.cpu(), stable=True)[:t].to(mw.device)] = True
        flips += int((mg != mw).sum())
    with capsys.disabled():
        print(f"\n[{name}] logits max/mean abs {err.max().item():.3e}/{err.mean().item():.3e}, scores rel {rel:.3e}, "
              f"mask bits differing at t={t}: {flips}")
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (err.max().item(), err.mean().item())
    assert rel <= SCORE_RTOL, rel
    assert flips <= 0.01 * sum(g_.numel() for g_ in got)
    api.release_engine(model)
