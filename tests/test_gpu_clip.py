"""CLIP image towers (timm `pre_norm=True`: `norm_pre`, QuickGELU MLPs, a bias-free patch embedding; OpenAI / LAION ViT-B/32,
B/16, L/14, L/14@336) through the engine and the drop-in API. GPU tests are marked `gpu`; the anatomy, refusal,
configuration, signature and planner checks at the top run without one.

Parity is against the stand-in's own fp32 forward and the oracle's hook-based functions, which run it unchanged (timm hook
point: `mlp.fc1`, before the activation). Tolerances are those of DESIGN §4.
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
import clip_synth as CS  # noqa: E402

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


def _quick_gelu(x):
    return x * torch.sigmoid(1.702 * x)


# ----------------------------------------------------------------------------------------------- no GPU needed
@pytest.fixture(scope="module")
def clip_models():
    return {}


def _model(cache, name):
    """The planner's models are kept for the module; the others (L/14@336: 300 M parameters) are built once and dropped."""
    if name in cache:
        return cache[name]
    m = CS.make_clip(name)
    if name in ("b32", "b16", "l14"):
        cache[name] = m
    return m


@pytest.mark.parametrize("name,T", [("tiny", 37), ("tiny192", 37), ("b32", 50), ("b16", 197), ("l14", 257), ("l14_336", 577)])
def test_anatomy_of_clip_towers(clip_models, name, T):
    from twossp_b200.anatomy import describe
    image, patch, dim, depth, heads, hidden, classes = CS.CLIP_SHAPES[name]
    m = _model(clip_models, name)
    a = describe(m)
    assert (a.kind, a.hidden, a.heads, a.image_size, a.patch_size, a.n_blocks, a.score_point, a.n_classes) == \
        ("timm", dim, heads, image, patch, depth, 1, classes)
    assert a.pre_norm and a.ffn_act == "quick_gelu" and a.ln_eps == CS.EPS
    assert (a.prefix_tokens, a.register_tokens, a.layer_scale, a.dist_token) == (1, 0, False, False)
    assert (image // patch) ** 2 + a.prefix_tokens == T
    assert a.globals_["patch_b"] is None                                      # bias=not pre_norm
    assert torch.equal(a.globals_["norm_pre_w"], m.norm_pre.weight) and torch.equal(a.globals_["norm_pre_b"], m.norm_pre.bias)


def test_anatomy_of_the_erf_and_non_affine_variants():
    from twossp_b200.anatomy import describe
    a = describe(CS.make_clip("tiny", act="gelu", pre_norm=False))
    assert not a.pre_norm and a.ffn_act == "gelu" and a.globals_["patch_b"] is not None and a.globals_["norm_pre_w"] is None
    m = CS.make_clip("tiny")
    m.norm_pre = torch.nn.LayerNorm(128, eps=CS.EPS, elementwise_affine=False)
    a = describe(m)
    assert a.pre_norm and torch.equal(a.globals_["norm_pre_w"], torch.ones(128)) and torch.equal(a.globals_["norm_pre_b"], torch.zeros(128))
    a = describe(CS.ClipLayerScaleViT())
    assert (a.pre_norm, a.ffn_act, a.layer_scale, a.register_tokens, a.pos_covers_prefix) == (True, "quick_gelu", True, 4, False)


def _mix(m):
    m.blocks[2].mlp.act = torch.nn.GELU()


@pytest.mark.parametrize("what,mutate,match", [
    ("tanh_gelu", lambda m: setattr(m.blocks[0].mlp, "act", torch.nn.GELU(approximate="tanh")),
     r"blocks\[0\]\.mlp\.act \(GELU, approximate='tanh'\)"),
    ("silu", lambda m: setattr(m.blocks[1].mlp, "act", torch.nn.SiLU()), r"blocks\[1\]\.mlp\.act \(SiLU\)"),
    ("mixed", _mix, r"blocks\[2\]\.mlp\.act \(GELU\) differs from blocks\[0\]\.mlp\.act \(QuickGELU\)"),
    ("norm_pre_rms", lambda m: setattr(m, "norm_pre", torch.nn.RMSNorm(128, eps=CS.EPS)), r"norm_pre \(RMSNorm\)"),
    ("norm_pre_width", lambda m: setattr(m, "norm_pre", torch.nn.LayerNorm(64, eps=CS.EPS)), r"norm_pre \(LayerNorm\)"),
    ("norm_pre_eps", lambda m: setattr(m, "norm_pre", torch.nn.LayerNorm(128, eps=1e-6)), r"norm_pre\.eps=1e-06 differs from norm\.eps"),
])
def test_refusals_name_the_attribute(what, mutate, match):
    from twossp_b200.anatomy import describe
    m = CS.make_clip("tiny")
    mutate(m)
    with pytest.raises(AttributeError, match=match):
        describe(m)


def test_tanh_gelu_vit_without_other_extras_is_refused():
    # before pre-norm / QuickGELU support this model ran with erf GELU and no error
    from twossp_b200.anatomy import describe
    m = synth.TimmLikeViT()
    for b in m.blocks:
        b.mlp.act = torch.nn.GELU(approximate="tanh")
    with pytest.raises(AttributeError, match=r"blocks\[0\]\.mlp\.act"):
        describe(m)
    describe(synth.TimmLikeViT())


def test_signature_changes_when_an_activation_is_swapped():
    from twossp_b200 import api
    m = CS.make_clip("tiny")
    before = api._signature(m)
    assert api._signature(m) == before
    m.blocks[1].mlp.act = torch.nn.GELU()
    erf = api._signature(m)
    assert erf != before
    m.blocks[1].mlp.act = torch.nn.GELU(approximate="tanh")
    assert api._signature(m) not in (before, erf)
    m.blocks[1].mlp.act = CS.QuickGELU()
    assert api._signature(m) == before


def _config(L, hidden=768, image=224, patch=16, score_point=1, heads=None):
    cfg = L.TsspConfig()
    cfg.n_blocks, cfg.hidden, cfg.heads = 2, hidden, hidden // 64 if heads is None else heads
    cfg.image_size, cfg.patch_size, cfg.channels = image, patch, 3
    cfg.n_classes, cfg.head_hidden, cfg.max_images = 10, 0, 4
    cfg.score_point, cfg.cache_blocks, cfg.ln_eps = score_point, 0, 1e-5
    for i in range(2):
        cfg.ffn_dims[i] = 4 * hidden
        cfg.attn_present[i] = 1
    return cfg


def test_create_model_validates_before_touching_a_device():
    import __graft_entry__ as g
    g.build()
    from twossp_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()

    def err(cfg, pre_norm, ffn_act, layout=(0, 0, 0, 0)):   # layout: (dist_token, register_tokens, pos_patches_only, layer_scale)
        cfg.pre_norm, cfg.ffn_act = pre_norm, ffn_act
        cfg.dist_token, cfg.register_tokens, cfg.pos_patches_only, cfg.layer_scale = layout
        assert lib.tssp_create(C.byref(cfg), 4096, C.byref(h)) != 0   # no device 4096
        return lib.tssp_last_error().decode()

    msg = err(_config(L), 2, 1)
    assert "pre_norm=2" in msg, msg
    msg = err(_config(L), 1, 2)
    assert "ffn_act=2" in msg, msg
    msg = err(_config(L, score_point=0), 1, 1)   # QuickGELU is scored before the activation only
    assert "score_point=1" in msg, msg
    msg = err(_config(L, hidden=1280, image=224, patch=14, heads=16), 1, 1)   # ViT-H/14 CLIP: head dim 80
    assert "config: hidden=1280" in msg, msg
    assert lib.tssp_create(None, 4096, C.byref(h)) != 0
    assert "NULL" in lib.tssp_last_error().decode()
    # every CLIP shape passes validation and fails on the device: B/32 (T = 50), B/16, L/14, L/14@336 (T = 577), with and
    # without the pre-norm, and the combined layout of registers and LayerScale
    for hidden, image, patch, opts, layout in ((768, 224, 32, (1, 1), (0, 0, 0, 0)), (768, 224, 16, (1, 1), (0, 0, 0, 0)),
                                               (1024, 224, 14, (1, 1), (0, 0, 0, 0)), (1024, 336, 14, (1, 1), (0, 0, 0, 0)),
                                               (768, 224, 16, (0, 1), (0, 0, 0, 0)), (128, 84, 14, (1, 1), (0, 4, 1, 1))):
        msg = err(_config(L, hidden=hidden, image=image, patch=patch), *opts, layout)
        assert "device" in msg.lower() and "config" not in msg and "options" not in msg, msg


@pytest.mark.parametrize("name", ["b32", "b16", "l14"])
@pytest.mark.parametrize("target", [0.25, 0.5])
def test_planner_matches_oracle_on_clip_towers(clip_models, name, target):
    from twossp_b200 import api
    m = _model(clip_models, name)
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


def _ulps(a_bf16, b_bf16):
    """|a - b| in bf16 ulps (ordered integer view of the bit patterns)."""
    def ordered(t):
        i = t.view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (ordered(a_bf16) - ordered(b_bf16)).abs()


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["qgelu", "qgelu_score_pre"])
def test_quickgelu_epilogue_is_within_one_bf16_ulp(ops, lib, gemm_form, mode, capsys):
    # A = 0, so every row of the output is quickgelu(bias): a dense fp32 grid over [-12, 12]
    M, K, N = 256, 64, 48000
    bias = torch.linspace(-12.0, 12.0, N, device="cuda")
    a = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    w = torch.zeros(N, K, device="cuda", dtype=torch.bfloat16)
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    if mode == "qgelu":
        ops.gemm(lib.EPI_BF16_QGELU, a, w, out, bias)
    else:
        partials = torch.full((2 * (M // 32), N), float("nan"), device="cuda")
        ops.gemm(lib.EPI_BF16_QGELU_SCORE_PRE, a, w, out, bias, partials=partials, tokens_per_image=M)
        # one image: the pre-activation squares of 32 rows per sub-tile, all of segment 0
        want = 32 * bias.bfloat16().float() ** 2
        assert torch.allclose(partials[0::2], want.expand(M // 32, N), rtol=1e-6)
    want = _quick_gelu(bias).bfloat16()
    assert torch.equal(out, out[:1].expand(M, N))
    u = _ulps(out[0], want)
    exact = float((u == 0).float().mean())
    with capsys.disabled():
        print(f"\n[quickgelu {mode}, {gemm_form} CTA] max {int(u.max())} bf16 ulp, exact roundings {100 * exact:.3f} % of {N}")
    assert int(u.max()) <= 1
    assert exact >= 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("n_img,T,N,K", [(16, 197, 3072, 768), (8, 257, 4096, 1024), (9, 197, 1000, 768), (6, 50, 2040, 768)])
def test_quickgelu_modes_match_torch(ops, lib, gemm_form, n_img, T, N, K):
    # the fc1 shapes of B/16 and L/14, a pruned width that is not a multiple of 64, and B/32's T = 50
    M = n_img * T
    g = torch.Generator().manual_seed(T + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = (torch.randn(N, generator=g) - 1.0).cuda()
    z = a.float() @ w.float().t() + bias
    act = _quick_gelu(z)
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.gemm(lib.EPI_BF16_QGELU, a, w, out, bias)
    # one bf16 rounding (half an ulp <= 2^-8 relative) of a value within a few fp32 ulps of the fp32 result
    assert ((out.float() - act).abs() <= act.abs() * (2 ** -8 + 1e-4) + 1e-5).all()
    out8 = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    partials = torch.full((2 * ((M + 31) // 32), N), float("nan"), device="cuda")
    ops.gemm(lib.EPI_BF16_QGELU_SCORE_PRE, a, w, out8, bias, partials=partials, tokens_per_image=T)
    assert torch.equal(out8, out)
    norms = ops.score_finish(partials, n_img, T, N)
    want = z.reshape(n_img, T, N).double().pow(2).sum(1).sqrt()
    assert ((norms.double() - want).abs() / want.clamp_min(1e-9)).max().item() <= 5e-3


@pytest.mark.gpu
@pytest.mark.parametrize("n_img,T,N,K", [(16, 197, 3072, 768), (7, 50, 1000, 768), (5, 37, 512, 128)])
def test_quickgelu_score_partials_equal_the_erf_ones(ops, lib, gemm_form, n_img, T, N, K):
    # the score is taken before the activation: mode 8's partials are mode 3's, bit for bit
    M = n_img * T
    g = torch.Generator().manual_seed(M + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = (torch.randn(N, generator=g) - 1.0).cuda()
    parts = {}
    for mode in (lib.EPI_BF16_GELU_SCORE_PRE, lib.EPI_BF16_QGELU_SCORE_PRE):
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        parts[mode] = torch.full((2 * ((M + 31) // 32), N), float("nan"), device="cuda")
        ops.gemm(mode, a, w, out, bias, partials=parts[mode], tokens_per_image=T)
    assert torch.equal(parts[lib.EPI_BF16_GELU_SCORE_PRE], parts[lib.EPI_BF16_QGELU_SCORE_PRE])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 5])
def test_im2col_patch32_is_bit_exact(ops, n):
    px = torch.randn(n, 3, 224, 224, device="cuda")
    out = ops.im2col(px, 32)
    K = 3 * 32 * 32
    assert out.shape == (n * 50, K)
    ref = torch.nn.functional.unfold(px, 32, stride=32).transpose(1, 2)
    ref = torch.cat([torch.zeros(n, 1, K, device="cuda"), ref], dim=1).bfloat16().reshape(-1, K)
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [128, 192, 384, 768, 1024])
def test_layernorm_f32(ops, D):
    rows = 50 * 7 + 3
    g = torch.Generator(device="cuda").manual_seed(D)
    x = torch.randn(rows, D, device="cuda", generator=g) * 3 + 0.5
    gamma = 1 + 0.1 * torch.randn(D, device="cuda", generator=g)
    beta = 0.05 * torch.randn(D, device="cuda", generator=g)
    out = ops.layernorm_f32(x, gamma, beta, CS.EPS)
    ref = torch.nn.functional.layer_norm(x.double(), (D,), gamma.double(), beta.double(), CS.EPS)
    assert (out.double() - ref).abs().max().item() <= 2e-5
    # the bf16 LayerNorm's bits, rounded from the fp32 form
    assert torch.equal(out.bfloat16().view(torch.int16), ops.layernorm(x, gamma, beta, CS.EPS).view(torch.int16))
    # in place, and into a wider row pitch
    y = x.clone()
    ops.layernorm_f32(y, gamma, beta, CS.EPS, out=y)
    assert torch.equal(y, out)
    wide = torch.full((rows, D + 4), float("nan"), device="cuda")
    ops.layernorm_f32(x, gamma, beta, CS.EPS, out=wide[:, :D])
    assert torch.equal(wide[:, :D], out) and wide[:, D:].isnan().all()


@pytest.mark.gpu
def test_load_weights_refuses_a_table_that_disagrees_with_its_config(lib):
    L = lib
    lb = L.load()
    n = L.W_GLOBAL_COUNT + 2 * L.BW_COUNT
    buf = torch.zeros(1 << 20, device="cuda")   # what every set slot points at: large enough for any entry, never read
    required = [L.W_PATCH_W, L.W_CLS, L.W_POS, L.W_FINAL_LN_W, L.W_FINAL_LN_B, L.W_HEAD_W] + \
               [L.W_GLOBAL_COUNT + b * L.BW_COUNT + i for b in range(2) for i in range(L.BW_LS1)]

    def refused(fields, set_slots=(), null_slots=(), entries=n):
        """the message of tssp_load_weights for an engine of _config + fields and a table with every plain-ViT entry set"""
        cfg = _config(L, hidden=128, image=48, patch=8)
        for k, v in fields.items():
            setattr(cfg, k, v)
        table = (C.c_void_p * max(n, entries))()
        for i in [i for i in required if i not in null_slots] + list(set_slots):
            table[i] = buf.data_ptr()
        h = C.c_void_p()
        L.check(lb.tssp_create(C.byref(cfg), 0, C.byref(h)))
        try:
            assert lb.tssp_load_weights(h, table, entries, None) != 0
            return lb.tssp_last_error().decode()
        finally:
            lb.tssp_destroy(h)

    clip = {"pre_norm": 1, "ffn_act": 1}
    for entries in (n - 2, n + 2):   # a table of another length: the count is named
        msg = refused(clip, entries=entries)
        assert f"expected {n} pointers" in msg and f"got {entries}" in msg, msg
    msg = refused(clip, null_slots=required)   # all NULL: refused by name, nothing read
    assert "NULL" in msg, msg
    msg = refused(clip)
    assert "norm_pre weight or bias is NULL" in msg, msg
    msg = refused({"ffn_act": 1}, set_slots=[L.W_NORM_PRE_W, L.W_NORM_PRE_B])
    assert "TSSP_W_NORM_PRE_W" in msg and "pre_norm=0" in msg, msg
    # the same for the LayerScale gammas and the distillation token
    msg = refused({"layer_scale": 1}, set_slots=[L.W_GLOBAL_COUNT + L.BW_LS1, L.W_GLOBAL_COUNT + L.BW_COUNT + L.BW_LS1])
    assert "block 0 LS2 gamma is NULL" in msg, msg
    msg = refused({}, set_slots=[L.W_GLOBAL_COUNT + L.BW_COUNT + L.BW_LS1])
    assert "block 1 TSSP_BW_LS1" in msg and "layer_scale=0" in msg, msg
    msg = refused({"dist_token": 1})
    assert "distillation token is NULL" in msg, msg
    msg = refused({}, set_slots=[L.W_DIST_TOKEN])
    assert "TSSP_W_DIST_TOKEN" in msg and "dist_token=0" in msg, msg


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
def test_block0_scores_do_not_depend_on_the_activation(api):
    qg = CS.make_clip("tiny")
    erf = copy.deepcopy(qg)
    for b in erf.blocks:
        b.mlp.act = torch.nn.GELU()
    px = synth.make_pixels(24, 48, seed=10)
    batches = [{"pixel_values": px[:12]}, {"pixel_values": px[12:]}]
    got = {}
    for key, m in (("qg", qg), ("erf", erf)):
        gm = copy.deepcopy(m).cuda()
        got[key] = api._compute_ffn_activation_importance(gm, batches, device="cuda")
        api.release_engine(gm)
    assert torch.equal(got["qg"][0], got["erf"][0])
    assert not torch.equal(got["qg"][1], got["erf"][1])


# ----------------------------------------------------------------------------------------------- tiny stand-ins
def _tiny_models():
    return {"tiny": lambda: CS.make_clip("tiny"), "tiny192": lambda: CS.make_clip("tiny192"), "reg4_ls": CS.ClipLayerScaleViT,
            "p32": lambda: CS.TimmLikeClipViT(image=224, patch=32, depth=2)}   # B/32's T = 50 at the test width


@pytest.fixture(scope="module", params=["tiny", "tiny192", "reg4_ls"])
def tiny(request):
    """(name, model on CPU, 24 pixels, fp32 logits of the module, self-labels)"""
    model = _tiny_models()[request.param]()
    px = synth.make_pixels(24, 84 if request.param == "reg4_ls" else 48, seed=1234)
    logits = _fp32_logits(model, px)
    return request.param, model, px, logits, logits.argmax(-1)


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
def test_engine_is_rebuilt_when_the_activation_is_swapped(api):
    model = CS.make_clip("tiny").cuda()
    px = synth.make_pixels(8, 48, seed=4)
    first = api.engine_for(model, "cuda", batch_hint=8).logits(px).cpu()
    for b in model.blocks:
        b.mlp.act = torch.nn.GELU()
    eng = api.engine_for(model, "cuda", batch_hint=8)
    assert eng.anatomy.ffn_act == "gelu"
    swapped = eng.logits(px).cpu()
    assert not torch.equal(first, swapped)
    assert (swapped - _fp32_logits(model, px)).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(model)


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
@pytest.mark.parametrize("name,image", [("tiny", 48), ("reg4_ls", 84), ("p32", 224)])
def test_tiny_first_host_batch_split_gives_the_same_bits(api, name, image):
    # T = 37 / 41: gcd(T, 32) = 1, so the parts are multiples of 32 images; T = 50: gcd 2, multiples of 16. Either way every
    # image keeps its 32-row sub-tile offsets
    n = 160
    model = _tiny_models()[name]().cuda()
    px = synth.make_pixels(n, image, seed=11)
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
    # the mutated module (odd widths, a bypassed attention) against the engine
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
@pytest.mark.parametrize("name,n", [("b16", 256), ("l14_336", 128)])
def test_full_size_against_fp32_module(api, fp32_cuda_reference, name, n, capsys):
    model = CS.make_clip(name).cuda()
    px = synth.make_pixels(n, CS.image_size(name), seed=21).cuda()
    with torch.no_grad():
        ref = torch.cat([model(px[s:s + 32]).float() for s in range(0, n, 32)])
    labels = ref.argmax(-1)
    batches = [{"pixel_values": px[s:s + 64], "labels": labels[s:s + 64]} for s in range(0, n, 64)]
    logits = api.engine_for(model, "cuda", batch_hint=64).logits(px)
    err = (logits - ref).abs()
    got = api._compute_ffn_activation_importance(model, batches, device="cuda")
    want = O.s1_scores(model, batches, "cuda", None, autocast=False)
    rels = torch.cat([((g.cpu() - w.cpu()).abs() / w.cpu().abs()) for g, w in zip(got, want)])
    with capsys.disabled():
        print(f"\n[{name}, {n} images] logits max/mean abs {err.max().item():.3e}/{err.mean().item():.3e}, scores rel max "
              f"{rels.max().item():.3e}, 99.9 % quantile {rels.quantile(0.999).item():.3e}")
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (err.max().item(), err.mean().item())
    if len(got) > 12:   # the ViT-L depth rule of DESIGN §4: 99.9 % <= 1e-2, worst <= 1.5e-2
        assert rels.quantile(0.999).item() <= SCORE_RTOL and rels.max().item() <= 1.5e-2
    else:
        assert rels.max().item() <= SCORE_RTOL
    api.release_engine(model)
