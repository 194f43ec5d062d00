"""DeiT models (two prefix tokens: CLS and distillation token; the averaged two-head classifier; 192-wide encoders) through
the engine and the drop-in API. GPU tests are marked `gpu`; the anatomy, refusal, configuration and planner checks at the
top run without one.

Tolerances are those of tests/test_gpu_parity.py. No golden vectors of the reference exist for DeiT: parity is against the
module's own fp32 forward (which is the reference's forward: it calls the module) and against the oracle's functions
(`O.s1_scores`, `O.s2_candidate_scores`, `O.plan`), which run on the DeiT modules unchanged.
"""
import copy
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth
from oracle import twossp_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import deit_synth as DS  # noqa: E402

SCORE_RTOL = 1e-2
LOGIT_MAX_ABS = 3e-2
LOGIT_MEAN_ABS = 5e-3
DELTA = 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(got, want):
    return max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, want))


def _logit_err(got, want):
    err = (got - want).abs()
    return err.max().item(), err.mean().item()


@torch.no_grad()
def _fp32_logits(model, px, batch=16):
    model = copy.deepcopy(model).float().cpu().eval()
    out = []
    for s in range(0, px.shape[0], batch):
        o = model(pixel_values=px[s:s + batch]) if hasattr(model, "config") else model(px[s:s + batch])
        out.append(O._logits_of(o).float())
    return torch.cat(out)


# ----------------------------------------------------------------------------------------------- no GPU needed
@pytest.mark.parametrize("head", DS.HEADS)
def test_anatomy_of_hf_deit(head):
    from twossp_b200.anatomy import describe
    a = describe(DS.make_deit("tiny", 0, head))
    assert (a.kind, a.prefix_tokens, a.hidden, a.heads, a.image_size, a.patch_size, a.n_blocks) == ("hf", 2, 192, 3, 48, 8, 3)
    assert a.globals_["pos"].reshape(-1, 192).shape[0] == 6 * 6 + 2
    assert a.globals_["dist"] is not None and a.score_point == 0
    assert a.dist_head == (head == "teacher")
    assert a.n_classes == (0 if head is None else 10)
    assert (a.globals_["head_dist_w"] is not None) == (head == "teacher")


def test_anatomy_of_timm_shaped_distilled_model():
    from twossp_b200.anatomy import describe
    a = describe(DS.TimmLikeDistilledViT())
    assert (a.kind, a.prefix_tokens, a.dist_head, a.n_classes, a.image_size, a.hidden, a.heads, a.score_point) == \
        ("timm", 2, True, 10, 48, 192, 3, 1)
    # a plain ViT keeps one prefix token and no distillation head
    a = describe(synth.make_vit("tiny", seed=0))
    assert (a.prefix_tokens, a.dist_head) == (1, False)


def test_refusals_name_the_problem():
    from twossp_b200.anatomy import describe
    m = DS.TimmLikeDistilledViT()
    m.head = torch.nn.Sequential(torch.nn.Linear(192, 32, bias=False), torch.nn.GELU(), torch.nn.Linear(32, 10))
    with pytest.raises(AttributeError, match="distillation head combined with a Sequential"):
        describe(m)
    m = DS.TimmLikeDistilledViT()
    m.pos_embed = torch.nn.Parameter(torch.zeros(1, 6 * 6 + 1, 192))  # the one-token layout next to a distillation token
    with pytest.raises(AttributeError, match="fits neither layout"):
        describe(m)
    m = DS.make_deit("tiny", 0, "teacher")
    m.deit.embeddings.position_embeddings = torch.nn.Parameter(torch.zeros(1, 40, 192))
    with pytest.raises(AttributeError, match="fits neither layout"):
        describe(m)


def test_attention_bypass_on_a_deit_module():
    from twossp_b200.anatomy import get_blocks, has_attention, install_bypass
    m = DS.make_deit("tiny", 0, "teacher")
    ref = copy.deepcopy(m)
    px = synth.make_pixels(3, 48, seed=5)
    install_bypass(m, 1)
    O.remove_attention(ref, 1)
    kind, blocks = get_blocks(m)
    assert [has_attention(kind, b) for b in blocks] == [True, False, True]
    with torch.no_grad():
        got, want = m(pixel_values=px).logits, ref(pixel_values=px).logits
        full = DS.make_deit("tiny", 0, "teacher")(pixel_values=px).logits
    assert torch.equal(got, want) and not torch.equal(got, full)


def _config(L, hidden=192, image=48, patch=8):
    cfg = L.TsspConfig()
    cfg.n_blocks, cfg.hidden, cfg.heads = 2, hidden, max(1, hidden // 64)
    cfg.image_size, cfg.patch_size, cfg.channels = image, patch, 3
    cfg.n_classes, cfg.head_hidden, cfg.max_images = 10, 0, 4
    cfg.score_point, cfg.cache_blocks, cfg.ln_eps = 0, 0, 1e-12
    for i in range(2):
        cfg.ffn_dims[i] = 256
        cfg.attn_present[i] = 1
    return cfg


def test_create_ex_validates_before_touching_a_device():
    import __graft_entry__ as g
    g.build()
    from twossp_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()

    def err(cfg, dist_token):
        cfg.dist_token = dist_token
        assert lib.tssp_create(C.byref(cfg), 4096, C.byref(h)) != 0   # device 4096 exists nowhere
        return lib.tssp_last_error().decode()

    for dist_token in (-1, 2):
        msg = err(_config(L), dist_token)
        assert f"dist_token={dist_token}" in msg, msg
    msg = err(_config(L, hidden=100), 1)
    assert "hidden=100" in msg and "192" in msg, msg
    msg = err(_config(L, image=40, patch=8), 1)            # T = 25 + 2 = 27
    assert "T=27" in msg and "[32,1025]" in msg, msg
    msg = err(_config(L, image=256, patch=8), 1)           # T = 1024 + 2
    assert "T=1026" in msg and "[32,1025]" in msg, msg
    # valid shapes pass validation and fail on the device: D = 192, T = 38 / 198 / 578
    for image, patch in ((48, 8), (224, 16), (384, 16)):
        msg = err(_config(L, image=image, patch=patch), 1)
        assert "device" in msg.lower() and "config" not in msg, msg
    # without a distillation token (one prefix token) T = 1025 is the last accepted
    assert "device" in err(_config(L, image=512, patch=16), 0).lower()


@pytest.fixture(scope="module")
def deit_planner_models():
    return {name: DS.make_deit(name, 0, "teacher") for name in ("ti", "small", "base")}


@pytest.mark.parametrize("name", ["ti", "small", "base"])
@pytest.mark.parametrize("target", [0.25, 0.375, 0.5])
def test_planner_matches_oracle_on_deit(deit_planner_models, name, target, capsys):
    from twossp_b200 import api
    m = deit_planner_models[name]
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


@pytest.fixture(scope="module")
def tiny_teacher():
    """(model on CPU, 24 pixels, fp32 logits of the module, self-labels)"""
    model = DS.make_deit("tiny", 0, "teacher")
    px = synth.make_pixels(24, 48, seed=1234)
    logits = _fp32_logits(model, px)
    return model, px, logits, logits.argmax(-1)


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
def test_im2col_with_one_and_two_prefix_rows_is_bit_exact(ops):
    for (n, Cc, H, P) in ((2, 3, 48, 8), (3, 3, 224, 16), (2, 3, 384, 16)):
        px = torch.randn(n, Cc, H, H, device="cuda")
        G = H // P
        patches = px.view(n, Cc, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(n, G * G, Cc * P * P)
        for prefix in (1, 2):
            out = ops.im2col(px, P, prefix=prefix)
            ref = torch.cat([torch.zeros(n, prefix, Cc * P * P, device="cuda"), patches], dim=1).bfloat16()
            assert torch.equal(out.view(torch.int16), ref.reshape(n * (G * G + prefix), -1).view(torch.int16))


@pytest.mark.gpu
def test_layernorm_at_192(ops):
    D = 192
    for rows in (333, 20011):
        x = torch.randn(rows, D, device="cuda") * 3 + 1
        g_, b_ = torch.randn(D, device="cuda"), torch.randn(D, device="cuda")
        ref = torch.nn.functional.layer_norm(x, (D,), g_, b_, 1e-12)
        out1 = ops.layernorm(x, g_, b_, 1e-12)
        out2 = ops.layernorm(x, g_, b_, 1e-12)   # consecutive launches walk the rows in opposite directions
        assert torch.equal(out1, out2)
        assert ((out1.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-4).all()
    # the prefix rows of every image (row pitch T*D), as the classifier tail reads them
    x = torch.randn(5 * 38, D, device="cuda")
    for r in (0, 1):
        out = ops.layernorm(x[r:], torch.ones(D, device="cuda"), torch.zeros(D, device="cuda"), 1e-6, row_stride=38 * D, rows=5)
        ref = torch.nn.functional.layer_norm(x.view(5, 38, D)[:, r], (D,), eps=1e-6)
        assert ((out.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-4).all()


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", [(198 * 16, 192, 192), (198 * 16, 192, 768), (38 * 9, 192, 192), (16, 1000, 192), (38 * 5, 10, 192)])
@pytest.mark.parametrize("reduce_add", [False, True])
def test_gemm_fp32_epilogue_at_192(ops, lib, gemm_form, M, N, K, reduce_add):
    # proj (K = 192), fc2 / patch-embed (K = 768), the tiny model's rows, the classifier heads (N = 1000 / 10)
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    base = torch.randn(M, N, generator=g).cuda()
    Np = (N + 7) // 8 * 8
    out = torch.full((M, Np), float("nan"), device="cuda")
    if reduce_add:
        out[:, :N] = base
    wp = torch.zeros(Np, K, dtype=torch.bfloat16, device="cuda")
    wp[:N] = w
    bp = torch.zeros(Np, device="cuda")
    bp[:N] = bias
    ops.gemm(lib.EPI_F32, a, wp, out, bp, reduce_add=reduce_add)
    ref = a.double() @ w.double().t() + bias.double() + (base.double() if reduce_add else 0)
    got = out[:, :N]
    assert torch.isfinite(got).all()
    assert (got.double() - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "gelu"])
@pytest.mark.parametrize("M,N,K", [(198 * 16, 576, 192), (38 * 9, 576, 192), (198 * 16, 768, 192), (38 * 9, 768, 192)])
def test_gemm_bf16_epilogue_at_192(ops, lib, gemm_form, mode, M, N, K):
    # QKV (N = 576: two 256-column tiles and a partial one of 64 columns) and fc1 (N = 768)
    g = torch.Generator().manual_seed(M * 3 + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.gemm(lib.EPI_BF16 if mode == "plain" else lib.EPI_BF16_GELU, a, w, out, bias)
    ref = a.float() @ w.float().t() + bias
    if mode == "gelu":
        ref = torch.nn.functional.gelu(ref)
    assert torch.isfinite(out.float()).all()
    assert ((out.float() - ref).abs() <= ref.abs() * (2 ** -8 + 2e-4) + 1e-5).all()


@pytest.mark.gpu
@pytest.mark.parametrize("M,heads", [(198 * 16, 3), (38 * 9, 3), (198 * 4, 12)])
def test_gemm_rownorm_epilogue_at_deit_shapes(ops, lib, gemm_form, M, heads):
    # the QKV GEMM with |q|^2 and |k|^2 per (row, head): N = 576 ends in a partial tile at D = 192
    D = heads * 64
    g = torch.Generator().manual_seed(M + heads)
    a = (torch.randn(M, D, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(3 * D, D, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(3 * D, generator=g).cuda()
    out = torch.full((M, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    norms = ops.gemm_rownorm(a, w, out, bias, 2 * heads)
    ref = a.float() @ w.float().t() + bias
    assert ((out.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-5).all()
    want = ref[:, : 2 * D].double().view(M, 2 * heads, 64).pow(2).sum(-1)
    assert torch.isfinite(norms).all()
    assert ((norms.double() - want).abs() <= want * 1e-4 + 1e-4).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("n_img,T,N,K", [(9, 38, 768, 192), (16, 198, 768, 192), (3, 578, 384, 192)])
def test_gemm_score_epilogue_at_192(ops, lib, gemm_form, pre, n_img, T, N, K):
    M = n_img * T
    g = torch.Generator().manual_seed(T + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    partials = torch.full((2 * ((M + 31) // 32), N), float("nan"), device="cuda")
    ops.gemm(lib.EPI_BF16_GELU_SCORE_PRE if pre else lib.EPI_BF16_GELU_SCORE, a, w, out, bias, partials=partials, tokens_per_image=T)
    norms = ops.score_finish(partials, n_img, T, N)
    z = a.float() @ w.float().t() + bias
    hooked = z if pre else torch.nn.functional.gelu(z)
    want = hooked.reshape(n_img, T, N).double().pow(2).sum(1).sqrt()
    rel = ((norms.double() - want).abs() / want.clamp_min(1e-9)).max().item()
    assert rel <= 5e-3, rel


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,heads", [(4, 198, 3), (3, 198, 12), (2, 578, 12), (5, 38, 3)])
def test_attention_at_deit_shapes(ops, n, T, heads):
    D = heads * 64
    g = torch.Generator(device="cuda").manual_seed(T * 7 + heads)
    qkv = torch.randn(n * T, 3 * D, device="cuda", generator=g).bfloat16()
    ctx = ops.attention(qkv, n, T, heads)
    q, k, v = qkv.float().view(n, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(n * T, D)
    assert torch.isfinite(ctx.float()).all()
    assert ((ctx.float() - ref).abs() <= ref.abs() * 2 ** -7 + 6e-3).all()


# ----------------------------------------------------------------------------------------------- tiny distilled DeiT
@pytest.mark.gpu
def test_tiny_teacher_logits_and_input_placement(api, tiny_teacher):
    model, px, ref, _ = tiny_teacher
    gm = copy.deepcopy(model).cuda()
    eng = api.engine_for(gm, "cuda", batch_hint=24)
    assert (eng.anatomy.prefix_tokens, eng.anatomy.dist_head) == (2, True)
    logits = eng.logits(px).cpu()
    mx, mean = _logit_err(logits, ref)
    assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    assert torch.equal(eng.logits(px.cuda()).cpu(), logits)          # device-resident pixels: same bits
    assert torch.equal(eng.logits(px.pin_memory()).cpu(), logits)    # pinned host pixels: same bits
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_teacher_scores_and_stage2_counts(api, tiny_teacher):
    model, px, _, labels = tiny_teacher
    batches = [{"pixel_values": px[:12], "labels": labels[:12]}, {"pixel_values": px[12:], "labels": labels[12:]}]
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    want = O.s1_scores(model, batches, "cpu", None, autocast=False)
    assert _rel(got, want) <= SCORE_RTOL
    base, cand, total = api.attention_removal_counts(gm, batches, "cuda", None)
    rb, rc, rt = O.s2_candidate_scores(model, batches, "cpu", None, autocast=False)
    assert total == rt == 24 and abs(base - rb) <= DELTA and all(abs(a - b) <= DELTA for a, b in zip(cand, rc)), (base, cand, rb, rc)
    for i in range(len(cand)):
        assert api._top1_counts(gm, batches, "cuda", None, skip_attn=[i]) == (cand[i], total), i
        trial = copy.deepcopy(model)
        O.remove_attention(trial, i)
        ours = api.engine_for(gm, "cuda", batch_hint=24).logits(px, skip_attn=[i]).cpu()
        assert (ours - _fp32_logits(trial, px)).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_teacher_captured_chains_equal_eager_launches(api, lib, tiny_teacher):
    model, px, _, labels = tiny_teacher
    batches = [{"pixel_values": px[:12], "labels": labels[:12]}, {"pixel_values": px[12:], "labels": labels[12:]}]
    out = {}
    for graphs in (0, 1):
        lib.check(lib.load().tssp_set_graphs(graphs))
        try:
            gm = copy.deepcopy(model).cuda()
            scores = api._compute_ffn_activation_importance(gm, batches, device="cuda")
            counts = api.attention_removal_counts(gm, batches, "cuda", None)
            logits = api.engine_for(gm, "cuda", batch_hint=12).logits(px[:12]).cpu()
            out[graphs] = (scores, counts, logits)
            api.release_engine(gm)
        finally:
            lib.check(lib.load().tssp_set_graphs(1))
    assert all(torch.equal(a, b) for a, b in zip(out[0][0], out[1][0]))
    assert out[0][1] == out[1][1] and torch.equal(out[0][2], out[1][2])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [160, 128])
def test_tiny_teacher_first_host_batch_split_gives_the_same_bits(api, lib, n):
    # T = 38: gcd(38, 32) = 2, so the parts are multiples of 16 images and keep their 32-row sub-tile offsets
    model = DS.make_deit("tiny", 0, "teacher").cuda()
    px = synth.make_pixels(n, 48, seed=11)
    eng = api.engine_for(model, "cuda", batch_hint=n)
    lib.check(lib.load().tssp_set_gemm_form(1))
    try:
        out = {}
        for where in ("device", "host"):
            eng.s1_reset()
            src = px.cuda() if where == "device" else px.pin_memory()
            norms = torch.zeros(n, sum(eng.ffn_dims), device="cuda")
            eng.s1_batch(src, img_norms=norms)
            eng.s1_batch(src[: n // 2])
            out[where] = (norms.cpu(), eng.s1_score_sums().clone())
    finally:
        lib.check(lib.load().tssp_set_gemm_form(0))
    assert float(out["device"][0].abs().min()) > 0
    assert torch.equal(out["device"][0], out["host"][0]) and torch.equal(out["device"][1], out["host"][1])
    api.release_engine(model)


@pytest.mark.gpu
def test_tiny_teacher_fit_and_both_prune_functions(api, tiny_teacher, capsys):
    model, px, _, labels = tiny_teacher
    batches = synth.make_batches(px, labels, 8)
    gm = copy.deepcopy(model).cuda()
    att, mlp = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None).fit()
    separate = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert all(torch.equal(a, b) for a, b in zip(mlp, separate))   # fused fit() sweep: the bits of the separate sweep
    ref_scores = O.s1_scores(model, batches, "cpu", None, autocast=False)
    assert _rel(mlp, ref_scores) <= SCORE_RTOL
    t = 200
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
        print(f"\n[tiny DeiT] mask disagreements vs oracle (block, neuron, rel. gap to cut): {len(listed)} of {got.size}: {listed}")
    assert [fc1.out_features for fc1, _ in api._gather_mlp_pairs(gm)] == [768 - t] * 3

    # Stage 2 on the width-pruned module: the selection must be the oracle's wherever the counts decide it
    pruned_cpu = copy.deepcopy(gm).cpu()
    rb, rc, rt = O.s2_candidate_scores(pruned_cpu, batches, "cpu", None, autocast=False)
    impacts = sorted(O.s2_impacts(rb, rc, rt))
    res = api.prune_vit_attention_blocks(gm, 0.0, dataloader=batches, device="cuda", batch_limit=None, importance_mode="copy",
                                         show_progress=False, num_to_prune=1)
    want = O.s2_prune(pruned_cpu, 0.0, batches, "cpu", batch_limit=None, num_to_prune=1, autocast=False)
    if impacts[1] - impacts[0] > 2 * DELTA / rt:
        assert res["pruned_indices"] == want["pruned_indices"], (res["pruned_indices"], want["pruned_indices"], impacts)
    assert len(res["pruned_indices"]) == 1 and res["final_metrics"] is not None
    assert api._count_attention_params_per_block(gm)[res["pruned_indices"][0]] == 0
    # the mutated module's own fp32 forward (odd widths, bypassed attention) agrees with the engine's logits
    el = api.engine_for(gm, "cuda", batch_hint=8).logits(px).cpu()
    mx, mean = _logit_err(el, _fp32_logits(gm, px))
    assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_teacher_odd_width_pruned_model_runs(api):
    model = DS.make_deit("tiny", 0, "teacher").cuda()
    g_ = torch.Generator().manual_seed(3)
    imps = [torch.rand(768, generator=g_) for _ in range(3)]
    api.prune_vit_mlp_width(model, n_to_prune_per_block=[5, 61, 123], precomputed_importance=imps, min_remaining=8)
    api.prune_vit_attention_blocks(model, 0.0, selected_indices=[2], num_to_prune=1)   # the last block: tail without attention
    px = synth.make_pixels(5, 48, seed=2)
    got = api.engine_for(model, "cuda", batch_hint=5).logits(px).cpu()
    assert (got - _fp32_logits(model, px)).abs().max().item() <= LOGIT_MAX_ABS
    scores = api._compute_ffn_activation_importance(model, [{"pixel_values": px}], device="cuda")
    assert [s.numel() for s in scores] == [763, 707, 645]
    ref_scores = O.s1_scores(copy.deepcopy(model).cpu(), [{"pixel_values": px}], "cpu", None, autocast=False)
    assert _rel(scores, ref_scores) <= SCORE_RTOL
    api.release_engine(model)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["cls", "timm", "bare"])
def test_other_deit_layouts(api, which):
    """DeiTForImageClassification (tail on row 0 only), the timm-shaped distilled stand-in (pre-GELU score point) and the
    bare DeiTModel (scores only)."""
    if which == "timm":
        model = DS.TimmLikeDistilledViT()
    else:
        model = DS.make_deit("tiny", 0, "cls" if which == "cls" else None)
    px = synth.make_pixels(10, 48, seed=9)
    batches = [{"pixel_values": px[:6]}, {"pixel_values": px[6:]}]
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert _rel(got, O.s1_scores(model, batches, "cpu", None, autocast=False)) <= SCORE_RTOL
    eng = api.engine_for(gm, "cuda", batch_hint=10)
    assert eng.anatomy.dist_head == (which == "timm")
    if which == "bare":
        with pytest.raises(Exception, match="no classification head"):
            eng.logits(px)
    else:
        mx, mean = _logit_err(eng.logits(px).cpu(), _fp32_logits(model, px))
        assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    api.release_engine(gm)


@pytest.mark.gpu
def test_plain_vit_at_192(api):
    synth.SHAPES.setdefault("vit_ti4", (224, 16, 192, 4, 3, 768, 100))   # ViT-Ti/16 width, four blocks, T = 197
    model = synth.make_vit("vit_ti4", seed=0)
    px = synth.make_pixels(8, 224, seed=21)
    ref = O.vit_forward(O.extract_weights(model), px)
    gm = copy.deepcopy(model).cuda()
    mx, mean = _logit_err(api.engine_for(gm, "cuda", batch_hint=8).logits(px).cpu(), ref["logits"])
    assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    got = api._compute_ffn_activation_importance(gm, [{"pixel_values": px}], device="cuda")
    assert _rel(got, [nm.sum(0) / 8 for nm in ref["norms"]]) <= SCORE_RTOL
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_teacher_recycled_buffers_under_pool_poison():
    # engines built on recycled (0xFF-poisoned) device blocks give the bits of the first engine
    code = """
import copy, sys, torch
sys.path.insert(0, %r)
sys.path.insert(0, %r)
from oracle import synth
import deit_synth as DS
from twossp_b200 import api, _lib as L
model = DS.make_deit("tiny", 0, "teacher")
px = synth.make_pixels(12, 48, seed=1234)
with torch.no_grad():
    labels = model(pixel_values=px).logits.argmax(-1)
batches = synth.make_batches(px, labels, 4)
outs = []
for rep in range(3):
    gm = copy.deepcopy(model).cuda()
    att, mlp = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None).fit()
    logits = api.engine_for(gm, "cuda", batch_hint=4, need_cache=True).logits(px).cpu()
    outs.append((att, mlp, logits))
    api.release_engine(gm)
for att, mlp, logits in outs[1:]:
    assert torch.equal(att, outs[0][0]) and torch.equal(logits, outs[0][2])
    assert all(torch.equal(a, b) for a, b in zip(mlp, outs[0][1])) and all(bool(torch.isfinite(t).all()) for t in mlp)
assert bool(torch.isfinite(outs[0][2]).all())
assert L.load().tssp_trim_pool() == 0
print("recycled ok")
""" % (ROOT, os.path.join(ROOT, "tests"))
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    env = dict(os.environ, TSSP_POOL_POISON="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "recycled ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ----------------------------------------------------------------------------------------------- full size
@pytest.fixture
def fp32_cuda_reference():
    """The module's own forward on the GPU in true fp32 (no TF32 in the patch convolution or the matmuls)."""
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


@pytest.mark.gpu
def test_deit_base_distilled_224_against_fp32_module(api, fp32_cuda_reference):
    """DeiT-B-distilled/16 at 224^2 (T = 198) on 64 images: scores, logits and Stage-2 counts against the module's own
    fp32 forward (run on the GPU so that the 13 Stage-2 forwards stay affordable)."""
    model = DS.make_deit("base", 0, "teacher")
    n_img = 64
    px = synth.make_pixels(n_img, 224, seed=21)
    ref_model = copy.deepcopy(model).cuda()
    with torch.no_grad():
        ref_logits = torch.cat([ref_model(pixel_values=px[s:s + 16].cuda()).logits.float().cpu() for s in range(0, n_img, 16)])
    labels = ref_logits.argmax(-1)
    batches = synth.make_batches(px, labels, 32)
    ref_scores = O.s1_scores(ref_model, batches, "cuda", None, autocast=False)
    rb, rc, rt = O.s2_candidate_scores(ref_model, batches, "cuda", None, autocast=False)
    del ref_model
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    rel = torch.cat([((a - b).abs() / b.abs()) for a, b in zip(got, ref_scores)])
    assert float(rel.mean()) <= 2e-3 and float(torch.quantile(rel, 0.999)) <= SCORE_RTOL and float(rel.max()) <= 1.5 * SCORE_RTOL, \
        (float(rel.mean()), float(rel.max()))
    mx, mean = _logit_err(api.engine_for(gm, "cuda", batch_hint=32).logits(px).cpu(), ref_logits)
    assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    base, cand, total = api.attention_removal_counts(gm, batches, "cuda", None)
    tol = max(DELTA, int(0.01 * n_img))
    assert total == rt == n_img and abs(base - rb) <= tol and all(abs(a - b) <= tol for a, b in zip(cand, rc)), (base, cand, rb, rc)
    api.release_engine(gm, trim=True)


@pytest.mark.gpu
def test_deit_base_distilled_384_logits(api, fp32_cuda_reference):
    """DeiT-B-distilled/16 at 384^2 (T = 578: the key-tiled attention kernel) on 4 images."""
    model = DS.make_deit("base384", 0, "teacher")
    px = synth.make_pixels(4, 384, seed=22)
    ref_model = copy.deepcopy(model).cuda()
    with torch.no_grad():
        ref = ref_model(pixel_values=px.cuda()).logits.float().cpu()
    del ref_model
    gm = copy.deepcopy(model).cuda()
    mx, mean = _logit_err(api.engine_for(gm, "cuda", batch_hint=4).logits(px).cpu(), ref)
    assert mx <= LOGIT_MAX_ABS and mean <= LOGIT_MEAN_ABS, (mx, mean)
    api.release_engine(gm, trim=True)
