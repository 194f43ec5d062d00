"""ViTs with more than 208 tokens per image (384^2 at patch 16: T = 577; patch 8: T = 290 at 136^2, 785 at 224^2): the
key-tiled attention kernel (csrc/attention_long_tcgen05.cuh) and the engine around it. GPU tests are marked `gpu`; the
configuration check at the bottom runs without one.

Tolerances are those stated at the top of tests/test_gpu_parity.py. No golden vectors recorded from the unmodified
reference exist at these shapes (the reference is not available where these tests were written): parity is against the
fp32 oracle (oracle/twossp_oracle.py), which is pinned to the reference's goldens at the recorded sizes and runs the HF
module, or a functional restatement of it, at any shape.
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

SCORE_RTOL = 1e-2
LOGIT_MAX_ABS = 3e-2
LOGIT_MEAN_ABS = 5e-3
DELTA = 2

# (image, patch, hidden, layers, heads, ffn, labels) in the layout of synth.SHAPES
LONG_SHAPES = {
    "tiny_long": (136, 8, 128, 3, 2, 256, 10),      # T = 290: three query tiles, one of them 34 rows
    "base384": (384, 16, 768, 12, 12, 3072, 1000),  # T = 577: ViT-B/16 at 384^2
}
for _name, _shape in LONG_SHAPES.items():
    synth.SHAPES.setdefault(_name, _shape)


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


@pytest.fixture(scope="module")
def tiny_long():
    """(model on CPU, 24 pixels, fp32 oracle forward of them)"""
    model = synth.make_vit("tiny_long", seed=0)
    px = synth.make_pixels(24, 136, seed=1234)
    return model, px, O.vit_forward(O.extract_weights(model), px)


# ----------------------------------------------------------------------------------------------- kernel
@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 0.05, 3.0])   # 3.0 makes the Cauchy-Schwarz shift too loose: exact two-sweep route
@pytest.mark.parametrize("n,T,heads", [(2, 209, 2), (2, 224, 4), (3, 257, 2), (3, 290, 2), (2, 577, 12), (1, 785, 12),
                                       (1, 1025, 16), (130, 577, 12)])
def test_long_attention(ops, n, T, heads, scale):
    D = heads * 64
    g = torch.Generator(device="cuda").manual_seed(T * 31 + n)
    qkv = (torch.randn(n * T, 3 * D, device="cuda", generator=g) * scale).bfloat16()
    ctx = ops.attention(qkv, n, T, heads)
    q, k, v = qkv.float().view(n, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(n * T, D)
    assert torch.isfinite(ctx.float()).all()
    # bf16 P and one bf16 rounding of outputs of magnitude O(scale)
    assert ((ctx.float() - ref).abs() <= ref.abs() * 2 ** -7 + 6e-3 * max(1.0, scale)).all()
    assert torch.equal(ops.attention(qkv, n, T, heads), ctx)


@pytest.mark.gpu
def test_long_attention_rejects_sequences_past_its_range(ops, lib):
    qkv = torch.zeros(1026, 3 * 128, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(lib.TsspError, match="1025"):
        ops.attention(qkv, 1, 1026, 2)


# ----------------------------------------------------------------------------------------------- tiny_long model
@pytest.mark.gpu
def test_tiny_long_logits_and_scores(api, tiny_long):
    model, px, ref = tiny_long
    gm = copy.deepcopy(model).cuda()
    eng = api.engine_for(gm, "cuda", batch_hint=24)
    logits = eng.logits(px).cpu()
    err = (logits - ref["logits"]).abs()
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (err.max().item(), err.mean().item())
    assert torch.equal(eng.logits(px.cuda()).cpu(), logits)   # device-resident input: same bits
    got = api._compute_ffn_activation_importance(gm, [{"pixel_values": px[:16]}, {"pixel_values": px[16:]}], device="cuda")
    want = [nm.sum(0) / 24 for nm in ref["norms"]]
    rel = max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, want))
    assert rel <= SCORE_RTOL, rel
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_long_stage2_counts_and_suffix_recompute(api, tiny_long):
    model, px, ref = tiny_long
    labels = ref["logits"].argmax(-1)
    batches = [{"pixel_values": px[:12], "labels": labels[:12]}, {"pixel_values": px[12:], "labels": labels[12:]}]
    gm = copy.deepcopy(model).cuda()
    base, cand, total = api.attention_removal_counts(gm, batches, "cuda", None)
    rb, rc, rt = O.s2_candidate_scores(model, batches, "cpu", None, autocast=False)
    assert total == rt == 24 and abs(base - rb) <= DELTA and all(abs(a - b) <= DELTA for a, b in zip(cand, rc)), (base, cand, rb, rc)
    for i in range(len(cand)):
        assert api._top1_counts(gm, batches, "cuda", None, skip_attn=[i]) == (cand[i], total), i
        skipped = O.vit_forward(O.extract_weights(model), px, skip_attention=(i,))["logits"]
        ours = api.engine_for(gm, "cuda", batch_hint=24).logits(px, skip_attn=[i]).cpu()
        assert (ours - skipped).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_long_fit_and_both_prune_functions(api, tiny_long, capsys):
    model, px, ref = tiny_long
    labels = ref["logits"].argmax(-1)
    batches = synth.make_batches(px, labels, 8)
    gm = copy.deepcopy(model).cuda()
    att, mlp = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None).fit()
    ref_scores = O.s1_scores(model, batches, "cpu", None, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(mlp, ref_scores)) <= SCORE_RTOL
    t = 64
    res = api.prune_vit_mlp_width(gm, n_to_prune_per_block=[t] * 3, strategy="act_l2", precomputed_importance=[s.float() for s in mlp],
                                  collect_masks=True, min_remaining=8)
    got = np.asarray(res["ffn_prune_masks"], dtype=np.uint8)
    listed = []
    for b, rs in enumerate(ref_scores):
        rs = rs.numpy()
        order = np.argsort(rs, kind="stable")
        want = np.zeros_like(got[b])
        want[order[:t]] = 1
        cut = np.sort(rs)[t - 1: t + 1].mean()
        for j in np.nonzero(got[b] != want)[0]:
            gap = abs(rs[j] - cut) / cut
            listed.append((b, int(j), float(gap)))
            assert gap <= SCORE_RTOL, f"block {b} neuron {j} flipped with relative gap {gap:.3e} to the cut"
    with capsys.disabled():
        print(f"\n[tiny_long] mask disagreements vs oracle (block, neuron, rel. gap to cut): {len(listed)} of {got.size}: {listed[:12]}")
    assert [fc1.out_features for fc1, _ in api._gather_mlp_pairs(gm)] == [256 - t] * 3
    res = api.prune_vit_attention_blocks(gm, 0.0, dataloader=batches, device="cuda", batch_limit=None, importance_mode="copy",
                                         show_progress=False, num_to_prune=1)
    assert len(res["pruned_indices"]) == 1 and res["final_metrics"] is not None
    assert api._count_attention_params_per_block(gm)[res["pruned_indices"][0]] == 0
    with torch.no_grad():
        tl = gm(pixel_values=px.cuda()).logits.float().cpu()
    el = api.engine_for(gm, "cuda", batch_hint=8).logits(px).cpu()
    assert (tl - el).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_long_captured_chains_equal_eager_launches(api, lib, tiny_long):
    model, px, ref = tiny_long
    labels = ref["logits"].argmax(-1)
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
def test_tiny_long_first_host_batch_split_gives_the_same_bits(api, lib, n):
    # T = 290 is even but gcd(290, 32) = 2: the parts are multiples of 16 images, so every image keeps its row offset
    # inside the 32-row score sub-tiles
    model = synth.make_vit("tiny_long", seed=0).cuda()
    px = synth.make_pixels(n, 136, seed=11)
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
def test_timm_shaped_long_model_pre_activation_scores(api):
    m = synth.TimmLikeViT(image=136, patch=8)
    px = synth.make_pixels(6, 136, seed=9)
    batches = [{"pixel_values": px[:4]}, {"pixel_values": px[4:]}]
    ref_scores = O.s1_scores(m, batches, "cpu", None, autocast=False)
    with torch.no_grad():
        ref_logits = m(px)
    gm = copy.deepcopy(m).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, ref_scores)) <= SCORE_RTOL
    logits = api.engine_for(gm, "cuda", batch_hint=6).logits(px).cpu()
    assert (logits - ref_logits).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(gm)


@pytest.mark.gpu
def test_tiny_long_odd_width_pruned_model_runs(api):
    model = synth.make_vit("tiny_long", seed=0).cuda()
    g_ = torch.Generator().manual_seed(3)
    imps = [torch.rand(256, generator=g_) for _ in range(3)]
    api.prune_vit_mlp_width(model, n_to_prune_per_block=[5, 61, 123], precomputed_importance=imps, min_remaining=8)
    api.prune_vit_attention_blocks(model, 0.0, selected_indices=[1], num_to_prune=1)
    px = synth.make_pixels(5, 136, seed=2)
    with torch.no_grad():
        ref = model(pixel_values=px.cuda()).logits.float().cpu()
    got = api.engine_for(model, "cuda", batch_hint=5).logits(px).cpu()
    assert (got - ref).abs().max().item() <= LOGIT_MAX_ABS
    scores = api._compute_ffn_activation_importance(model, [{"pixel_values": px}], device="cuda")
    assert [s.numel() for s in scores] == [251, 195, 133]
    ref_scores = O.s1_scores(copy.deepcopy(model).cpu(), [{"pixel_values": px}], "cpu", None, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(scores, ref_scores)) <= SCORE_RTOL
    api.release_engine(model)


@pytest.mark.gpu
def test_tiny_long_recycled_buffers_under_pool_poison():
    # engines built on recycled (0xFF-poisoned) device blocks give the bits of the first engine at T = 290
    code = """
import copy, sys, torch
sys.path.insert(0, %r)
from oracle import synth
synth.SHAPES.setdefault("tiny_long", %r)
from twossp_b200 import api, _lib as L
model = synth.make_vit("tiny_long", seed=0)
px = synth.make_pixels(12, 136, seed=1234)
labels = synth.self_labels(model, px)
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
assert L.load().tssp_trim_pool() == 0
print("recycled ok")
""" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), LONG_SHAPES["tiny_long"])
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    env = dict(os.environ, TSSP_POOL_POISON="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "recycled ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ----------------------------------------------------------------------------------------------- full size
@pytest.mark.gpu
def test_base384_against_oracle(api):
    """ViT-B/16 at 384^2 (T = 577) on 8 images: score contract, logits, Stage-2 on candidates 0, 6 and 11 against the
    oracle's skipped forward; the HF module goes through fit() and both prune functions."""
    model = synth.make_vit("base384", seed=0)
    n_img = 8
    px = synth.make_pixels(n_img, 384, seed=21)
    w = O.extract_weights(model)
    ref = O.vit_forward(w, px)
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, [{"pixel_values": px}], device="cuda")
    want = [nm.sum(0) / n_img for nm in ref["norms"]]
    rel = torch.cat([((a - b).abs() / b.abs()) for a, b in zip(got, want)])
    assert float(rel.mean()) <= 2e-3 and float(torch.quantile(rel, 0.999)) <= SCORE_RTOL and float(rel.max()) <= 1.5 * SCORE_RTOL, \
        (float(rel.mean()), float(rel.max()))
    logits = api.engine_for(gm, "cuda", batch_hint=n_img).logits(px).cpu()
    err = (logits - ref["logits"]).abs()
    assert err.max().item() <= LOGIT_MAX_ABS and err.mean().item() <= LOGIT_MEAN_ABS, (err.max().item(), err.mean().item())
    labels = ref["logits"].argmax(-1)
    lb = [{"pixel_values": px, "labels": labels}]
    base, cand, total = api.attention_removal_counts(gm, lb, "cuda", None)
    assert total == n_img and abs(base - n_img) <= 1
    for i in (0, 6, 11):
        skipped = O.vit_forward(w, px, skip_attention=(i,))["logits"]
        ours = api.engine_for(gm, "cuda", batch_hint=n_img).logits(px, skip_attn=[i]).cpu()
        assert (ours - skipped).abs().max().item() <= LOGIT_MAX_ABS
        assert int((ours.argmax(-1) == labels).sum()) == cand[i]
    att, mlp = api.B200Auto2SSPInterface(gm, lb, device="cuda", batch_limit=None).fit()
    assert att.shape == (12,) and all(torch.isfinite(s).all() for s in mlp)
    api.prune_vit_mlp_width(gm, n_to_prune_per_block=[1120] * 12, strategy="act_l2", precomputed_importance=[s.float() for s in mlp],
                            min_remaining=512)
    res = api.prune_vit_attention_blocks(gm, 0.0, dataloader=lb, device="cuda", batch_limit=None, importance_mode="copy",
                                         show_progress=False, num_to_prune=2)
    assert len(res["pruned_indices"]) == 2
    with torch.no_grad():
        tl = gm(pixel_values=px.cuda()).logits.float().cpu()
    assert (api.engine_for(gm, "cuda", batch_hint=n_img).logits(px).cpu() - tl).abs().max().item() <= LOGIT_MAX_ABS
    api.release_engine(gm, trim=True)


# ----------------------------------------------------------------------------------------------- no GPU needed
def _config(L, image, patch):
    cfg = L.TsspConfig()
    cfg.n_blocks, cfg.hidden, cfg.heads = 2, 128, 2
    cfg.image_size, cfg.patch_size, cfg.channels = image, patch, 3
    cfg.n_classes, cfg.head_hidden, cfg.max_images = 10, 0, 4
    cfg.score_point, cfg.cache_blocks, cfg.ln_eps = 0, 0, 1e-12
    for i in range(2):
        cfg.ffn_dims[i] = 256
        cfg.attn_present[i] = 1
    return cfg


def test_config_token_range_is_checked_before_any_device_query():
    import __graft_entry__ as g
    g.build()
    from twossp_b200 import _lib as L
    lib = L.load()
    h = C.c_void_p()
    # T = 577 passes validation; device 4096 exists nowhere, so creation fails on the device, not on the shape
    assert lib.tssp_create(C.byref(_config(L, 384, 16)), 4096, C.byref(h)) != 0
    msg = lib.tssp_last_error().decode()
    assert "tokens per image" not in msg and "device" in msg.lower(), msg
    # T = 33^2 + 1 = 1090 is past the range: rejected by the configuration check, which names it
    assert lib.tssp_create(C.byref(_config(L, 264, 8)), 4096, C.byref(h)) != 0
    msg = lib.tssp_last_error().decode()
    assert "T=1090" in msg and "[32,1025]" in msg, msg
