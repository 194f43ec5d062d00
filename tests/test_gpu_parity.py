"""Parity of the CUDA path (through the C ABI of libtssp_b200.so) against the CPU oracle and the golden vectors
recorded from the unmodified reference. Needs a B200: run with `-m gpu`.

Tolerances (stated once, used below):
  * integer / index / byte results (gather, masks given identical scores, top-1 counts of identical logits,
    im2col, argmax): bit-exact;
  * Stage-1 scores of the bf16-operand path vs the fp32 oracle: <= 1e-2 relative (BASELINE.json north_star);
  * logits vs the fp32 oracle: max-abs <= 3e-2, mean-abs <= 5e-3 on logits of std ~0.5 (SURVEY.md section 8c: the
    reference's own bf16 CPU path is 0.024 / 0.004 away from its fp32 path);
  * end-to-end masks: identical except neurons whose oracle score lies within 1e-2 relative of the block's cut
    value, which are listed;
  * Stage-2 correct-counts: within +-DELTA images of the oracle, selection identical wherever count gaps > DELTA.
"""
import copy
import os
import sys

import numpy as np
import pytest
import torch

from oracle import synth
from oracle import twossp_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import attention_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-2
LOGIT_MAX_ABS = 3e-2
LOGIT_MEAN_ABS = 5e-3
DELTA = 2


@pytest.fixture(scope="module", autouse=True)
def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    torch.cuda.set_device(0)


@pytest.fixture(scope="module")
def lib():
    from twossp_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ops():
    from twossp_b200 import ops as o
    return o


@pytest.fixture(scope="module")
def api():
    from twossp_b200 import api as a
    return a


@pytest.fixture(params=[1, 2], ids=["cta1", "pair"])
def gemm_form(request, lib):
    """Run a GEMM test in both tile forms (single CTA, CTA pair), then restore the automatic choice."""
    lib.check(lib.load().tssp_set_gemm_form(request.param))
    yield request.param
    lib.check(lib.load().tssp_set_gemm_form(0))


def _unpack(bits, width):
    return np.unpackbits(bits, axis=-1)[..., :width]


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (300, 264, 200), (7, 1000, 384), (197 * 16, 768, 3072),
                                   (197 * 8, 384, 1536), (197 * 8, 384, 384), (333, 128, 128), (600, 640, 256), (300, 192, 72), (515, 960, 128)])  # 128- and 192-column tiles
@pytest.mark.parametrize("reduce_add", [False, True])
def test_gemm_fp32_epilogue(ops, lib, gemm_form, M, N, K, reduce_add):
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    base = torch.randn(M, N, generator=g).cuda()
    out = base.clone() if reduce_add else torch.full((M, N), float("nan"), device="cuda")
    ops.gemm(lib.EPI_F32, a, w, out, bias, reduce_add=reduce_add)
    ref = a.double() @ w.double().t() + bias.double() + (base.double() if reduce_add else 0)
    assert torch.isfinite(out).all()
    assert (out.double() - ref).abs().max().item() <= 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("mode", ["plain", "gelu"])
@pytest.mark.parametrize("M,N,K", [(256, 512, 128), (300, 264, 200), (197 * 8, 2304, 768)])
def test_gemm_bf16_epilogue(ops, lib, gemm_form, mode, M, N, K):
    g = torch.Generator().manual_seed(M * 3 + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.gemm(lib.EPI_BF16 if mode == "plain" else lib.EPI_BF16_GELU, a, w, out, bias)
    ref = a.float() @ w.float().t() + bias
    if mode == "gelu":
        ref = torch.nn.functional.gelu(ref)
    # one bf16 rounding of the fp32 result (half an ulp <= 2^-8 relative) + the GELU approximation (<= 1.6e-4 relative,
    # gemm_tcgen05.cuh: gelu_erf_x2), which can move a value across a rounding boundary
    assert torch.isfinite(out.float()).all()
    assert ((out.float() - ref).abs() <= ref.abs() * (2 ** -8 + 2e-4) + 1e-5).all()


@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("n_img,T,N,K", [(9, 37, 256, 128), (5, 65, 520, 128), (16, 197, 3072, 768), (3, 32, 264, 64)])
def test_gemm_score_epilogue(ops, lib, gemm_form, pre, n_img, T, N, K):
    M = n_img * T
    g = torch.Generator().manual_seed(T + N)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().cuda()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    bias = torch.randn(N, generator=g).cuda()
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    partials = torch.full((2 * ((M + 31) // 32), N), float("nan"), device="cuda")
    ops.gemm(lib.EPI_BF16_GELU_SCORE_PRE if pre else lib.EPI_BF16_GELU_SCORE, a, w, out, bias, partials=partials, tokens_per_image=T)
    scores = torch.zeros(N, device="cuda")
    norms = ops.score_finish(partials, n_img, T, N, scores)
    z = a.float() @ w.float().t() + bias
    act = torch.nn.functional.gelu(z)
    hooked = z if pre else act
    want = hooked.reshape(n_img, T, N).double().pow(2).sum(1).sqrt()
    assert ((out.float() - act).abs() <= act.abs() * (2 ** -8 + 2e-4) + 1e-5).all()
    rel = ((norms.double() - want).abs() / want.clamp_min(1e-9)).max().item()
    assert rel <= 5e-3, rel          # norm of bf16-stored activations vs norm of fp32 activations
    assert torch.allclose(scores.double(), norms.double().sum(0), rtol=1e-5)
    if not pre:
        # the stored activations reproduce the norms exactly up to fp32 summation order
        stored = out.float().reshape(n_img, T, N).double().pow(2).sum(1).sqrt()
        assert ((norms.double() - stored).abs() / stored.clamp_min(1e-9)).max().item() <= 1e-5


def test_layernorm(ops):
    # every width with a persistent instance (128-wide and 256-wide slabs, gamma/beta in registers or re-read), few rows and
    # more rows than the persistent grid holds warps; two calls each: consecutive launches walk the rows in opposite directions
    for D in (128, 256, 384, 512, 640, 768, 896, 1024):
        for rows in (333, 20011):
            x = torch.randn(rows, D, device="cuda") * 3 + 1
            g_, b_ = torch.randn(D, device="cuda"), torch.randn(D, device="cuda")
            ref = torch.nn.functional.layer_norm(x, (D,), g_, b_, 1e-12)
            out1 = ops.layernorm(x, g_, b_, 1e-12)
            out2 = ops.layernorm(x, g_, b_, 1e-12)
            assert torch.equal(out1, out2)
            assert ((out1.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-4).all()
    x = torch.randn(5 * 37, 256, device="cuda")
    out = ops.layernorm(x, torch.ones(256, device="cuda"), torch.zeros(256, device="cuda"), 1e-6, row_stride=37 * 256, rows=5)
    ref = torch.nn.functional.layer_norm(x.view(5, 37, 256)[:, 0], (256,), eps=1e-6)
    assert ((out.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-4).all()


# the short-sequence kernel at the edges of its structure: 16-31 keys (one 16- or 32-column chunk), 127 / 128 / 129 (one
# vs two query tiles), 144 (a 16-wide last chunk), 192 / 193 and 208 (its limit); n makes >= 1e5 outputs for the bias check
_SHORT_T = [(R.images_for(T, h), T, h) for T, h in ((16, 2), (17, 3), (31, 1), (33, 4), (127, 2), (128, 3), (129, 2),
                                                    (144, 6), (192, 2), (193, 3), (208, 2))]


@pytest.mark.parametrize("scale", [1.0, 0.05, 3.0])   # 3.0 makes the Cauchy-Schwarz shift too loose: exact two-pass route
@pytest.mark.parametrize("n,T,heads", [(3, 37, 2), (2, 65, 4), (4, 197, 12), (2, 208, 6), (1, 32, 1), (130, 197, 12)] + _SHORT_T)
def test_attention(ops, n, T, heads, scale):
    qkv = R.iid_qkv(n, T, heads, scale, seed=T * 13 + n, device="cuda")
    R.run_and_check(ops, qkv, n, T, heads, scale=scale)


# units (image, head) just past one and two per SM: a CTA's two chains get unequal tile counts (the `other_tiles`
# alternation of the two chains' softmax phases)
@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("extra", ["sms+1", "2sms-1", "2sms+1"])
def test_attention_at_unit_counts_around_the_sm_count(ops, extra, scale):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = {"sms+1": sms + 1, "2sms-1": 2 * sms - 1, "2sms+1": 2 * sms + 1}[extra]
    qkv = R.iid_qkv(n, 197, 1, scale, seed=n, device="cuda")
    R.run_and_check(ops, qkv, n, 197, 1, scale=scale)


def test_im2col_is_bit_exact(ops):
    for (n, C, H, P) in ((2, 3, 48, 8), (3, 3, 224, 16)):
        px = torch.randn(n, C, H, H, device="cuda")
        out = ops.im2col(px, P)
        G = H // P
        ref = px.view(n, C, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(n, G * G, C * P * P)
        ref = torch.cat([torch.zeros(n, 1, C * P * P, device="cuda"), ref], 1).reshape(n * (G * G + 1), -1).bfloat16()
        assert torch.equal(out, ref)


@pytest.mark.parametrize("F,D,k", [(3072, 768, 1952), (256, 128, 101), (1536, 384, 960), (4096, 1024, 2026), (3072, 768, 3071), (3072, 768, 1)])
def test_gather_is_bit_exact(ops, F, D, k):
    w1, b1, w2 = torch.randn(F, D, device="cuda"), torch.randn(F, device="cuda"), torch.randn(D, F, device="cuda")
    keep = torch.sort(torch.randperm(F, device="cuda")[:k])[0]
    o1, ob, o2 = ops.ffn_gather(w1, b1, w2, keep)
    assert torch.equal(o1, w1[keep]) and torch.equal(ob, b1[keep]) and torch.equal(o2, w2[:, keep])
    o1, ob, o2 = ops.ffn_gather(w1, None, w2, keep)
    assert ob is None and torch.equal(o1, w1[keep])


def test_gather_round_trip_at_full_size(ops):
    # size-independent property at ViT-L size: scattering the kept and the dropped parts back restores the matrix
    F, D = 4096, 1024
    w1, b1, w2 = torch.randn(F, D, device="cuda"), torch.randn(F, device="cuda"), torch.randn(D, F, device="cuda")
    perm = torch.randperm(F, device="cuda")
    keep, drop = torch.sort(perm[:2026])[0], torch.sort(perm[2026:])[0]
    k1, kb, k2 = ops.ffn_gather(w1, b1, w2, keep)
    d1, db, d2 = ops.ffn_gather(w1, b1, w2, drop)
    r1, rb, r2 = torch.empty_like(w1), torch.empty_like(b1), torch.empty_like(w2)
    r1[keep], r1[drop], rb[keep], rb[drop] = k1, d1, kb, db
    r2[:, keep], r2[:, drop] = k2, d2
    assert torch.equal(r1, w1) and torch.equal(rb, b1) and torch.equal(r2, w2)


def _gather_case(F, D, k, bias=True, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    w1 = torch.randn(F, D, device="cuda", generator=g)
    b1 = torch.randn(F, device="cuda", generator=g) if bias else None
    w2 = torch.randn(D, F, device="cuda", generator=g)
    keep = torch.sort(torch.randperm(F, device="cuda", generator=g)[:k])[0]
    return w1, b1, w2, keep


def test_gather_batch_is_bit_exact_on_ragged_blocks(ops):
    # one launch over blocks of different widths: aligned (bulk-copy route), odd F (scalar staging), odd k (scalar
    # stores), k = 1, k = F, a block without bias
    D = 384
    shapes = [(1536, 960, True), (1536, 576, True), (1533, 700, True), (1536, 961, False), (1530, 1, True), (264, 264, True),
              (2411, 1207, True), (1536, 1535, True)]
    blocks = [_gather_case(F, D, k, bias, seed=i) for i, (F, k, bias) in enumerate(shapes)]
    outs = ops.ffn_gather_batch(blocks)
    assert len(outs) == len(blocks)
    for (w1, b1, w2, keep), (o1, ob, o2) in zip(blocks, outs):
        assert torch.equal(o1, w1[keep]) and torch.equal(o2, w2[:, keep])
        assert (ob is None) if b1 is None else torch.equal(ob, b1[keep])
        assert o1.shape == (keep.numel(), D) and o2.shape == (D, keep.numel())


def test_gather_batch_matches_per_block_calls_and_chunks_long_models(ops):
    # 40 blocks > the 32 one launch takes: the library chunks; results equal the per-block entry point
    D = 128
    blocks = [_gather_case(512, D, 100 + 7 * i, seed=100 + i) for i in range(40)]
    outs = ops.ffn_gather_batch(blocks)
    for (w1, b1, w2, keep), (o1, ob, o2) in zip(blocks, outs):
        s1, sb, s2 = ops.ffn_gather(w1, b1, w2, keep)
        assert torch.equal(o1, s1) and torch.equal(ob, sb) and torch.equal(o2, s2)
        assert torch.equal(o1, w1[keep]) and torch.equal(o2, w2[:, keep])


@pytest.mark.parametrize("B,F,D,k", [(12, 3072, 768, 1952), (24, 4096, 1024, 2026)])
def test_gather_batch_at_baseline_sizes(ops, B, F, D, k):
    # BASELINE configs 3 and 4 (ViT-B/16 keep 1952, ViT-L/16 keep 2026), all blocks in one launch
    blocks = [_gather_case(F, D, k, seed=b) for b in range(B)]
    outs = ops.ffn_gather_batch(blocks)
    for (w1, b1, w2, keep), (o1, ob, o2) in zip(blocks, outs):
        assert torch.equal(o1, w1[keep]) and torch.equal(ob, b1[keep]) and torch.equal(o2, w2[:, keep])


def test_gather_batch_rejects_bad_arguments(ops):
    from twossp_b200._lib import TsspError
    w1, b1, w2, keep = _gather_case(256, 128, 64)
    with pytest.raises(ValueError):
        ops.ffn_gather_batch([(w1, b1, w2, keep), (torch.randn(256, 64, device="cuda"), None, torch.randn(64, 256, device="cuda"), keep)])
    with pytest.raises(TsspError):
        ops.ffn_gather_batch([(w1, b1, w2, keep[:0])])  # k = 0
    assert ops.ffn_gather_batch([]) == []


def test_argmax_count(ops):
    logits = torch.randn(77, 1000, device="cuda")
    logits[5, 10] = logits[5, 20] = 99.0
    labels = logits.argmax(-1)
    labels[::3] = 0
    preds, correct = ops.argmax_count(logits, labels)
    ref = logits.argmax(-1)
    assert torch.equal(preds.long(), ref) and int(preds[5]) == 10
    assert int(correct.item()) == int((ref == labels).sum().item())


# ----------------------------------------------------------------------------------------------- engine vs oracle
def _setup(name, meta, golden_dir):
    m = meta[name]
    model = synth.make_vit(name, seed=0)
    assert synth.state_sha(model) == m["state_sha"]
    pixels = synth.make_pixels(m["n_img"], synth.SHAPES[name][0], seed=1234)
    g = np.load(f"{golden_dir}/{name}_ref.npz")
    labels = torch.from_numpy(g["labels"].copy())
    return model, pixels, labels, g, m


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_logits_match_fp32_reference(api, name, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    eng = api.engine_for(copy.deepcopy(model).cuda(), "cuda", batch_hint=m["batch"])
    got = eng.logits(pixels).cpu().numpy()
    err = np.abs(got - g["logits_fp32"])
    assert err.max() <= LOGIT_MAX_ABS and err.mean() <= LOGIT_MEAN_ABS, (err.max(), err.mean())
    # device-resident input gives the same bits as host input
    assert np.array_equal(eng.logits(pixels.cuda()).cpu().numpy(), got)


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_s1_scores_match_reference(api, name, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    batches = synth.make_batches(pixels, None, m["batch"])
    got = api._compute_ffn_activation_importance(copy.deepcopy(model).cuda(), batches, device="cuda")
    assert len(got) == g["scores_fp32"].shape[0] and all(t.device.type == "cpu" and t.dtype == torch.float32 for t in got)
    got = torch.stack(got).numpy()
    rel = np.abs(got - g["scores_fp32"]) / np.abs(g["scores_fp32"])
    assert rel.max() <= SCORE_RTOL, rel.max()
    # the reference's own bf16 CPU path is further from its fp32 path than we are
    ref_rel = np.abs(g["scores_asis"] - g["scores_fp32"]) / np.abs(g["scores_fp32"])
    assert rel.mean() <= ref_rel.mean()


def test_s1_scores_do_not_depend_on_the_gemm_form(api, lib, golden_meta, golden_dir):
    """Single-CTA and CTA-pair tiles run the same K order per output element: Stage-1 scores and logits agree to fp32
    rounding, whatever the dispatch picks per GEMM."""
    model, pixels, labels, g, m = _setup("base", golden_meta, golden_dir)
    batches = synth.make_batches(pixels, None, m["batch"])
    out = {}
    for form in (1, 2):
        lib.check(lib.load().tssp_set_gemm_form(form))
        try:
            gm = copy.deepcopy(model).cuda()
            out[form] = (torch.stack(api._compute_ffn_activation_importance(gm, batches, device="cuda")),
                         api.engine_for(gm, "cuda", batch_hint=m["batch"]).logits(pixels).cpu())
            api.release_engine(gm)
        finally:
            lib.check(lib.load().tssp_set_gemm_form(0))
    rel = ((out[1][0] - out[2][0]).abs() / out[1][0].abs()).max().item()
    assert rel <= 1e-5, rel
    assert (out[1][1] - out[2][1]).abs().max().item() <= 1e-3
    for form in (1, 2):
        r = (out[form][0].numpy() - g["scores_fp32"]) / g["scores_fp32"]
        assert np.abs(r).max() <= SCORE_RTOL


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_end_to_end_masks_differ_only_at_near_ties(api, name, golden_meta, golden_dir, capsys):
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    batches = synth.make_batches(pixels, None, m["batch"])
    gm = copy.deepcopy(model).cuda()
    scores = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    nb = len(scores)
    res = api.prune_vit_mlp_width(gm, n_to_prune_per_block=[m["t_prune"]] * nb, strategy="act_l2",
                                  precomputed_importance=[s.float() for s in scores], collect_masks=True, min_remaining=8)
    want = _unpack(g["masks_bits"], int(g["mask_width"]))
    got = np.asarray(res["ffn_prune_masks"], dtype=np.uint8)
    assert got.shape == want.shape and (got.sum(1) == m["t_prune"]).all()
    listed = []
    for b in range(nb):
        ref_scores = g["scores_fp32"][b]
        cut = np.sort(ref_scores)[m["t_prune"] - 1: m["t_prune"] + 1].mean()   # between last pruned and first kept
        for j in np.nonzero(got[b] != want[b])[0]:
            gap = abs(ref_scores[j] - cut) / cut
            listed.append((b, int(j), float(gap)))
            assert gap <= SCORE_RTOL, f"block {b} neuron {j} flipped with relative gap {gap:.3e} to the cut"
    with capsys.disabled():
        print(f"\n[{name}] mask disagreements vs reference (block, neuron, rel. gap to cut): {len(listed)} of {got.size}: {listed[:12]}")
    assert len(listed) <= 0.02 * got.size


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_masks_and_gather_bit_exact_given_reference_scores(api, name, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    gm = copy.deepcopy(model).cuda()
    scores = [torch.from_numpy(s.copy()) for s in g["scores_fp32"]]
    res = api.prune_vit_mlp_width(gm, n_to_prune_per_block=[m["t_prune"]] * len(scores), strategy="act_l2",
                                  precomputed_importance=scores, collect_masks=True, min_remaining=8)
    assert res["model"] is gm
    want = _unpack(g["masks_bits"], int(g["mask_width"]))
    assert np.array_equal(np.asarray(res["ffn_prune_masks"], dtype=np.uint8), want)
    for row, idx in zip(want, res["ffn_pruned_indices"]):
        assert np.array_equal(np.nonzero(row)[0], np.asarray(idx))
    pairs = api._gather_mlp_pairs(gm)
    assert synth.sha256_tensors([t for a, b in pairs for t in (a.weight, a.bias, b.weight)]) == m["gathered_sha"]
    assert all(a.out_features == w and b.in_features == w and a.weight.requires_grad for (a, b), w in zip(pairs, m["pruned_widths"]))
    # model-out is still an ordinary torch module, and the engine follows the mutation
    with torch.no_grad():
        torch_logits = gm(pixel_values=pixels[:4].cuda()).logits.float().cpu()
    eng_logits = api.engine_for(gm, "cuda", batch_hint=4).logits(pixels[:4]).cpu()
    assert (torch_logits - eng_logits).abs().max().item() <= LOGIT_MAX_ABS


def test_prune_api_contract(api):
    model = synth.make_vit("tiny", seed=0).cuda()
    with pytest.raises(ValueError):
        api.prune_vit_mlp_width(model, n_to_prune_per_block=[1, 2])
    with pytest.raises(ValueError):
        api.prune_vit_mlp_width(model)
    with pytest.raises(AssertionError):
        api.prune_vit_mlp_width(model, sparsity=1.0)
    with pytest.raises(ValueError):
        api.prune_vit_mlp_width(model, sparsity=0.1, precomputed_importance=[torch.zeros(256)])
    with pytest.raises(RuntimeError):
        api.prune_vit_mlp_width(model, sparsity=0.1, precomputed_importance=[torch.zeros(5)] * 3)
    with pytest.raises(RuntimeError):
        api.prune_vit_mlp_width(model, sparsity=0.1, strategy="act_l2")
    with pytest.raises(ValueError):
        api.prune_vit_mlp_width(model, sparsity=0.1, strategy="nope")
    res = api.prune_vit_mlp_width(model, n_to_prune_per_block=[0, 5, 0], collect_masks=True, min_remaining=8)
    assert len(res["ffn_prune_masks"]) == 1 and sum(res["ffn_prune_masks"][0]) == 5   # skipped blocks leave no entry
    # weight-L1 strategy against the oracle
    ref = O.s1_prune(synth.make_vit("tiny", seed=0), sparsity=0.25, strategy="l1", min_remaining=8)
    got = api.prune_vit_mlp_width(synth.make_vit("tiny", seed=0).cuda(), sparsity=0.25, strategy="l1", min_remaining=8, collect_masks=True)
    assert got["ffn_prune_masks"] == ref["ffn_prune_masks"]
    # +-1 scores of the apply_mask_prune flow (experiments/vit_pruning/apply_mask_prune.py:259-280)
    g_ = torch.Generator().manual_seed(7)
    pm = [(torch.rand(256, generator=g_) < 0.3) for _ in range(3)]
    imp = [torch.where(m_, torch.tensor(-1.0), torch.tensor(1.0)) for m_ in pm]
    got = api.prune_vit_mlp_width(synth.make_vit("tiny", seed=0).cuda(), n_to_prune_per_block=[int(m_.sum()) for m_ in pm],
                                  precomputed_importance=imp, collect_masks=True, min_remaining=8)
    assert all(torch.equal(torch.tensor(a, dtype=torch.bool), m_) for a, m_ in zip(got["ffn_prune_masks"], pm))


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_stage2_counts_and_selection(api, name, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    batches = synth.make_batches(pixels, labels, m["batch"])
    gm = copy.deepcopy(model).cuda()
    base, cand, total = api.attention_removal_counts(gm, batches, "cuda", None)
    ref_imp = g["att_importance_fp32"]
    ref_base = round(m["s2"]["baseline_acc"] * m["n_img"])
    ref_cand = [ref_base - round(float(x) * m["n_img"]) for x in ref_imp]
    assert total == m["n_img"] and abs(base - ref_base) <= DELTA
    assert all(abs(a - b) <= DELTA for a, b in zip(cand, ref_cand)), (cand, ref_cand)
    # suffix recompute == full recompute with the block skipped: identical counts, not just close
    for i in range(len(cand)):
        c, t = api._top1_counts(gm, batches, "cuda", None, skip_attn=[i])
        assert (c, t) == (cand[i], total), i
    assert api._top1_counts(gm, batches, "cuda", None) == (base, total)
    # interface: impacts and their order
    iface = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None)
    att = iface._compute_att_depth_importance()
    assert att.dtype == torch.float32 and att.shape == (len(cand),) and att.device.type == "cpu"
    k = m["s2"]["num_to_prune"]
    ours = sorted(range(len(cand)), key=lambda i: float(att[i]))[:k]
    theirs = sorted(range(len(cand)), key=lambda i: float(ref_imp[i]))[:k]
    gaps_ok = all(abs(ref_cand[i] - ref_cand[j]) > DELTA for i in theirs for j in range(len(cand)) if j not in theirs)
    if gaps_ok:
        assert sorted(ours) == sorted(theirs)


def test_prune_attention_blocks_api(api, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup("tiny", golden_meta, golden_dir)
    batches = synth.make_batches(pixels, labels, m["batch"])
    gm = copy.deepcopy(model).cuda()
    assert api.prune_vit_attention_blocks(gm, 0.0)["pruned_indices"] == []
    with pytest.raises(AssertionError):
        api.prune_vit_attention_blocks(gm, 1.0)
    res = api.prune_vit_attention_blocks(gm, 0.0, dataloader=batches, device="cuda", batch_limit=None, importance_mode="copy",
                                         show_progress=False, num_to_prune=1)
    assert res["model"] is gm and len(res["pruned_indices"]) == 1
    assert res["original_metrics"] is not None and res["final_metrics"] is not None
    idx = res["pruned_indices"][0]
    assert api._count_attention_params_per_block(gm)[idx] == 0
    # final metric is the top-1 of the mutated module, through torch and through the engine alike
    with torch.no_grad():
        tl = gm(pixel_values=pixels.cuda()).logits.float().argmax(-1).cpu()
    assert abs(float((tl == labels).float().mean()) - res["final_metrics"]) <= DELTA / m["n_img"]
    # explicit indices keep at least one block and are returned sorted (src/vit_pruning.py:444,451-456,517)
    gm2 = copy.deepcopy(model).cuda()
    res2 = api.prune_vit_attention_blocks(gm2, 0.99, selected_indices=[2, 0, 1, 7])
    assert res2["pruned_indices"] == [0, 1] and res2["original_metrics"] is None and res2["final_metrics"] is None
    res3 = api.prune_vit_attention_blocks(copy.deepcopy(model).cuda(), 0.34, importance_mode="heuristic")
    assert res3["pruned_indices"] == [0]
    # scoring a model that already lost an attention block (README flow: S2 after S1 on the mutated model)
    s = api._compute_ffn_activation_importance(gm2, batches, device="cuda")
    ref = O.s1_scores(_bypass_cpu(model, [0, 1]), batches, "cpu", None, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(s, ref)) <= SCORE_RTOL


def _bypass_cpu(model, idx):
    m = copy.deepcopy(model)
    for i in idx:
        O.remove_attention(m, i)
    return m


def test_interface_fit_contract(api, golden_meta, golden_dir):
    model, pixels, labels, g, m = _setup("tiny", golden_meta, golden_dir)
    batches = synth.make_batches(pixels, labels, m["batch"])
    iface = api.B200Auto2SSPInterface(copy.deepcopy(model).cuda(), batches, device="cuda", batch_limit=2)
    assert iface.att_prune_type == api.PruningTypes.DEPTH and iface.mlp_prune_type == api.PruningTypes.WIDTH
    att, mlp = iface.fit()
    assert isinstance(att, torch.Tensor) and att.dim() == 1 and att.numel() == 3
    assert isinstance(mlp, list) and len(mlp) == 3 and all(t.dim() == 1 and t.numel() == 256 for t in mlp)
    # batch_limit counts batches (src/vit_pruning.py:175): 2 batches of 4 images
    ref = O.s1_scores(model, batches, "cpu", 2, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(mlp, ref)) <= SCORE_RTOL
    # no dataloader: heuristic depth scores + weight-L1 FFN scores (mask_conjunction.py:289-304)
    att2, mlp2 = api.B200Auto2SSPInterface(copy.deepcopy(model).cuda(), None, device="cuda").fit()
    assert att2.tolist() == [0.0, 1.0, 1.0]
    assert torch.allclose(mlp2[0], model.vit.encoder.layer[0].intermediate.dense.weight.abs().sum(1), rtol=1e-6)


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_fit_fused_pass_equals_the_two_separate_passes(api, golden_meta, golden_dir, name):
    # fit() takes the Stage-1 scores from the Stage-2 baseline pass (tssp_s2_batch with TSSP_S2_WITH_SCORES): same counts,
    # and the SAME BITS as a separate Stage-1 sweep over the same batches
    model, pixels, labels, g, m = _setup(name, golden_meta, golden_dir)
    batches = synth.make_batches(pixels, labels, m["batch"])
    gm = copy.deepcopy(model).cuda()
    fused = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None)
    att_f, mlp_f = fused.fit()
    plain = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None, fuse_passes=False)
    att_p, mlp_p = plain.fit()
    assert torch.equal(att_f, att_p) and fused.last_counts == plain.last_counts
    assert len(mlp_f) == len(mlp_p) and all(torch.equal(a, b) for a, b in zip(mlp_f, mlp_p))
    assert all(t.device.type == "cpu" and t.dtype == torch.float32 for t in mlp_f)
    # the stand-alone methods never reuse a fused result
    assert fused._fused_mlp is None and not fused._fusing
    sep = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert all(torch.equal(a, b) for a, b in zip(mlp_f, sep))
    # function API: the fourth return value, with a batch limit
    base, cand, total, scores = api.attention_removal_counts(gm, batches, "cuda", 1, with_scores=True)
    assert total == m["batch"] and all(torch.equal(a, b) for a, b in zip(scores, api._compute_ffn_activation_importance(gm, batches, "cuda", 1)))
    assert (base, cand, total) == api.attention_removal_counts(gm, batches, "cuda", 1)
    # empty loader: zeros, as Stage 1 returns for it (src/vit_pruning.py:197-198)
    b0, c0, t0, s0 = api.attention_removal_counts(gm, [], "cuda", None, with_scores=True)
    assert (b0, t0) == (0, 0) and all(float(t.abs().sum()) == 0.0 for t in s0)


def test_recycled_engine_buffers_do_not_leak_state():
    # tssp_destroy parks device buffers in a pool and the next engine of the same shape gets them back. With
    # TSSP_POOL_POISON=1 parked blocks are filled with 0xFF bytes (NaNs): every result of an engine built on recycled
    # blocks must equal, bit for bit, the result of the first engine (which got fresh memory).
    import subprocess
    import sys
    code = """
import copy, sys, torch
sys.path.insert(0, %r)
from oracle import synth
from twossp_b200 import api, _lib as L
model = synth.make_vit("tiny", seed=0)
px = synth.make_pixels(12, 48, seed=1234)
labels = synth.self_labels(model, px)
batches = synth.make_batches(px, labels, 4)
outs = []
for rep in range(3):
    gm = copy.deepcopy(model).cuda()
    iface = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None)
    att, mlp = iface.fit()
    logits = api.engine_for(gm, "cuda", batch_hint=4, need_cache=True).logits(px).cpu()
    outs.append((att, mlp, iface.last_counts, logits))
    api.release_engine(gm)
for att, mlp, counts, logits in outs[1:]:
    assert torch.equal(att, outs[0][0]) and counts == outs[0][2] and torch.equal(logits, outs[0][3])
    assert all(torch.equal(a, b) for a, b in zip(mlp, outs[0][1])) and all(bool(torch.isfinite(t).all()) for t in mlp)
assert L.load().tssp_trim_pool() == 0
print("recycled ok")
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TSSP_POOL_POISON="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "recycled ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_edge_batches(api):
    model = synth.make_vit("tiny", seed=0)
    gm = copy.deepcopy(model).cuda()
    assert all(float(t.abs().sum()) == 0 and t.numel() == 256 for t in api._compute_ffn_activation_importance(gm, [], device="cuda"))
    px = synth.make_pixels(11, 48, seed=5)
    ragged = [{"pixel_values": px[:1]}, {"pixel_values": px[1:8]}, {"pixel_values": px[8:11]}]
    got = api._compute_ffn_activation_importance(gm, ragged, device="cuda")
    ref = O.s1_scores(model, ragged, "cpu", None, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, ref)) <= SCORE_RTOL
    # re-batching moves images to other row offsets inside the 32-row sub-tiles, which only re-associates fp32 sums
    whole = api._compute_ffn_activation_importance(gm, [{"pixel_values": px}], device="cuda")
    assert all(torch.allclose(a, b, rtol=1e-5) for a, b in zip(got, whole))
    again = api._compute_ffn_activation_importance(gm, [{"pixel_values": px}], device="cuda")
    assert all(torch.equal(a, b) for a, b in zip(again, whole))      # same batching: same bits, run to run
    with pytest.raises(ValueError):
        api._compute_ffn_activation_importance(gm, [{"pixel_values": torch.zeros(2, 3, 32, 32)}], device="cuda")
    assert api.evaluate_top1(gm, [], device="cuda") == 0.0


@pytest.mark.parametrize("name,n", [("tiny", 160), ("tiny", 128), ("small", 256)])
def test_first_host_batch_split_gives_the_same_bits(api, lib, name, n):
    """The first HOST batch after a reset is copied and swept as two sub-batches (engine.cu: s1_head_images) so that
    compute starts under the copy; the split keeps every image on its 32-row sub-tile alignment, so per-image norms and
    the accumulated scores carry the same bits as the unsplit (device-resident) batch."""
    model = synth.make_vit(name, seed=0).cuda()
    px = synth.make_pixels(n, synth.SHAPES[name][0], seed=11)
    eng = api.engine_for(model, "cuda", batch_hint=n)
    lib.check(lib.load().tssp_set_gemm_form(1))            # one tile form for both runs (the dispatch looks at M)
    try:
        out = {}
        for where in ("device", "host"):
            eng.s1_reset()
            src = px.cuda() if where == "device" else px.pin_memory()
            norms = torch.zeros(n, sum(eng.ffn_dims), device="cuda")
            eng.s1_batch(src, img_norms=norms)
            eng.s1_batch(src[: n // 2])                     # a second batch: never split
            out[where] = (norms.cpu(), eng.s1_score_sums().clone())
    finally:
        lib.check(lib.load().tssp_set_gemm_form(0))
    assert float(out["device"][0].abs().min()) > 0
    assert torch.equal(out["device"][0], out["host"][0])
    assert torch.equal(out["device"][1], out["host"][1])


# ----------------------------------------------------------------------------------------------- timm-shaped model
def test_timm_shaped_model_pre_activation_scores(api):
    """timm layout: fused qkv, eps 1e-6, and the hook sits on mlp.fc1, i.e. BEFORE the GELU (src/vit_pruning.py:135)."""
    m = synth.TimmLikeViT()
    px = synth.make_pixels(6, 48, seed=9)
    batches = [{"pixel_values": px[:4]}, {"pixel_values": px[4:]}]
    ref_scores = O.s1_scores(m, batches, "cpu", None, autocast=False)
    with torch.no_grad():
        ref_logits = m(px)
        labels = ref_logits.argmax(-1)
    gm = copy.deepcopy(m).cuda()
    got = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(got, ref_scores)) <= SCORE_RTOL
    logits = api.engine_for(gm, "cuda", batch_hint=6).logits(px).cpu()
    assert (logits - ref_logits).abs().max().item() <= LOGIT_MAX_ABS
    lb = [{"pixel_values": px, "labels": labels}]
    base, cand, total = api.attention_removal_counts(gm, lb, "cuda", None)
    rb, rc, rt = O.s2_candidate_scores(m, lb, "cpu", None, autocast=False)
    assert total == rt and abs(base - rb) <= DELTA and all(abs(a - b) <= DELTA for a, b in zip(cand, rc))
    res = api.prune_vit_attention_blocks(gm, 0.5, selected_indices=[1])
    assert res["pruned_indices"] == [1] and api._count_attention_params_per_block(gm) [1] == 0
    with torch.no_grad():
        after = gm(px.cuda()).float().cpu()      # the mutated timm-shaped module still runs in torch
    ref_after = copy.deepcopy(m)
    O.remove_attention(ref_after, 1)
    with torch.no_grad():
        assert torch.allclose(after, ref_after(px), atol=1e-3)


# ----------------------------------------------------------------------------------------------- full-size properties
def test_full_size_properties_vit_base(api):
    """BASELINE config 3 sizes (ViT-B/16, batches of 128): properties that need no oracle run."""
    model = synth.make_vit("base", seed=0).cuda()
    px = synth.make_pixels(256, 224, seed=77)
    a = torch.stack(api._compute_ffn_activation_importance(model, [{"pixel_values": px[:128]}], device="cuda"))
    b = torch.stack(api._compute_ffn_activation_importance(model, [{"pixel_values": px[128:]}], device="cuda"))
    ab = torch.stack(api._compute_ffn_activation_importance(model, [{"pixel_values": px[:128]}, {"pixel_values": px[128:]}], device="cuda"))
    assert torch.isfinite(ab).all() and (ab > 0).all()
    assert torch.allclose(ab, (a + b) / 2, rtol=1e-5)          # additivity over images
    again = torch.stack(api._compute_ffn_activation_importance(model, [{"pixel_values": px}], device="cuda"))
    assert torch.equal(ab, again)                                # run-to-run and batching-invariant bits
    # image permutation inside a batch only reorders a fixed-order fp32 sum
    perm = torch.randperm(128)
    ap = torch.stack(api._compute_ffn_activation_importance(model, [{"pixel_values": px[:128][perm]}], device="cuda"))
    assert torch.allclose(ap, a, rtol=1e-5)
    # planner + select + gather at 37.5 %: t = 1120, keep = 1952, masks have exactly t ones
    plan = api.plan_2ssp_allocation(model, 0.375, min_remaining=512)
    assert (plan.blocks_to_prune, plan.per_block_neurons_to_prune) == (5, 1120)
    res = api.prune_vit_mlp_width(model, n_to_prune_per_block=[1120] * 12, strategy="act_l2", precomputed_importance=list(ab),
                                  collect_masks=True, min_remaining=512)
    assert all(sum(mk) == 1120 for mk in res["ffn_prune_masks"])
    for mk, imp in zip(res["ffn_prune_masks"], ab):
        mk = torch.tensor(mk, dtype=torch.bool)
        assert imp[mk].max() <= imp[~mk].min()                   # everything pruned scores no higher than anything kept
    logits = api.engine_for(model, "cuda", batch_hint=128).logits(px[:128])
    assert torch.isfinite(logits).all() and logits.shape == (128, 1000)


# ----------------------------------------------------------------------------------------------- other model sizes
@pytest.mark.parametrize("name,n_img", [("small", 6), ("large", 8)])
def test_small_and_large_shapes_against_oracle(api, name, n_img):
    """BASELINE configs[1] (ViT-S/16: D=384 -> N is 1.5 GEMM tiles, LayerNorm slab path off) and configs[3]
    (ViT-L/16: D=1024, 16 heads, 24 blocks) against the fp32 functional oracle on a few images."""
    model = synth.make_vit(name, seed=0)
    px = synth.make_pixels(n_img, 224, seed=21)
    ref = O.vit_forward(O.extract_weights(model), px)
    gm = copy.deepcopy(model).cuda()
    got = api._compute_ffn_activation_importance(gm, [{"pixel_values": px}], device="cuda")
    want = [nm.sum(0) / n_img for nm in ref["norms"]]
    assert len(got) == len(want)
    rel = torch.cat([((a - b).abs() / b.abs()) for a, b in zip(got, want)])
    # A handful of images does not average the bf16 rounding noise the way a calibration set does, and a 24-block model
    # compounds it: the bulk must be inside the 1e-2 contract, the worst of ~10^5 neurons gets 1.5x.
    assert float(rel.mean()) <= 2e-3 and float(torch.quantile(rel, 0.999)) <= SCORE_RTOL and float(rel.max()) <= 1.5 * SCORE_RTOL, \
        (float(rel.mean()), float(rel.max()))
    logits = api.engine_for(gm, "cuda", batch_hint=n_img).logits(px).cpu()
    err = (logits - ref["logits"]).abs()
    depth_scale = 2.0 if name == "large" else 1.0   # tolerances were calibrated on 12 blocks (SURVEY 8c); 24 blocks compound twice the rounding
    assert err.max().item() <= depth_scale * LOGIT_MAX_ABS and err.mean().item() <= depth_scale * LOGIT_MEAN_ABS
    # Stage 2 on this shape: suffix recompute equals the full forward with the block skipped, and matches the oracle's
    # skipped forward within the logit tolerance
    labels = ref["logits"].argmax(-1)
    base, cand, total = api.attention_removal_counts(gm, [{"pixel_values": px, "labels": labels}], "cuda", None)
    nb = len(cand)
    assert total == n_img and abs(base - n_img) <= 1
    for i in (0, nb // 2, nb - 1):
        skipped = O.vit_forward(O.extract_weights(model), px, skip_attention=(i,))["logits"]
        ours = api.engine_for(gm, "cuda", batch_hint=n_img).logits(px, skip_attn=[i]).cpu()
        assert (ours - skipped).abs().max().item() <= depth_scale * LOGIT_MAX_ABS
        assert int((ours.argmax(-1) == labels).sum()) == cand[i]
    api.release_engine(gm)


def test_pruned_model_with_odd_widths_runs_in_the_engine(api):
    """Widths that are not multiples of 8 (2411, 1195, ...) are zero-padded inside the engine (TMA needs 16-byte rows);
    the logical nn.Linear shapes stay odd. Checked against the torch forward of the same mutated module."""
    model = synth.make_vit("tiny", seed=0).cuda()
    g_ = torch.Generator().manual_seed(3)
    imps = [torch.rand(256, generator=g_) for _ in range(3)]
    api.prune_vit_mlp_width(model, n_to_prune_per_block=[5, 61, 123], precomputed_importance=imps, min_remaining=8)
    assert [fc1.out_features for fc1, _ in api._gather_mlp_pairs(model)] == [251, 195, 133]
    api.prune_vit_attention_blocks(model, 0.0, selected_indices=[1], num_to_prune=1)
    px = synth.make_pixels(5, 48, seed=2)
    with torch.no_grad():
        ref = model(pixel_values=px.cuda()).logits.float().cpu()
    got = api.engine_for(model, "cuda", batch_hint=5).logits(px).cpu()
    assert (got - ref).abs().max().item() <= LOGIT_MAX_ABS
    scores = api._compute_ffn_activation_importance(model, [{"pixel_values": px}], device="cuda")
    assert [s.numel() for s in scores] == [251, 195, 133]
    ref_scores = O.s1_scores(copy.deepcopy(model).cpu(), [{"pixel_values": px}], "cpu", None, autocast=False)
    assert max(float(((a - b).abs() / b.abs()).max()) for a, b in zip(scores, ref_scores)) <= SCORE_RTOL
