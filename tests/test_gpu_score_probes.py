"""Stage-1 score path on integer-coded inputs whose every expected value is exact (tests/score_ref.py): the fc1 score
epilogue in its three modes and two tile forms, the finisher on its own, the engine's all-blocks finisher after a
width prune, the erf-GELU epilogue on a dense grid, and the plain / fp32 / LayerScale / row-norm epilogues. Norms and
scores are compared bit for bit, so one token counted in the wrong image, a dropped tail row, a wrong block offset or a
missing k-step fails. Every launch runs twice and the two results must carry the same bits: consecutive launches walk
their tiles in opposite directions.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import score_ref as S  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCORE_MODES = ["gelu_score", "gelu_score_pre", "qgelu_score_pre"]


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as g
    g.build()
    torch.cuda.set_device(0)
    from twossp_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ops(lib):
    from twossp_b200 import ops as o
    return o


@pytest.fixture(scope="module")
def api(lib):
    from twossp_b200 import api as a
    return a


@pytest.fixture(params=[1, 2], ids=["cta1", "pair"])
def gemm_form(request, lib):
    """Run a GEMM test in both tile forms (single CTA, CTA pair), then restore the automatic choice."""
    lib.check(lib.load().tssp_set_gemm_form(request.param))
    yield request.param
    lib.check(lib.load().tssp_set_gemm_form(0))


def _bits(t: torch.Tensor) -> torch.Tensor:
    """An integer view of the same bytes: NaNs compare equal to themselves."""
    return t.contiguous().view({4: torch.int32, 2: torch.int16}[t.element_size()])


def _twice(run):
    """run() twice; both results (tuples of tensors) must carry the same bits. Returns the first."""
    first, second = run(), run()
    for x, y in zip(first, second):
        assert torch.equal(_bits(x), _bits(y)), "two launches of the same work gave different bits"
    return first


def _cuda(x, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(x)).to("cuda", dtype)


def _ldp(N: int) -> int:
    return (N + 7) // 8 * 8 + 8  # a multiple of 8, larger than N


def _mode(lib, name):
    return {"gelu_score": lib.EPI_BF16_GELU_SCORE, "gelu_score_pre": lib.EPI_BF16_GELU_SCORE_PRE,
            "qgelu_score_pre": lib.EPI_BF16_QGELU_SCORE_PRE}[name]


def _check_activation(out: np.ndarray, z: np.ndarray, act: str):
    """The stored activation against the fp64 one, with the bounds gemm_tcgen05.cuh states: within 1 bf16 ulp where the
    function is resolved (erf GELU at z >= -5, QuickGELU at |z| <= 50), below that only non-positive and tiny."""
    ref = S.gelu_erf64(z) if act == "gelu" else S.quick_gelu64(z)
    lo, tiny = (-5.0, 1.5e-6) if act == "gelu" else (-50.0, 1e-30)
    near = z >= lo
    assert (np.abs(out - ref)[near] <= S.bf16_ulp(ref[near])).all()
    assert (out[~near] <= 0).all() and (np.abs(out[~near]) <= tiny).all()


# ----------------------------------------------------------------------------------------------- 1. epilogue + finisher
def _score_shapes():
    shapes = [pytest.param(T, n, N, id=f"T{T}-n{n}-N{N}") for T, n, N in S.PROBE_SHAPES]
    return shapes + [pytest.param(None, name, None, id=name) for name in ("sms+1", "2sms-1", "2sms+1")]


@pytest.mark.parametrize("mode", SCORE_MODES)
@pytest.mark.parametrize("T,n_img,N", _score_shapes())
def test_score_epilogue_and_finisher_are_bit_exact(ops, lib, gemm_form, mode, T, n_img, N):
    if T is None:  # single-CTA tile counts around the SM count: the last wave holds one tile, or one short of full
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        _, T, n_img, N = {c[0]: c for c in S.sm_cases(sms)}[n_img]
    M, kind = n_img * T, ("post" if mode == "gelu_score" else "pre")
    K = 64 * (1 + T % 3)  # one to three K blocks (the codes live in k = 0, 1)
    f = S.row_codes(M, T, kind)
    g, h = S.col_codes(N, kind)
    a, w, bias = S.operands(f, g, h, K)
    z = S.z_of(f, g, h)
    want = S.norms_of(S.image_sums(z, T))
    base = np.arange(N, dtype=np.float32) % 7
    a_d, w_d, b_d = _cuda(a, torch.bfloat16), _cuda(w, torch.bfloat16), _cuda(bias)

    def run():
        out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        partials = torch.full((2 * ((M + 31) // 32), _ldp(N)), float("nan"), device="cuda")
        ops.gemm(_mode(lib, mode), a_d, w_d, out, b_d, partials=partials, tokens_per_image=T)
        scores = _cuda(base)
        norms = ops.score_finish(partials, n_img, T, N, scores)
        return out, partials, norms, scores

    out, partials, norms, scores = _twice(run)
    part = partials.cpu().numpy()
    emu_part, _ = S.emulate(z, T)
    assert np.array_equal(part[:, :N].reshape(-1, 2, N), emu_part), "partials differ from the exact per-segment sums"
    assert np.isnan(part[:, N:]).all(), "a partial was written past N"
    got = norms.cpu().numpy()
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} norms differ, first (image, neuron) {bad[:4].tolist()}: {got[tuple(bad[0])]} != {want[tuple(bad[0])]}"
    assert np.array_equal(scores.cpu().numpy(), S.accumulate(want, base))
    stored = out.float().cpu().numpy().astype(np.float64)
    if mode == "gelu_score":
        assert np.array_equal(stored, z.astype(np.float64)), "gelu(z) must be z itself on {0} U [6, 60]"
    else:
        _check_activation(stored, z.astype(np.float64), "gelu" if mode == "gelu_score_pre" else "qgelu")


# ----------------------------------------------------------------------------------------------- 2. finisher alone
@pytest.mark.parametrize("T,n_img,F", [(T, n, N - 3) for T, n, N in S.PROBE_SHAPES])
def test_finisher_reads_exactly_its_slots(ops, T, n_img, F):
    """Partials built on the host: exact integers only in the (sub-tile, slot) pairs the finisher must read, NaN in the
    other slot of every sub-tile and in the padding columns. A finisher that reads a wrong slot, a wrong sub-tile or past
    F turns a norm into NaN or moves it off the exact value."""
    M, ldp = n_img * T, _ldp(F)
    rng = np.random.default_rng(T * 1009 + F)
    part = np.full((2 * ((M + 31) // 32), ldp), np.nan, np.float32)
    sums = np.zeros((n_img, F), np.int64)
    for img, s, seg in S.finisher_slots(n_img, T):
        v = rng.integers(0, 4096, F)
        part[2 * s + seg, :F] = v
        sums[img] += v
    want = S.norms_of(sums)
    base = (np.arange(F) % 5).astype(np.float32)
    part_d = _cuda(part)

    def run():
        scores = _cuda(base)
        return ops.score_finish(part_d, n_img, T, F, scores), scores

    norms, scores = _twice(run)
    got = norms.cpu().numpy()
    assert not np.isnan(got).any()
    assert np.array_equal(got, want)
    assert np.array_equal(scores.cpu().numpy(), S.accumulate(want, base))


# ----------------------------------------------------------------------------------------------- 3. engine finisher
N_IMAGES, CAPACITY = 37, 16  # three engine chunks (16, 16, 5)


def _model(name):
    """(model, image size, T) of the synthetic models the suite already builds."""
    from oracle import synth
    if name == "hf_vit":
        return synth.make_vit("tiny", seed=0), 48, 37
    if name == "timm":
        return synth.TimmLikeViT(), 48, 37
    if name == "tiny_long":
        synth.SHAPES.setdefault("tiny_long", (136, 8, 128, 3, 2, 256, 10))
        return synth.make_vit("tiny_long", seed=0), 136, 290
    if name == "deit_teacher":
        import deit_synth as DS
        return DS.make_deit("ti", seed=0, head="teacher"), 224, 198
    if name == "ls_reg4":
        import layerscale_synth as LS
        return LS.make_ls("tiny_reg4"), 84, 41
    if name == "clip":
        import clip_synth as CS
        return CS.make_clip("tiny"), 48, 37
    raise KeyError(name)


ENGINE_MODELS = ["hf_vit", "timm", "deit_teacher", "ls_reg4", "clip", "tiny_long"]


def _coded_pruned_model(api, name):
    """The model width-pruned to different F per block (some not a multiple of 8), then coded: ln2 outputs exactly e_0
    on every token (weight 0, bias e_0), so fc1 gives z_c = fc1.weight[c, 0] + fc1.bias[c] on every row. Returns the
    model, its image size, T and the per-block z codes."""
    from twossp_b200.anatomy import gather_mlp_pairs, get_blocks
    model, image, T = _model(name)
    model = model.cuda().eval()
    pairs = gather_mlp_pairs(model)
    gen = torch.Generator().manual_seed(5)
    cuts = [[77, 5, 0, 13][b % 4] for b in range(len(pairs))]
    api.prune_vit_mlp_width(model, n_to_prune_per_block=cuts, precomputed_importance=[torch.rand(fc1.out_features, generator=gen)
                                                                                     for fc1, _ in pairs], min_remaining=8)
    kind, blocks = get_blocks(model)
    codes = []
    with torch.no_grad():
        for b, (blk, (fc1, _)) in enumerate(zip(blocks, gather_mlp_pairs(model))):
            ln2 = blk.layernorm_after if kind == "hf" else blk.norm2
            ln2.weight.zero_()
            ln2.bias.zero_()
            ln2.bias[0] = 1.0
            g, h = S.col_codes(fc1.out_features, "post", seed=b + 1)
            fc1.weight[:, 0] = torch.from_numpy(g).float()
            fc1.bias.copy_(torch.from_numpy(h).float())
            codes.append(g + h)
    Fs = [c.size for c in codes]
    assert len(set(Fs)) > 1 and any(F % 8 for F in Fs), Fs
    return model, image, T, codes


def _engine_probe(api, name):
    from oracle import synth
    model, image, T, codes = _coded_pruned_model(api, name)
    row = np.concatenate([np.sqrt((T * c.astype(np.int64) ** 2).astype(np.float32)) for c in codes])
    want_norms = np.tile(row, (N_IMAGES, 1))
    want_sums = S.accumulate(want_norms)
    px = synth.make_pixels(N_IMAGES, image, seed=17)
    eng = api.engine_for(model, "cuda", batch_hint=CAPACITY)
    assert eng.max_images == CAPACITY

    def run():
        eng.s1_reset()
        norms = torch.full((N_IMAGES, sum(eng.ffn_dims)), float("nan"), device="cuda")
        eng.s1_batch(px.cuda(), img_norms=norms)
        return norms, eng.s1_score_sums().clone()

    norms, sums = _twice(run)
    got = norms.cpu().numpy()
    for b, (lo, hi) in enumerate(zip(np.cumsum([0] + [c.size for c in codes])[:-1], np.cumsum([c.size for c in codes]))):
        assert np.array_equal(got[:, lo:hi], want_norms[:, lo:hi]), f"{name}: block {b} per-image norms"
    assert np.array_equal(sums.numpy(), want_sums), f"{name}: s1_score_sums"
    # the API's Stage-1 importance: batches of 16 and 21 images (the second one in two engine chunks), from the host
    batches = [{"pixel_values": px[:CAPACITY], "index": torch.arange(CAPACITY)},
               {"pixel_values": px[CAPACITY:], "index": torch.arange(CAPACITY, N_IMAGES)}]
    want_api = torch.from_numpy(want_sums) / N_IMAGES
    for exact in (False, True):
        got_api = torch.cat(api._compute_ffn_activation_importance(model, batches, device="cuda", exact=exact))
        assert torch.equal(got_api, want_api), f"{name}: importance (exact={exact})"
    api.release_engine(model)


@pytest.mark.parametrize("name", ENGINE_MODELS)
def test_engine_finisher_is_bit_exact_on_pruned_blocks(api, name):
    _engine_probe(api, name)


def test_engine_finisher_without_graphs_on_a_poisoned_pool(lib):
    """The same probes with eager launches (TSSP_GRAPHS=0) and with parked buffers filled with NaN patterns
    (TSSP_POOL_POISON=1), each model twice so that the second engine takes the first one's parked buffers back."""
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_score_probes as t\n"
            "from twossp_b200 import api\n"
            "for name in t.ENGINE_MODELS:\n"
            "    t._engine_probe(api, name)\n"
            "    t._engine_probe(api, name)\n"
            "print('ok')\n") % (ROOT, os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TSSP_GRAPHS="0", TSSP_POOL_POISON="1")
    proc = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert proc.returncode == 0 and proc.stdout.strip().endswith("ok"), proc.stdout[-3000:] + proc.stderr[-3000:]


# ----------------------------------------------------------------------------------------------- 4. erf-GELU grid
@pytest.mark.parametrize("mode", ["gelu", "gelu_score_pre"])
def test_gelu_erf_epilogue_dense_grid(ops, lib, gemm_form, mode, capsys):
    """A = 0, so every row is gelu(bias) on a dense fp32 grid over [-12, 12]: within 1 bf16 ulp of the fp64 erf GELU and
    mostly its exact rounding on [-5, 12]; below -5 non-positive and at most 1.5e-6 in magnitude
    (gemm_tcgen05.cuh: gelu_erf_x2)."""
    M, K, N = 32, 64, 48000
    bias = torch.linspace(-12.0, 12.0, N, device="cuda")
    a = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    w = torch.zeros(N, K, device="cuda", dtype=torch.bfloat16)

    def run():
        out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        partials = torch.full((2, N), float("nan"), device="cuda")
        if mode == "gelu":
            ops.gemm(lib.EPI_BF16_GELU, a, w, out, bias)
        else:
            ops.gemm(lib.EPI_BF16_GELU_SCORE_PRE, a, w, out, bias, partials=partials, tokens_per_image=M)
        return out, partials

    out, partials = _twice(run)
    assert torch.equal(_bits(out), _bits(out[:1].expand(M, N)))
    if mode == "gelu_score_pre":  # one image, one sub-tile: 32 exact squares of bf16(bias) in slot 0, nothing in slot 1
        b16 = bias.bfloat16().float()
        assert torch.equal(partials[0], 32 * b16 * b16) and torch.equal(partials[1], torch.zeros_like(partials[1]))
    x = bias.cpu().numpy().astype(np.float64)
    o = out[0].float().cpu().numpy().astype(np.float64)
    ref = S.gelu_erf64(x)
    hi = x >= -5.0
    ulps = np.abs(o - ref)[hi] / S.bf16_ulp(ref[hi])
    exact = float(np.mean(o[hi] == S.bf16_rne(ref[hi])))
    with capsys.disabled():
        print(f"\n[erf gelu {mode}, form {gemm_form}] on [-5, 12]: max {ulps.max():.3f} bf16 ulp, exact roundings "
              f"{100 * exact:.3f} % of {int(hi.sum())}")
    assert ulps.max() <= 1.0
    assert exact >= 0.99
    assert (o[~hi] <= 0).all() and (np.abs(o[~hi]) <= 1.5e-6).all()


# ----------------------------------------------------------------------------------------------- 5. other epilogues
# (M, N, K): M from the probe shapes; N picks the fp32 tile widths gemm() chooses: 128 (N % 256 <= 128, K <= 512),
# 192 (N a multiple of 192 but not of 256) and 256 (the rest, and every bf16 epilogue)
PLAIN_SHAPES = [(333, 264, 384), (591, 384, 3072), (1005, 576, 768), (771, 1000, 1000), (195, 136, 200), (3075, 3072, 3072)]


def _int_operands(M, N, K, lim, seed):
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(-lim, lim + 1, (M, K), generator=g).float()
    w = torch.randint(-lim, lim + 1, (N, K), generator=g).float()
    bias = torch.randint(-8, 9, (N,), generator=g).float()
    return a.cuda(), w.cuda(), bias.cuda()


@pytest.mark.parametrize("M,N,K", PLAIN_SHAPES)
def test_plain_epilogues_are_bit_exact(ops, lib, gemm_form, M, N, K):
    """Integer a, w in [-4, 4]: |acc| <= 49152, so the fp32 accumulator is the exact product. EPI_F32 (stored and
    reduce-added onto an integer base) and EPI_BF16 (one RNE rounding of the exact value) are bit-exact; EPI_F32_SCALED is
    float32(gamma * float32(acc + bias)) plus the base. A dropped or repeated k-step or a misplaced row or column fails."""
    a, w, bias = _int_operands(M, N, K, 4, M + N + K)
    exact = (a.double() @ w.double().t() + bias.double())  # integers < 2^24: exact in fp64 and in fp32
    base = torch.randint(-64, 65, (M, N), generator=torch.Generator().manual_seed(N)).float().cuda()
    gamma = (torch.rand(N, generator=torch.Generator().manual_seed(K)) * 2 - 1).cuda()
    a16, w16 = a.bfloat16(), w.bfloat16()

    def run():
        f32 = torch.full((M, N), float("nan"), device="cuda")
        ops.gemm(lib.EPI_F32, a16, w16, f32, bias)
        f32_add = base.clone()
        ops.gemm(lib.EPI_F32, a16, w16, f32_add, bias, reduce_add=True)
        b16 = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        ops.gemm(lib.EPI_BF16, a16, w16, b16, bias)
        scaled = base.clone()
        ops.gemm_scaled(a16, w16, scaled, bias, gamma, reduce_add=True)
        return f32, f32_add, b16, scaled

    f32, f32_add, b16, scaled = _twice(run)
    assert torch.equal(f32, exact.float())
    assert torch.equal(f32_add, exact.float() + base)
    assert torch.equal(b16, exact.float().bfloat16())
    assert torch.equal(scaled, gamma * exact.float() + base)


@pytest.mark.parametrize("M,N,K", [(333, 384, 128), (1005, 576, 192), (3075, 2304, 192), (195, 1152, 64)])
def test_rownorm_epilogue_is_bit_exact(ops, gemm_form, M, N, K):
    """The QKV epilogue with entries in {-1, 0, 1} and K <= 192: outputs are integers of at most 200 (exact in bf16) and a
    64-column sum of squares stays below 2^24, so the output and every |q|^2, |k|^2 chunk are exact."""
    a, w, bias = _int_operands(M, N, K, 1, 3 * M + N)
    exact = (a.double() @ w.double().t() + bias.double())
    chunks = 2 * N // 3 // 64  # the q and k heads of a fused qkv
    want_norms = exact.pow(2).reshape(M, N // 64, 64).sum(-1)[:, :chunks].float()
    a16, w16 = a.bfloat16(), w.bfloat16()

    def run():
        out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
        return out, ops.gemm_rownorm(a16, w16, out, bias, chunks)

    out, rownorm = _twice(run)
    assert torch.equal(out, exact.float().bfloat16())
    assert torch.equal(rownorm, want_norms)
