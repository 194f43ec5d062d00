"""uint8 pixel batches normalised on the device (`api.set_pixel_normalization`). The checks without a GPU come first:
`normalize_pixels` is the written formula, and bad registrations are refused before any device work. The GPU checks
require bit equality, not a tolerance. Through `ops.im2col` and through every API path, a uint8 batch gives the bits
of its fp32 image `normalize_pixels(u, mean, std, rescale)`. That holds for pinned host, pageable host and
device-resident batches.
"""
import copy
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import clip_synth as CS  # noqa: E402
import deit_synth as DS  # noqa: E402
import layerscale_synth as LS  # noqa: E402

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
CLIP = ((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711))


def _bytes(n, image, seed, channels=3):
    """Random pixels with both ends of the range present in every channel."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randint(0, 256, (n, channels, image, image), generator=g, dtype=torch.uint8)
    u[:, :, 0, 0] = 0
    u[:, :, 0, 1] = 255
    return u


# ----------------------------------------------------------------------------------------------- no GPU needed
def test_normalize_pixels_is_the_written_formula():
    from twossp_b200 import api
    u = _bytes(3, 16, seed=1)
    mean, std = IMAGENET
    got = api.normalize_pixels(u, mean, std)
    assert got.dtype == torch.float32
    want = (u.float() * (1 / 255) - torch.tensor(mean).view(1, 3, 1, 1)) / torch.tensor(std).view(1, 3, 1, 1)
    assert torch.equal(got, want)
    # the same three roundings, one fp32 operation at a time, in numpy
    a = u.numpy().astype(np.float32) * np.float32(1 / 255)
    a = (a - np.asarray(mean, np.float32).reshape(1, 3, 1, 1)) / np.asarray(std, np.float32).reshape(1, 3, 1, 1)
    assert np.array_equal(got.numpy(), a.astype(np.float32))
    assert torch.equal(api.normalize_pixels(u, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), rescale=1.0), u.float())


@pytest.mark.parametrize("mean,std,rescale,match", [
    ((0.5, 0.5), (0.2, 0.2, 0.2), 1 / 255, "one value per channel"),
    ((0.5, 0.5, 0.5), (0.2, 0.2, 0.2, 0.2), 1 / 255, "one value per channel"),
    ((0.5, 0.5, 0.5), (0.2, 0.0, 0.2), 1 / 255, "std must be > 0"),
    ((0.5, 0.5, 0.5), (0.2, -1.0, 0.2), 1 / 255, "std must be > 0"),
    ((0.5, 0.5, 0.5), (0.2, 1e-50, 0.2), 1 / 255, "std must be > 0"),          # 0 in fp32
    ((0.5, float("nan"), 0.5), (0.2, 0.2, 0.2), 1 / 255, "finite"),
    ((0.5, 0.5, 0.5), (0.2, float("inf"), 0.2), 1 / 255, "finite"),
    ((0.5, 0.5, 1e300), (0.2, 0.2, 0.2), 1 / 255, "finite"),                   # inf in fp32
    ((0.5, 0.5, 0.5), (0.2, 0.2, 0.2), float("nan"), "finite"),
])
def test_set_pixel_normalization_refuses_bad_values_before_device_work(monkeypatch, mean, std, rescale, match):
    from twossp_b200 import api

    def no_device(*a, **k):
        raise AssertionError("device work before validation")
    monkeypatch.setattr(api, "Engine", no_device)
    monkeypatch.setattr(api, "_cuda_device", no_device)
    model = synth.TimmLikeViT()
    with pytest.raises(ValueError, match=match):
        api.set_pixel_normalization(model, mean, std, rescale)
    assert model not in api._PIXEL_NORMS
    api.set_pixel_normalization(model, *IMAGENET)          # a valid one is stored, and cleared again
    assert api._PIXEL_NORMS[model][2] == C.c_float(1 / 255).value
    api.clear_pixel_normalization(model)
    assert model not in api._PIXEL_NORMS


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


# name -> (model factory, image size, mean / std)
MODELS = {
    "hf_vit": (lambda: synth.make_vit("tiny"), 48, IMAGENET),
    "timm": (lambda: synth.TimmLikeViT(), 48, IMAGENET),
    "deit_teacher": (lambda: DS.make_deit("tiny", head="teacher"), 48, IMAGENET),
    "tiny_reg4": (lambda: LS.make_ls("tiny_reg4"), 84, IMAGENET),
    "clip": (lambda: CS.make_clip("tiny"), 48, CLIP),
}


def _where(u, where):
    return {"pinned": lambda: u.pin_memory(), "pageable": lambda: u.clone(), "device": lambda: u.cuda()}[where]()


def _batches(px, labels, size):
    return [{"pixel_values": px[s:s + size], "labels": labels[s:s + size], "index": torch.arange(s, min(s + size, px.shape[0]))}
            for s in range(0, px.shape[0], size)]


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.gpu
@pytest.mark.parametrize("prefix", [1, 2, 5])
@pytest.mark.parametrize("P,H", [(16, 64), (14, 84), (8, 48), (32, 96), (5, 45)])
def test_im2col_u8_equals_fp32_on_the_normalised_image(api, ops, P, H, prefix):
    u = _bytes(3, H, seed=P * 10 + prefix).cuda()
    mean, std = IMAGENET
    got = ops.im2col(u, P, prefix=prefix, mean=mean, std=std)
    want = ops.im2col(api.normalize_pixels(u, mean, std), P, prefix=prefix)
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    K = 3 * P * P
    assert not got[:, K:].view(torch.int16).any()                          # zero padding columns
    T = (H // P) ** 2 + prefix
    assert not got.view(3, T, -1)[:, :prefix].view(torch.int16).any()     # zero prefix rows


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [1, 2, 4])
def test_im2col_u8_other_channel_counts(api, ops, channels):
    u = _bytes(2, 32, seed=channels, channels=channels).cuda()
    mean, std = [0.1 * (c + 1) for c in range(channels)], [0.2 + 0.05 * c for c in range(channels)]
    got = ops.im2col(u, 16, mean=mean, std=std, rescale=1 / 127.5)
    want = ops.im2col(api.normalize_pixels(u, mean, std, 1 / 127.5), 16)
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


# ----------------------------------------------------------------------------------------------- the whole path
def _results(api, model, batches, norm, batch_hint):
    """Everything the API computes from pixels, for one copy of `model` (on the GPU)."""
    gm = copy.deepcopy(model).cuda()
    if norm is not None:
        api.set_pixel_normalization(gm, *norm)
    out = {}
    out["scores"] = api._compute_ffn_activation_importance(gm, batches, device="cuda")
    out["exact"] = api._compute_ffn_activation_importance(gm, batches, device="cuda", exact=True)
    eng = api.engine_for(gm, "cuda", batch_hint=batch_hint)
    norms = []
    for b in batches:
        eng.s1_reset()
        buf = torch.zeros(b["pixel_values"].shape[0], sum(eng.ffn_dims), device="cuda")
        eng.s1_batch(b["pixel_values"], img_norms=buf)
        norms.append(buf.cpu())
    out["img_norms"] = torch.cat(norms)
    out["logits"] = torch.cat([eng.logits(b["pixel_values"]).cpu() for b in batches])
    out["top1"] = api.evaluate_top1(gm, batches, "cuda")
    out["s2"] = api.attention_removal_counts(gm, batches, "cuda", None)
    out["s2_scored"] = api.attention_removal_counts(gm, batches, "cuda", None, with_scores=True)
    att, mlp = api.B200Auto2SSPInterface(gm, batches, device="cuda", batch_limit=None).fit()
    out["fit"] = (att, mlp)
    width = api._gather_mlp_pairs(gm)[0][0].out_features
    res = api.prune_vit_mlp_width(gm, strategy="act_l2", dataloader=batches, device="cuda", batch_limit=None,
                                  n_to_prune_per_block=[width // 2 - 3] * len(mlp), collect_masks=True, min_remaining=8)
    out["masks"], out["indices"] = res["ffn_prune_masks"], res["ffn_pruned_indices"]
    api.release_engine(gm)   # the rebuilt engine must keep the registration
    out["pruned_logits"] = torch.cat([api.engine_for(gm, "cuda", batch_hint=batch_hint).logits(b["pixel_values"]).cpu()
                                      for b in batches])
    api.release_engine(gm)
    return out


def _assert_same(x, y):
    def same(a, b):
        if isinstance(a, torch.Tensor):
            return torch.equal(a, b)
        if isinstance(a, (list, tuple)):
            return len(a) == len(b) and all(same(p, q) for p, q in zip(a, b))
        return a == b
    for k in x:
        assert same(x[k], y[k]), k


@pytest.fixture(scope="module", params=sorted(MODELS))
def case(request, cuda_ready):
    """(name, model, uint8 pixels, fp32 reference results through normalize_pixels, norm, labels)"""
    from twossp_b200 import api
    make, image, norm = MODELS[request.param]
    model = make()
    u = _bytes(24, image, seed=77)
    f = api.normalize_pixels(u, *norm)
    gm = copy.deepcopy(model).cuda()
    labels = api.engine_for(gm, "cuda", batch_hint=24).logits(f).argmax(-1).cpu()
    labels[::5] = (labels[::5] + 1) % 10   # some wrong predictions
    api.release_engine(gm)
    ref = _results(api, model, _batches(f, labels, 8), None, 8)
    assert 0 < ref["top1"] < 1
    return request.param, model, u, ref, norm, labels


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["pinned", "pageable", "device"])
def test_uint8_batches_give_the_bits_of_their_normalised_images(api, case, where):
    name, model, u, ref, norm, labels = case
    got = _results(api, model, _batches(_where(u, where), labels, 8), norm, 8)
    _assert_same(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hf_vit", "tiny_reg4"])
def test_split_first_host_batch_gives_the_device_bits(api, name):
    # 160 images: the first host batch after s1_reset is copied and swept in two parts
    make, image, norm = MODELS[name]
    model = make().cuda()
    n = 160
    u = _bytes(n, image, seed=5)
    api.set_pixel_normalization(model, *norm)
    eng = api.engine_for(model, "cuda", batch_hint=n)
    out = {}
    for where, px in (("device_u8", u.cuda()), ("host_u8", u.pin_memory()), ("device_f32", api.normalize_pixels(u, *norm).cuda())):
        eng.s1_reset()
        norms = torch.zeros(n, sum(eng.ffn_dims), device="cuda")
        eng.s1_batch(px, img_norms=norms)
        eng.s1_batch(px[: n // 2])
        out[where] = (norms.cpu(), eng.s1_score_sums().clone())
    assert float(out["device_u8"][0].abs().min()) > 0
    for k in ("host_u8", "device_f32"):
        assert torch.equal(out["device_u8"][0], out[k][0]) and torch.equal(out["device_u8"][1], out[k][1]), k
    api.release_engine(model)
    api.clear_pixel_normalization(model)


@pytest.mark.gpu
def test_pinned_buffer_overwritten_after_every_call(api):
    make, image, norm = MODELS["timm"]
    model = make().cuda()
    u = _bytes(32, image, seed=9)
    labels = torch.arange(32) % 10
    api.set_pixel_normalization(model, *norm)
    eng = api.engine_for(model, "cuda", batch_hint=8, need_cache=True)

    def sweep(feed):
        eng.s1_reset()
        eng.s2_reset()
        for s in range(0, 32, 8):
            eng.s1_batch(feed(u[s:s + 8]))
            eng.s2_batch(feed(u[s:s + 8]), labels[s:s + 8])
        return eng.s1_score_sums().clone(), eng.s2_counts()

    want = sweep(lambda b: b.clone().pin_memory())
    buf = torch.empty(8, 3, image, image, dtype=torch.uint8).pin_memory()
    junk = _bytes(8, image, seed=10)

    def reused(b):
        buf.copy_(b)
        return buf
    got_s, got_c = [], []
    eng.s1_reset()
    eng.s2_reset()
    for s in range(0, 32, 8):
        eng.s1_batch(reused(u[s:s + 8]))
        buf.copy_(junk)                     # the caller's buffer is overwritten as soon as the call returns
        eng.s2_batch(reused(u[s:s + 8]), labels[s:s + 8])
        buf.copy_(junk)
    got = eng.s1_score_sums().clone(), eng.s2_counts()
    assert torch.equal(got[0], want[0]) and got[1] == want[1]
    api.release_engine(model)


@pytest.mark.gpu
def test_alternating_formats_in_one_sweep(api, lib):
    make, image, norm = MODELS["hf_vit"]
    model = make().cuda()
    u = _bytes(32, image, seed=12)
    f = api.normalize_pixels(u, *norm)
    api.set_pixel_normalization(model, *norm)
    eng = api.engine_for(model, "cuda", batch_hint=8)
    captures = lib.load().tssp_graph_capture_count

    def sweep(pick):
        eng.s1_reset()
        for i, s in enumerate(range(0, 32, 8)):
            eng.s1_batch(pick(i)[s:s + 8].pin_memory())
        logits = torch.cat([eng.logits(pick(i)[s:s + 8].cuda()).cpu() for i, s in enumerate(range(0, 32, 8))])
        return eng.s1_score_sums().clone(), logits

    f32 = sweep(lambda i: f)
    before = captures()
    u8 = sweep(lambda i: u)
    mixed = sweep(lambda i: u if i % 2 else f)
    mixed2 = sweep(lambda i: f if i % 2 else u)
    assert captures() == before           # the format is not part of any captured chain
    for r in (u8, mixed, mixed2):
        assert torch.equal(r[0], f32[0]) and torch.equal(r[1], f32[1])
    api.release_engine(model)
    api.clear_pixel_normalization(model)


@pytest.mark.gpu
def test_uint8_without_registration_keeps_the_float_conversion(api):
    make, image, norm = MODELS["timm"]
    model = make().cuda()
    u = _bytes(16, image, seed=13)

    def run(px):
        api._compute_ffn_activation_importance(model, [{"pixel_values": px}], device="cuda")
        return api.engine_for(model, "cuda", batch_hint=16).s1_score_sums().clone(), api.engine_for(model, "cuda").logits(px).cpu()

    want = run(u.float())                 # what a uint8 batch has always meant: raw 0..255 values as fp32
    for px in (u, u.cuda(), u.pin_memory()):
        got = run(px)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    api.set_pixel_normalization(model, *norm)
    normalised = run(u)
    assert not torch.equal(normalised[1], want[1])
    api.clear_pixel_normalization(model)
    got = run(u)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    api.release_engine(model)


# ----------------------------------------------------------------------------------------------- C ABI validation
@pytest.mark.gpu
def test_c_abi_refusals_name_the_fault(api, lib):
    L = lib
    raw = L.load()
    out = torch.empty(4 * 17, 768, device="cuda", dtype=torch.bfloat16)
    u = torch.zeros(4 * 3 * 64 * 64 + 16, device="cuda", dtype=torch.uint8)
    good = L.pixel_input(L.PIXELS_U8, IMAGENET[0], IMAGENET[1], 1 / 255)
    s = L.current_stream()

    def msg():
        return raw.tssp_last_error().decode()
    assert raw.tssp_op_im2col(L.ptr(u), L.ptr(out), 4, 3, 64, 64, 16, 1, good, s) == 0
    five = torch.zeros(5 * 64 * 64, device="cuda", dtype=torch.uint8)
    assert raw.tssp_op_im2col(L.ptr(five), L.ptr(out), 1, 5, 64, 64, 16, 1, L.pixel_input(L.PIXELS_U8, [0.0] * 4, [1.0] * 4), s) != 0
    assert "channels" in msg() and "C=5" in msg()
    bad = L.pixel_input(L.PIXELS_U8, IMAGENET[0], (0.2, 0.0, 0.2), 1 / 255)
    assert raw.tssp_op_im2col(L.ptr(u), L.ptr(out), 4, 3, 64, 64, 16, 1, bad, s) != 0
    assert "std[1]" in msg()
    assert raw.tssp_op_im2col(C.c_void_p(u.data_ptr() + 1), L.ptr(out), 4, 3, 64, 64, 16, 1, good, s) != 0
    assert "aligned" in msg()
    assert raw.tssp_op_im2col(C.c_void_p(u.data_ptr() + 1), L.ptr(out), 1, 3, 28, 28, 14, 1, good, s) != 0
    assert "2-byte aligned" in msg()
    # the engine setter: bad values are refused and the engine keeps its format
    model = synth.TimmLikeViT().cuda()
    eng = api.engine_for(model, "cuda", batch_hint=16)
    assert raw.tssp_set_pixel_input(eng._handle, C.byref(bad)) != 0 and "std[1]" in msg()
    nan = L.pixel_input(L.PIXELS_U8, (0.5, float("nan"), 0.5), IMAGENET[1], 1 / 255)
    assert raw.tssp_set_pixel_input(eng._handle, C.byref(nan)) != 0 and "mean[1]" in msg()
    assert raw.tssp_set_pixel_input(eng._handle, C.byref(L.pixel_input(7))) != 0 and "format=7" in msg()
    # a misaligned device-resident batch through an entry point
    px = _bytes(2, 48, seed=1).cuda().view(-1)
    shifted = torch.empty(px.numel() + 1, device="cuda", dtype=torch.uint8)
    shifted[1:] = px
    assert raw.tssp_set_pixel_input(eng._handle, C.byref(good)) == 0
    assert raw.tssp_s1_batch(eng._handle, C.c_void_p(shifted.data_ptr() + 1), 2, 0, None, s) != 0 and "aligned" in msg()
    torch.cuda.synchronize()
    api.release_engine(model)
