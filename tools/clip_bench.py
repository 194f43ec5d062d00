"""CLIP image tower measurement: ViT-B/32 (T = 50), ViT-B/16 (T = 197), ViT-L/14 (T = 257) at 224^2 and ViT-L/14 at 336^2
(T = 577) with pre-norm and QuickGELU, on one B200.

Per model, on synthetic images in batches of 256 (timm-shaped stand-ins of tests/clip_synth.py):
  * Stage-1 sweep images/s on resident device pixels and through the API with pinned host pixels, and the same images
    through the torch CUDA baseline (`O.s1_scores(..., autocast=True)` on the module with its fc1 hooks);
  * the per-kernel-class split of a resident sweep (tssp_profile_begin / end);
  * ViT-B/16 only: prune end to end (tools/deit_bench.py's flow) and batch-256 inference of the dense and the pruned model;
and on their own, alternating the two forms in one loop:
  * fc1 with QuickGELU (modes 7 / 8) against the erf GELU instances (modes 1 / 3) at the fc1 shapes of B/16 and L/14,
    256 images, as microseconds per launch;
  * the pre-norm pass (the fp32 LayerNorm in place on the residual stream) at the B/16 and L/14 shapes, and its share of
    the resident sweep;
and the card's name, power limit and maximum SM clock, read in the same run (read-only nvidia-smi query).

Writes one JSON document (default profiles/clip_r1.json). Needs a GPU; there is no CPU fallback.

    python tools/clip_bench.py [--images 1024] [--batch 256] [--steps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from deit_bench import prune_end_to_end  # noqa: E402
from layerscale_bench import kernel_split  # noqa: E402
from long_seq_bench import gpu_info, timed  # noqa: E402

# key: (clip_synth shape, prune + inference measured)
MODELS = {
    "clip_vit_b32_224": ("b32", False),
    "clip_vit_b16_224": ("b16", True),
    "clip_vit_l14_224": ("l14", False),
    "clip_vit_l14_336": ("l14_336", False),
}


def alternating(fns: dict, rounds: int, per_round: int) -> dict:
    """us per launch of each function, the forms timed in turn `rounds` times (CUDA events around `per_round` launches);
    the median round of each is reported with all rounds listed."""
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, per_round, 2) * 1e3)
    return {k: {"us_per_launch": sorted(v)[len(v) // 2], "rounds_us": v} for k, v in out.items()}


def fc1_comparison(L, ops, dev) -> dict:
    res = {}
    for name, (T, D, F) in {"b16": (197, 768, 3072), "l14": (257, 1024, 4096)}.items():
        M = 256 * T
        g = torch.Generator(device=dev).manual_seed(T)
        a = (torch.randn(M, D, device=dev, generator=g) * 0.5).bfloat16()
        w = (torch.randn(F, D, device=dev, generator=g) * 0.05).bfloat16()
        bias = torch.randn(F, device=dev, generator=g) - 1.0
        out = torch.empty(M, F, device=dev, dtype=torch.bfloat16)
        partials = torch.empty(2 * ((M + 31) // 32), F, device=dev)

        def run(mode, score):
            if score:
                return lambda: ops.gemm(mode, a, w, out, bias, partials=partials, tokens_per_image=T)
            return lambda: ops.gemm(mode, a, w, out, bias)
        t = alternating({"erf_gelu_score_pre": run(L.EPI_BF16_GELU_SCORE_PRE, True),
                         "quick_gelu_score_pre": run(L.EPI_BF16_QGELU_SCORE_PRE, True),
                         "erf_gelu": run(L.EPI_BF16_GELU, False), "quick_gelu": run(L.EPI_BF16_QGELU, False)}, 5, 20)
        flop = 2.0 * M * F * D
        for v in t.values():
            v["TFLOP_per_s"] = flop / (v["us_per_launch"] * 1e-6) / 1e12
        res[name] = {"M": M, "N": F, "K": D, "launches": t,
                     "quick_over_erf_score_pre": t["quick_gelu_score_pre"]["us_per_launch"] / t["erf_gelu_score_pre"]["us_per_launch"],
                     "quick_over_erf_plain": t["quick_gelu"]["us_per_launch"] / t["erf_gelu"]["us_per_launch"]}
    return res


def pre_norm_cost(ops, dev) -> dict:
    res = {}
    for name, (T, D) in {"b16": (197, 768), "l14": (257, 1024), "l14_336": (577, 1024)}.items():
        M = 256 * T
        x = torch.randn(M, D, device=dev)
        gamma, beta = torch.ones(D, device=dev), torch.zeros(D, device=dev)
        ms = timed(lambda: ops.layernorm_f32(x, gamma, beta, 1e-5, out=x), 20, 3)
        n_bytes = 2 * M * D * 4
        res[name] = {"rows": M, "D": D, "us_per_launch": ms * 1e3, "GB_per_s": n_bytes / (ms * 1e-3) / 1e9,
                     "what": "fp32 rows read and written back in place, over CUDA-event time per launch"}
    return res


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sparsity", type=float, default=0.375)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "clip_r1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("clip_bench: no CUDA device", file=sys.stderr)
        return 2

    import __graft_entry__ as g
    g.build()
    import clip_synth as CS
    from oracle import twossp_oracle as O
    from twossp_b200 import _lib as L
    from twossp_b200 import api, ops

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.load()
    res = {"what": "timm-shaped CLIP image towers (pre-norm, QuickGELU, bias-free patch embedding), seeded weights "
                   "(tests/clip_synth.py), synthetic N(0,1) images", "gpu": gpu_info(dev.index),
           "sm_count": torch.cuda.get_device_properties(dev).multi_processor_count, "images": args.images, "batch": args.batch,
           "steps": args.steps, "warmup": args.warmup, "timing": "CUDA events around whole sweeps; wall clock around the prune flow",
           "models": {}}
    bs = args.batch
    for key, (shape, full) in MODELS.items():
        image, patch = CS.CLIP_SHAPES[shape][:2]
        gen = torch.Generator(device=dev).manual_seed(1234)
        px_dev = torch.randn(args.images, 3, image, image, device=dev, generator=gen)
        px_host = px_dev.cpu().pin_memory()
        dev_batches = [px_dev[s:s + bs] for s in range(0, args.images, bs)]
        host_batches = [{"pixel_values": px_host[s:s + bs]} for s in range(0, args.images, bs)]
        model = CS.make_clip(shape).to(dev)
        r = {"shape": dict(zip(("image", "patch", "hidden", "layers", "heads", "ffn", "labels"), CS.CLIP_SHAPES[shape])),
             "T": (image // patch) ** 2 + 1}
        eng = api.engine_for(model, dev, batch_hint=bs)

        def sweep_resident():
            eng.s1_reset()
            for b in dev_batches:
                eng.s1_batch(b)
            return eng.s1_score_sums(on_device=True)

        ms_res = timed(sweep_resident, args.steps, args.warmup)
        r["s1_resident"] = {"ms_per_sweep": ms_res, "images_per_s": args.images / (ms_res * 1e-3)}
        r["kernel_split_eager"] = kernel_split(lib, L, sweep_resident)
        ms_host = timed(lambda: api._compute_ffn_activation_importance(model, host_batches, device=dev), args.steps, max(args.warmup, 2))
        r["s1_host_pixels"] = {"ms_per_sweep": ms_host, "images_per_s": args.images / (ms_host * 1e-3),
                               "api": "api._compute_ffn_activation_importance(model, pinned host batches, device='cuda')"}
        tb = [{"pixel_values": b} for b in dev_batches]
        ms_torch = timed(lambda: O.s1_scores(model, tb, str(dev), None, autocast=True), max(1, args.steps - 1), 1)
        r["torch_cuda_baseline"] = {"ms_per_sweep": ms_torch, "images_per_s": args.images / (ms_torch * 1e-3),
                                    "what": "O.s1_scores(model.cuda(), batches, 'cuda', autocast=True): module + hooks under CUDA autocast",
                                    "speedup_resident": ms_torch / ms_res, "speedup_host_pixels": ms_torch / ms_host}
        if full:
            with torch.no_grad():
                labels = torch.cat([eng.logits(b).argmax(-1) for b in dev_batches]).cpu()   # self-labels
            api.release_engine(model)
            batches = [{"pixel_values": px_host[s:s + bs], "labels": labels[s:s + bs]} for s in range(0, args.images, bs)]
            r["prune_end_to_end"], work = prune_end_to_end(api, model, batches, dev, args.sparsity, 256)
            infer = {}
            for name, m in (("dense", model), ("pruned", work)):
                e_ = api.engine_for(m, dev, batch_hint=256)
                ms = timed(lambda: e_.logits(px_dev[:256]), 5, 2)
                infer[f"{name}_images_per_s_batch256"] = 256 / (ms * 1e-3)
                api.release_engine(m)
            r["inference"] = infer
            del work
        else:
            api.release_engine(model)
        res["models"][key] = r
        del model, eng, px_dev, px_host, dev_batches, host_batches
        api.trim_pool()
        torch.cuda.empty_cache()

    res["fc1_quick_gelu_vs_erf"] = fc1_comparison(L, ops, dev)
    res["pre_norm"] = pre_norm_cost(ops, dev)
    for key, (shape, _) in MODELS.items():
        if shape in res["pre_norm"]:
            m = res["models"][key]
            per_sweep_ms = res["pre_norm"][shape]["us_per_launch"] * 1e-3 * args.images / 256
            res["pre_norm"][shape]["share_of_resident_sweep"] = per_sweep_ms / m["s1_resident"]["ms_per_sweep"]

    res["torch"] = torch.__version__
    res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
