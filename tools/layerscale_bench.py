"""LayerScale measurement: DeiT-III-B/16 (T = 197), DINOv2-B/14 (T = 257) and DINOv2-B/14-reg4 (T = 261) at 224^2 on
one B200, next to a ViT-B/16 of the same shapes without LayerScale.

Per model, on 1024 synthetic images in batches of 256 (timm-shaped stand-ins of tests/layerscale_synth.py):
  * Stage-1 sweep images/s on resident device pixels and through the API with pinned host pixels, and the same images
    through the torch CUDA baseline (`O.s1_scores(..., autocast=True)` on the module with its fc1 hooks);
  * the per-kernel-class split of a resident sweep (tssp_profile_begin / end): proj and fc2 of DeiT-III-B/16 against
    those of the ViT-B/16 measure the gamma multiply of the scaled epilogue; attention's share at T = 261;
  * prune end to end (tools/deit_bench.py's flow) and batch-256 inference of the dense and the pruned model;
  * patch extraction at P = 14 on its own: bytes moved (fp32 pixels read, bf16 patch rows written) over kernel time;
and the card's name, power limit and maximum SM clock, read in the same run (read-only nvidia-smi query).

Writes one JSON document (default profiles/layerscale_r1.json). Needs a GPU; there is no CPU fallback.

    python tools/layerscale_bench.py [--images 1024] [--batch 256] [--steps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
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
from long_seq_bench import gpu_info, timed  # noqa: E402

# key: (layerscale_synth shape, LayerScale init or None, full measurement)
MODELS = {
    "vit_base_16_224_no_layerscale": ("deit3_base", None, False),
    "deit3_base_16_224": ("deit3_base", 0.5, True),
    "dinov2_base_14_224": ("dinov2_base", 0.5, True),
    "dinov2_base_14_reg4_224": ("dinov2_base_reg4", 0.5, True),
}


def kernel_split(lib, L, sweep) -> dict:
    torch.cuda.synchronize()
    lib.tssp_profile_begin()
    for _ in range(2):
        sweep()
    ms_arr = (C.c_double * len(L.PROFILE_CLASSES))()
    n_arr = (C.c_uint64 * len(L.PROFILE_CLASSES))()
    L.check(lib.tssp_profile_end(ms_arr, n_arr, len(L.PROFILE_CLASSES)))
    kernels = {name: {"ms_per_sweep": ms_arr[i] / 2, "launches_per_sweep": int(n_arr[i]) // 2}
               for i, name in enumerate(L.PROFILE_CLASSES) if n_arr[i] > 0}
    total = sum(k["ms_per_sweep"] for k in kernels.values())
    for k in kernels.values():
        k["share"] = k["ms_per_sweep"] / total
    return {"classes": kernels, "sum_ms_per_sweep": total}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sparsity", type=float, default=0.375)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "layerscale_r1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("layerscale_bench: no CUDA device", file=sys.stderr)
        return 2

    import __graft_entry__ as g
    g.build()
    import layerscale_synth as LS
    from oracle import twossp_oracle as O
    from twossp_b200 import _lib as L
    from twossp_b200 import api, ops

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.load()
    res = {"what": "timm-shaped LayerScale ViTs, seeded weights with gammas around 0.5 (tests/layerscale_synth.py), synthetic "
                   "N(0,1) 224x224 images", "gpu": gpu_info(dev.index),
           "sm_count": torch.cuda.get_device_properties(dev).multi_processor_count, "images": args.images, "batch": args.batch,
           "steps": args.steps, "warmup": args.warmup, "timing": "CUDA events around whole sweeps; wall clock around the prune flow",
           "models": {}}
    gen = torch.Generator(device=dev).manual_seed(1234)
    px_dev = torch.randn(args.images, 3, 224, 224, device=dev, generator=gen)
    px_host = px_dev.cpu().pin_memory()
    bs = args.batch
    dev_batches = [px_dev[s:s + bs] for s in range(0, args.images, bs)]
    host_batches = [{"pixel_values": px_host[s:s + bs]} for s in range(0, args.images, bs)]

    for key, (shape, init, full) in MODELS.items():
        model = LS.make_ls(shape, init_values=init).to(dev)
        image, patch = LS.LS_SHAPES[shape][:2]
        T = (image // patch) ** 2 + 1 + LS.LS_SHAPES[shape][7]
        r = {"shape": dict(zip(("image", "patch", "hidden", "layers", "heads", "ffn", "labels", "register_tokens", "no_embed_class"),
                               LS.LS_SHAPES[shape])), "layer_scale": init is not None, "T": T}
        eng = api.engine_for(model, dev, batch_hint=bs)

        def sweep_resident():
            eng.s1_reset()
            for b in dev_batches:
                eng.s1_batch(b)
            return eng.s1_score_sums(on_device=True)

        ms_res = timed(sweep_resident, args.steps, args.warmup)
        r["s1_resident"] = {"ms_per_sweep": ms_res, "images_per_s": args.images / (ms_res * 1e-3)}
        r["kernel_split_eager"] = kernel_split(lib, L, sweep_resident)
        if full:
            ms_host = timed(lambda: api._compute_ffn_activation_importance(model, host_batches, device=dev), args.steps, max(args.warmup, 2))
            r["s1_host_pixels"] = {"ms_per_sweep": ms_host, "images_per_s": args.images / (ms_host * 1e-3),
                                   "api": "api._compute_ffn_activation_importance(model, pinned host batches, device='cuda')"}
            tb = [{"pixel_values": b} for b in dev_batches]
            ms_torch = timed(lambda: O.s1_scores(model, tb, str(dev), None, autocast=True), max(1, args.steps - 1), 1)
            r["torch_cuda_baseline"] = {"ms_per_sweep": ms_torch, "images_per_s": args.images / (ms_torch * 1e-3),
                                        "what": "O.s1_scores(model.cuda(), batches, 'cuda', autocast=True): module + hooks under CUDA autocast",
                                        "speedup_resident": ms_torch / ms_res, "speedup_host_pixels": ms_torch / ms_host}
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
        del model, eng
        api.trim_pool()
        torch.cuda.empty_cache()

    base = res["models"]["vit_base_16_224_no_layerscale"]["kernel_split_eager"]["classes"]
    d3 = res["models"]["deit3_base_16_224"]["kernel_split_eager"]["classes"]
    res["gamma_multiply_cost"] = {c: {"vit_b16_ms": base[c]["ms_per_sweep"], "deit3_b16_ms": d3[c]["ms_per_sweep"],
                                      "ratio": d3[c]["ms_per_sweep"] / base[c]["ms_per_sweep"]} for c in ("proj", "fc2")}
    res["attention_share_T261"] = res["models"]["dinov2_base_14_reg4_224"]["kernel_split_eager"]["classes"]["attention"]["share"]

    # patch extraction at P = 14 alone (the padded path): 256 images, prefix 5
    px = px_dev[:256].contiguous()
    ms = timed(lambda: ops.im2col(px, 14, prefix=5), 20, 3)
    n_bytes = px.numel() * 4 + 256 * (16 * 16 + 5) * 592 * 2
    res["im2col_p14"] = {"images": 256, "ms": ms, "bytes": n_bytes, "GB_per_s": n_bytes / (ms * 1e-3) / 1e9,
                         "what": "fp32 pixels read once + bf16 rows [n*261, 592] written, over CUDA-event time per launch"}

    res["torch"] = torch.__version__
    res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
