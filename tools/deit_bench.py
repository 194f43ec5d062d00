"""DeiT measurement: DeiT-B-distilled/16 and DeiT-Ti-distilled/16 at 224^2 (T = 198) on one B200.

Per model, on 1024 synthetic images in batches of 256:
  * Stage-1 sweep images/s on resident device pixels and through the API with pinned host pixels, and the same images
    through the torch CUDA baseline (the reference's algorithm, `O.s1_scores(..., autocast=True)` on the HF module, as
    bench.py's torch_cuda_baseline runs it);
  * the per-kernel-class split of a resident sweep (tssp_profile_begin / end);
  * prune end to end, wall clock on a fresh copy: plan -> fit() (Stage-2 search, Stage-1 scores from its baseline pass) ->
    select + gather -> bypass -> JSON files (bench.py's end_to_end_prune; the faster of two warm runs);
  * batch-256 inference (logits) of the dense and the pruned model;
and the card's name, power limit and maximum SM clock, read in the same run (read-only nvidia-smi query).

Writes one JSON document (default profiles/deit_r1.json). Needs a GPU; there is no CPU fallback.

    python tools/deit_bench.py [--images 1024] [--batch 256] [--steps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import contextlib
import copy
import ctypes as C
import io
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from long_seq_bench import gpu_info, timed  # noqa: E402

MODELS = {"deit_base_distilled_224": "base", "deit_tiny_distilled_224": "ti"}


def prune_end_to_end(api, model, batches, dev, sparsity: float, min_remaining: int) -> dict:
    quiet = io.StringIO()
    runs, work = [], None
    for _ in range(3):   # the first run also pays one-time costs (allocator segments, kernels paged in): reported apart
        if work is not None:
            api.release_engine(work)
        work = copy.deepcopy(model)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(quiet):
            plan = api.plan_2ssp_allocation(work, sparsity, min_remaining=min_remaining)
            iface = api.B200Auto2SSPInterface(work, batches, device=dev, batch_limit=None, min_remaining=min_remaining)
            att, mlp = iface.fit()
            res = api.prune_vit_mlp_width(work, n_to_prune_per_block=[plan.per_block_neurons_to_prune] * plan.num_blocks_total,
                                          strategy="act_l2", precomputed_importance=[m.float() for m in mlp], collect_masks=True,
                                          min_remaining=min_remaining)
            sel = torch.argsort(att)[: plan.blocks_to_prune].tolist()
            out = api.prune_vit_attention_blocks(work, 0.0, dataloader=None, device=dev, num_to_prune=plan.blocks_to_prune,
                                                 selected_indices=sel)
            with tempfile.TemporaryDirectory() as d:
                api.save_ffn_importances(mlp, os.path.join(d, "ffn_importances.json"))
                api.save_ffn_masks(res["ffn_prune_masks"], res["ffn_pruned_indices"], os.path.join(d, "ffn_prune_masks.json"),
                                   min_remaining=min_remaining)
                api.save_attention_indices(out["pruned_indices"], os.path.join(d, "attention_pruned_indices.json"))
        torch.cuda.synchronize()
        runs.append(time.perf_counter() - t0)
    before, after = api.count_total_params(model), api.count_total_params(work)
    return {"seconds": min(runs[1:]), "first_run_seconds": runs[0], "warm_runs": runs[1:], "K": plan.blocks_to_prune,
            "t": plan.per_block_neurons_to_prune, "pruned_attention_blocks": out["pruned_indices"], "sparsity_target": sparsity,
            "min_remaining": min_remaining, "achieved_sparsity": api.compute_actual_sparsity(before, after)}, work


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sparsity", type=float, default=0.375)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deit_r1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("deit_bench: no CUDA device", file=sys.stderr)
        return 2

    import __graft_entry__ as g
    g.build()
    import deit_synth as DS
    from oracle import twossp_oracle as O
    from twossp_b200 import _lib as L
    from twossp_b200 import api

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.load()
    res = {"what": "HF DeiTForImageClassificationWithTeacher, random-init weights (tests/deit_synth.make_deit), synthetic "
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

    for key, shape in MODELS.items():
        model = DS.make_deit(shape, 0, "teacher").to(dev)
        r = {"shape": dict(zip(("image", "patch", "hidden", "layers", "heads", "ffn", "labels"), DS.DEIT_SHAPES[shape])), "T": 198}
        eng = api.engine_for(model, dev, batch_hint=bs)

        def sweep_resident():
            eng.s1_reset()
            for b in dev_batches:
                eng.s1_batch(b)
            return eng.s1_score_sums(on_device=True)

        ms_res = timed(sweep_resident, args.steps, args.warmup)
        ms_host = timed(lambda: api._compute_ffn_activation_importance(model, host_batches, device=dev), args.steps, max(args.warmup, 2))
        r["s1_resident"] = {"ms_per_sweep": ms_res, "images_per_s": args.images / (ms_res * 1e-3)}
        r["s1_host_pixels"] = {"ms_per_sweep": ms_host, "images_per_s": args.images / (ms_host * 1e-3),
                               "api": "api._compute_ffn_activation_importance(model, pinned host batches, device='cuda')"}
        tb = [{"pixel_values": b} for b in dev_batches]
        ms_torch = timed(lambda: O.s1_scores(model, tb, str(dev), None, autocast=True), max(1, args.steps - 1), 1)
        r["torch_cuda_baseline"] = {"ms_per_sweep": ms_torch, "images_per_s": args.images / (ms_torch * 1e-3),
                                    "what": "O.s1_scores(model.cuda(), batches, 'cuda', autocast=True): HF module + hooks under CUDA autocast",
                                    "speedup_resident": ms_torch / ms_res, "speedup_host_pixels": ms_torch / ms_host}

        torch.cuda.synchronize()
        lib.tssp_profile_begin()
        for _ in range(2):
            sweep_resident()
        ms_arr = (C.c_double * len(L.PROFILE_CLASSES))()
        n_arr = (C.c_uint64 * len(L.PROFILE_CLASSES))()
        L.check(lib.tssp_profile_end(ms_arr, n_arr, len(L.PROFILE_CLASSES)))
        kernels = {name: {"ms_per_sweep": ms_arr[i] / 2, "launches_per_sweep": int(n_arr[i]) // 2}
                   for i, name in enumerate(L.PROFILE_CLASSES) if n_arr[i] > 0}
        total = sum(k["ms_per_sweep"] for k in kernels.values())
        for k in kernels.values():
            k["share"] = k["ms_per_sweep"] / total
        r["kernel_split_eager"] = {"classes": kernels, "sum_ms_per_sweep": total}

        with torch.no_grad():
            labels = torch.cat([eng.logits(b).argmax(-1) for b in dev_batches]).cpu()   # self-labels
        api.release_engine(model)
        batches = [{"pixel_values": px_host[s:s + bs], "labels": labels[s:s + bs]} for s in range(0, args.images, bs)]
        r["prune_end_to_end"], work = prune_end_to_end(api, model, batches, dev, args.sparsity, 256)

        infer = {}
        px256 = px_dev[:256]
        for name, m in (("dense", model), ("pruned", work)):
            e_ = api.engine_for(m, dev, batch_hint=256)
            ms = timed(lambda: e_.logits(px256), 5, 2)
            infer[f"{name}_images_per_s_batch256"] = 256 / (ms * 1e-3)
            api.release_engine(m)
        r["inference"] = infer
        res["models"][key] = r
        del model, work, eng
        api.trim_pool()
        torch.cuda.empty_cache()

    res["torch"] = torch.__version__
    res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
