"""Long-sequence measurement: ViT-B/16 at 384^2 (T = 577) on one B200.

  * Stage-1 sweep images/s through the API on resident device pixels and on pinned host pixels, and the same images
    through the torch CUDA baseline (the reference's algorithm, `O.s1_scores(..., autocast=True)`, as bench.py's
    torch_cuda_baseline runs it);
  * the per-kernel-class split of a resident sweep (tssp_profile_begin / end), attention's share in particular;
  * the attention kernel alone against torch SDPA (bf16) on the same [n, heads, T, 64] tensors, with achieved FLOP/s and
    the floors of the key-tiled kernel (TMEM read port, MUFU exp2, tensor pipe; DESIGN.md section 3);
  * the card's name, power limit and maximum SM clock, read in the same run (read-only nvidia-smi query).

Writes one JSON document (default profiles/long_seq_r3.json). Needs a GPU; there is no CPU fallback.

    python tools/long_seq_bench.py [--images 512] [--batch 128] [--steps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

IMAGE, PATCH, HEADS, HD = 384, 16, 12, 64
T = (IMAGE // PATCH) ** 2 + 1
SHAPE = (IMAGE, PATCH, 768, 12, HEADS, 3072, 1000)   # synth.SHAPES layout: ViT-B/16 at 384^2
# per-SM rates the floors are computed with (DESIGN.md section 3): TMEM read port, exp2 on the MUFU pipe, dense bf16 MMA
TMEM_READ_B_PER_CLK = 64
MUFU_EX2_PER_CLK = 16
MMA_BF16_FLOP_PER_CLK = 8192


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, power, sm = [x.strip() for x in r.stdout.strip().split(",")]
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(sm)}
    except Exception as exc:  # the numbers below still stand, without the card's settings beside them
        return {"name": torch.cuda.get_device_name(index), "error": f"nvidia-smi query failed: {exc}"}


def timed(fn, steps: int, warmup: int) -> float:
    """ms per call, CUDA events around `steps` calls after `warmup` untimed ones"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def attention_floors(n: int, sm_count: int, sm_mhz: float) -> dict:
    """Least time of one key-tiled attention launch on n images at T = 577 under each per-SM limit (padded work: every item
    is a 128-query x 128-key tile)."""
    mt = -(-T // 128)
    items = n * HEADS * mt * mt                      # (query tile, key tile) pairs; K / V are shared by a group's tiles
    per_item = {
        "tmem_read_clk": (128 * 128 * 4 + 128 * 64 * 4) / TMEM_READ_B_PER_CLK,   # S fp32 read + P bf16 read by the PV MMA
        "mufu_clk": 128 * 128 / MUFU_EX2_PER_CLK,
        "tensor_clk": 2 * (2 * 128 * 128 * 64) / MMA_BF16_FLOP_PER_CLK,
    }
    o_clk = n * HEADS * mt * (128 * 64 * 4) / TMEM_READ_B_PER_CLK      # O read out once per query tile
    out = {"items": items, "per_item_clk": per_item, "sm_mhz": sm_mhz}
    for k, v in per_item.items():
        clk = items * v + (o_clk if k == "tmem_read_clk" else 0.0)
        out[k.replace("_clk", "_ms")] = clk / sm_count / (sm_mhz * 1e3)
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--attn-iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_seq_r3.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("long_seq_bench: no CUDA device", file=sys.stderr)
        return 2

    import __graft_entry__ as g
    g.build()
    from oracle import synth
    from oracle import twossp_oracle as O
    from twossp_b200 import _lib as L
    from twossp_b200 import api, ops

    synth.SHAPES.setdefault("base384", SHAPE)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.load()
    props = torch.cuda.get_device_properties(dev)
    res = {"what": "ViT-B/16 at 384x384 (T = 577), synthetic N(0,1) images, random-init weights (oracle/synth.make_vit)",
           "gpu": gpu_info(dev.index), "sm_count": props.multi_processor_count, "images": args.images, "batch": args.batch,
           "steps": args.steps, "warmup": args.warmup, "timing": "CUDA events around whole sweeps"}

    gen = torch.Generator(device=dev).manual_seed(1234)
    px_dev = torch.randn(args.images, 3, IMAGE, IMAGE, device=dev, generator=gen)
    px_host = px_dev.cpu().pin_memory()
    bs = args.batch
    model = synth.make_vit("base384", seed=0).to(dev)
    eng = api.engine_for(model, dev, batch_hint=bs)
    dev_batches = [px_dev[s:s + bs] for s in range(0, args.images, bs)]
    host_batches = [{"pixel_values": px_host[s:s + bs]} for s in range(0, args.images, bs)]

    def sweep_resident():
        eng.s1_reset()
        for b in dev_batches:
            eng.s1_batch(b)
        return eng.s1_score_sums(on_device=True)

    def sweep_host():
        return api._compute_ffn_activation_importance(model, host_batches, device=dev)

    ms_res = timed(sweep_resident, args.steps, args.warmup)
    ms_host = timed(sweep_host, args.steps, max(args.warmup, 2))
    res["s1_resident"] = {"ms_per_sweep": ms_res, "images_per_s": args.images / (ms_res * 1e-3)}
    res["s1_host_pixels"] = {"ms_per_sweep": ms_host, "images_per_s": args.images / (ms_host * 1e-3),
                             "api": "api._compute_ffn_activation_importance(model, pinned host batches, device='cuda')"}

    # torch CUDA baseline: the reference's algorithm on the same images and batches (bench.py: torch_cuda_baseline)
    tb = [{"pixel_values": b} for b in dev_batches]
    ms_torch = timed(lambda: O.s1_scores(model, tb, str(dev), None, autocast=True), max(1, args.steps - 1), 1)
    res["torch_cuda_baseline"] = {"ms_per_sweep": ms_torch, "images_per_s": args.images / (ms_torch * 1e-3),
                                  "what": "O.s1_scores(model.cuda(), batches, 'cuda', autocast=True): HF module + hooks under CUDA autocast",
                                  "speedup_resident": ms_torch / ms_res, "speedup_host_pixels": ms_torch / ms_host}

    # per-kernel-class split of resident sweeps (eager launches, each bracketed by events)
    torch.cuda.synchronize()
    prof_steps = 2
    lib.tssp_profile_begin()
    for _ in range(prof_steps):
        sweep_resident()
    ms_arr = (C.c_double * len(L.PROFILE_CLASSES))()
    n_arr = (C.c_uint64 * len(L.PROFILE_CLASSES))()
    L.check(lib.tssp_profile_end(ms_arr, n_arr, len(L.PROFILE_CLASSES)))
    kernels = {name: {"ms_per_sweep": ms_arr[i] / prof_steps, "launches_per_sweep": int(n_arr[i]) // prof_steps}
               for i, name in enumerate(L.PROFILE_CLASSES) if n_arr[i] > 0}
    total = sum(k["ms_per_sweep"] for k in kernels.values())
    for k in kernels.values():
        k["share"] = k["ms_per_sweep"] / total
    res["kernel_split"] = {"classes": kernels, "sum_ms_per_sweep": total, "attention_share": kernels.get("attention", {}).get("share")}
    api.release_engine(model, trim=True)
    del eng

    # attention alone: the key-tiled kernel against SDPA on the same tensors
    n = bs
    D = HEADS * HD
    qkv = torch.randn(n * T, 3 * D, device=dev, generator=gen).bfloat16()
    q, k, v = (t.contiguous() for t in qkv.view(n, T, 3, HEADS, HD).permute(2, 0, 3, 1, 4))
    ms_ours = timed(lambda: ops.attention(qkv, n, T, HEADS), args.attn_iters, 3)
    ms_sdpa = timed(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v), args.attn_iters, 3)
    ours = ops.attention(qkv, n, T, HEADS).float().view(n, T, HEADS, HD)
    theirs = torch.nn.functional.scaled_dot_product_attention(q, k, v).float().permute(0, 2, 1, 3)
    flop = 4.0 * n * HEADS * T * T * HD
    sm_mhz = res["gpu"].get("sm_max_mhz") or 1965.0
    floors = attention_floors(n, props.multi_processor_count, sm_mhz)
    bound = max(("tmem_read_ms", "mufu_ms", "tensor_ms"), key=lambda x: floors[x])
    res["attention"] = {"shape": {"n": n, "heads": HEADS, "T": T, "head_dim": HD}, "flop_per_call": flop,
                        "ours_ms": ms_ours, "ours_tflops": flop / (ms_ours * 1e-3) / 1e12,
                        "sdpa_ms": ms_sdpa, "sdpa_tflops": flop / (ms_sdpa * 1e-3) / 1e12,
                        "speedup_vs_sdpa": ms_sdpa / ms_ours, "max_abs_diff_vs_sdpa": float((ours - theirs).abs().max()),
                        "floors": floors, "bounding_floor": bound, "frac_of_bounding_floor": floors[bound] / ms_ours,
                        "sdpa_backend": "torch.nn.functional.scaled_dot_product_attention, bf16 [n, heads, T, 64], backend chosen by torch"}
    res["torch"] = torch.__version__
    res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
