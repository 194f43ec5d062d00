"""uint8 against fp32 host batches: the Stage-1 sweep through the API (`_compute_ffn_activation_importance` on pinned host
batches) fed the same images as normalised fp32 pixels and as uint8 bytes normalised on the device.

Per model (ViT-B/16 and DeiT-Ti/16 at 224^2, seeded weights, one fixed set of random uint8 images split evenly over the
ranks):
  * ms per sweep and images/s of both input forms, alternated for `--rounds` rounds after one warm-up sweep of each. Each
    sweep sits between a barrier and a device synchronise and is timed with a host clock (the call ends by copying the
    scores to the host); the max over ranks is reported;
  * the device-resident rate (fp32 batches already on the GPU, same API call) beside them for reference;
  * host-to-device bytes per image of both forms;
  * a check in the same run that the uint8 and fp32 scores are torch.equal (the script fails otherwise);
and, on rank 0, im2col at the ViT-B/16 shape (256 images, P = 16) from fp32 and from uint8 pixels, alternated, as
microseconds per launch of the library entry point (CUDA events, outputs preallocated) and as the kernels' device time
from torch.profiler. Four input buffers are used in turn, so the uint8 working set (154 MB) does not fit in L2 either.
The card's name, power limit and maximum SM clock are read in the same run (a read-only nvidia-smi query).

Run under torchrun; each run adds its result to the JSON document at --out under "n<world size>":

    torchrun --nproc-per-node N tools/uint8_input_bench.py [--images 1024] [--batch 256] [--rounds 3] [--out FILE]
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

from long_seq_bench import gpu_info, timed  # noqa: E402

IMAGENET = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))


def make_model(name: str):
    from oracle import synth
    import deit_synth as DS
    return {"vit_b16_224": lambda: synth.make_vit("base", seed=0), "deit_ti16_224": lambda: DS.make_deit("ti", head="teacher")}[name]()


def im2col_times(api, ops, dev, rounds: int) -> dict:
    from twossp_b200 import _lib as L
    lib = L.load()
    n, P, H = 256, 16, 224
    T, K = (H // P) ** 2 + 1, 3 * P * P
    gen = torch.Generator(device=dev).manual_seed(5)
    u8 = [torch.randint(0, 256, (n, 3, H, H), device=dev, dtype=torch.uint8, generator=gen) for _ in range(4)]
    f32 = [api.normalize_pixels(u, *IMAGENET) for u in u8]
    for u, f in zip(u8, f32):
        assert torch.equal(ops.im2col(u, P, mean=IMAGENET[0], std=IMAGENET[1]), ops.im2col(f, P))
    # outputs allocated and arguments marshalled once: the timed loop is the library call and the kernel launch only
    outs = [torch.empty(n * T, K, device=dev, dtype=torch.bfloat16) for _ in range(4)]
    norm = L.pixel_input(L.PIXELS_U8, IMAGENET[0], IMAGENET[1], 1 / 255)
    stream = L.current_stream()
    args_f = [(C.c_void_p(f.data_ptr()), C.c_void_p(o.data_ptr())) for f, o in zip(f32, outs)]
    args_u = [(C.c_void_p(u.data_ptr()), C.c_void_p(o.data_ptr())) for u, o in zip(u8, outs)]
    it = {"i": 0}

    def run(fp32: bool):
        def fn():
            i = it["i"] = (it["i"] + 1) % 4
            if fp32:
                rc = lib.tssp_op_im2col(*args_f[i], n, 3, H, H, P, 1, None, stream)
            else:
                rc = lib.tssp_op_im2col(*args_u[i], n, 3, H, H, P, 1, norm, stream)
            if rc:
                L.check(rc)
        return fn
    out = {"fp32": [], "uint8": []}
    for _ in range(rounds):
        out["fp32"].append(timed(run(True), 200, 10) * 1e3)
        out["uint8"].append(timed(run(False), 200, 10) * 1e3)
    # the same launches under torch.profiler: device time of the kernels themselves
    from torch.profiler import ProfilerActivity, profile
    kernel_us = {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            run(True)()
            run(False)()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "im2col_patches" in ev.key:   # im2col_patches_kernel / im2col_patches_u8_kernel
            kernel_us["uint8" if "u8_kernel" in ev.key else "fp32"] = ev.device_time
    written = n * T * K * 2
    res = {"images": n, "patch": P, "image": H,
           "what": "us per launch: CUDA events over 200 launches of the library entry point (outputs preallocated, 4 input "
                   "buffers in turn), median round, rounds listed; kernel_us_profiler: mean device time of the kernel from "
                   "torch.profiler over 50 launches of each"}
    for k, v in out.items():
        med = sorted(v)[len(v) // 2]
        read = n * 3 * H * H * (4 if k == "fp32" else 1)
        res[k] = {"us_per_launch": med, "rounds_us": v, "kernel_us_profiler": kernel_us.get(k), "bytes_read": read,
                  "bytes_written": written, "GB_per_s": (read + written) / (med * 1e-6) / 1e9}
    res["uint8_over_fp32"] = res["uint8"]["us_per_launch"] / res["fp32"]["us_per_launch"]
    return res


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=1024, help="images in the whole set, split over the ranks")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "uint8_input_r1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("uint8_input_bench: no CUDA device", file=sys.stderr)
        return 2
    import torch.distributed as dist
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
        from twossp_b200 import distributed as D
        D.bind_host_to_gpu(local)   # as bench.py: pinned batches on the GPU's own NUMA node
    if rank == 0:
        import __graft_entry__ as g
        g.build()
    if world > 1:
        dist.barrier()
    from twossp_b200 import api, ops

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        return float(t.item())

    def sweep_ms(fn) -> tuple:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return max_over_ranks((time.perf_counter() - t0) * 1e3), out

    per_rank = args.images // world
    bs = min(args.batch, per_rank)
    res = {"world_size": world, "gpu": gpu_info(local), "images": per_rank * world, "images_per_rank": per_rank,
           "batch_per_rank": bs, "rounds": args.rounds, "mean_std": IMAGENET, "rescale": "1/255",
           "api": "api._compute_ffn_activation_importance(model, pinned host batches, device, group=WORLD if N > 1)",
           "timing": "barrier, synchronize, host clock around one whole sweep, synchronize; max over ranks; median round",
           "models": {}}
    for name in ("vit_b16_224", "deit_ti16_224"):
        model = make_model(name).to(dev)
        g = torch.Generator().manual_seed(2024)
        u_all = torch.randint(0, 256, (per_rank * world, 3, 224, 224), dtype=torch.uint8, generator=g)
        u = u_all[rank * per_rank:(rank + 1) * per_rank]
        f = api.normalize_pixels(u, *IMAGENET)
        u_pin, f_pin = u.clone().pin_memory(), f.pin_memory()
        f_dev = f.to(dev)
        forms = {"fp32": [{"pixel_values": f_pin[s:s + bs]} for s in range(0, per_rank, bs)],
                 "uint8": [{"pixel_values": u_pin[s:s + bs]} for s in range(0, per_rank, bs)],
                 "resident_fp32": [{"pixel_values": f_dev[s:s + bs]} for s in range(0, per_rank, bs)]}
        api.set_pixel_normalization(model, *IMAGENET)

        def sweep(form):
            return lambda: api._compute_ffn_activation_importance(model, forms[form], device=dev, group=group)
        scores = {k: sweep_ms(sweep(k))[1] for k in forms}   # warm-up: engine, graphs, pinned staging
        same = all(torch.equal(a, b) for a, b in zip(scores["uint8"], scores["fp32"]))
        same_res = all(torch.equal(a, b) for a, b in zip(scores["uint8"], scores["resident_fp32"]))
        assert same and same_res, f"{name}: uint8 and fp32 scores differ"
        times = {k: [] for k in forms}
        for _ in range(args.rounds):
            for k in ("fp32", "uint8", "resident_fp32"):
                ms, out = sweep_ms(sweep(k))
                times[k].append(ms)
                assert all(torch.equal(a, b) for a, b in zip(out, scores["fp32"])), f"{name}: {k} scores changed between sweeps"
        chw = 3 * 224 * 224
        r = {"scores_torch_equal_uint8_fp32": same, "h2d_bytes_per_image": {"fp32": chw * 4, "uint8": chw}}
        for k, v in times.items():
            med = sorted(v)[len(v) // 2]
            r[k] = {"ms_per_sweep": med, "rounds_ms": v, "images_per_s": per_rank * world / (med * 1e-3)}
        r["uint8_over_fp32_rate"] = r["uint8"]["images_per_s"] / r["fp32"]["images_per_s"]
        res["models"][name] = r
        api.release_engine(model)
        del model, u_pin, f_pin, f_dev, forms
        api.trim_pool()
        torch.cuda.empty_cache()
    if rank == 0:
        res["im2col_b16"] = im2col_times(api, ops, dev, max(args.rounds, 3))
        res["torch"] = torch.__version__
        res["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
        doc = {}
        if os.path.exists(args.out):
            with open(args.out) as fh:
                doc = json.load(fh)
        doc.setdefault("what", __doc__.split("\n\n")[0].replace("\n", " "))
        doc.setdefault("runs", {})[f"n{world}"] = res
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
        print(json.dumps(res, indent=1))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
