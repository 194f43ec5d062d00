"""bench.py -- the reference's headline metric on B200: ViT-B/16 2SSP calibration images/s (+ end-to-end prune
seconds), BASELINE.json configs[2]: 37.5 % sparsity plan, 1024 synthetic 224x224 calibration images IN TOTAL,
data-parallel over the GPUs of the run (rank r sweeps its contiguous 1024/N share: 4 / 2 / 1 batches of 256 at
1 / 2 / 4 GPUs, one batch of 128 at 8), random-init weights.

    python bench.py [--gpus N --steps K --warmup W]            # this repository's CUDA path (one rank per GPU)
    python bench.py --impl reference [...]                     # the reference's CPU path (oracle port) on host cores
    python bench.py [...] --dump-outputs DIR                   # also save the last timed step's results as DIR/*.npy

A step = one Stage-1 calibration sweep over the whole 1024-image calibration set: embeddings, 12 encoder blocks with the
fused fc1+GELU+score GEMM, score finisher, and for N>1 the all-reduce of the score vector. `scaling` is "strong": the
work per step is fixed, so `value` at N GPUs against N x the 1-GPU value is the data-parallel efficiency of the path.
`value` has the images resident in HBM; `e2e` goes through the reference-facing API call
(`_compute_ffn_activation_importance`) with pinned HOST batches, H2D copies and the D2H score read inside the timed
region. Extra keys: `weak` (every rank sweeps all 1024 images: last round's line), `torch_cuda_baseline` (the reference
algorithm as it would run with device="cuda": HF module + hooks under CUDA autocast, on this GPU, same images),
`prune_e2e` (+ top-level `prune_e2e_seconds`), `configs` (BASELINE configs 2, 4 and 5). One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import contextlib
import copy
import ctypes as C
import io
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_TOKENS = 197
MODEL_NAMES = {"small": "ViT-S/16", "base": "ViT-B/16 (google/vit-base-patch16-224 shape)", "large": "ViT-L/16"}
SHAPE = {"small": (384, 1536, 12), "base": (768, 3072, 12), "large": (1024, 4096, 24)}   # D, F, blocks
PLAN_T = {("small", 0.375): 576, ("base", 0.25): 661, ("base", 0.375): 1120, ("base", 0.5): 1450, ("large", 0.5): 2070}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--images", type=int, default=1024, help="calibration images in total (sharded over the ranks)")
    ap.add_argument("--batch", type=int, default=256, help="images per calibration batch (64 / 128 / 256 / 512 measured: profiles/batch_sweep_r1.txt)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--ref-images", type=int, default=256, help="--impl reference: cap on the images of one step's bounded sample")
    ap.add_argument("--no-prune", action="store_true", help="skip the end-to-end prune timing")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="diagnosis only: do not sample nvidia-smi during the timed regions")
    ap.add_argument("--no-extra", action="store_true", help="skip torch_cuda_baseline, weak scaling and the other BASELINE configs")
    ap.add_argument("--model", default="base", choices=["small", "base", "large"], help="other BASELINE configs as the main line (not the bench line)")
    ap.add_argument("--sparsity", type=float, default=0.375)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save what the last one returned, float32: DIR/s1_score_sums.npy (resident sweep: "
                         "per-neuron sums over all images, blocks concatenated) and DIR/ffn_importance.npy (API call: [blocks, F])")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm (the reference arm sizes its sample by the host's speed)")
    return args


def flops_per_image(D=768, F=3072, B=12, T=T_TOKENS, C=1000):
    # SURVEY.md section 8d: B*(24 T D^2 + 4 T^2 D) + patch embed + head = 35.13 GFLOP for ViT-B/16
    return B * (24 * T * D * D + 4 * T * T * D) + 2 * 196 * 768 * D + 2 * D * C


def s1_flops_per_image(D=768, F=3072, B=12, T=T_TOKENS):
    # the Stage-1 sweep stops after the last block's fc1: no last fc2, final LN or head
    # (general F: the 24 T D^2 term assumes F = 4 D, true for ViT-S/B/L)
    return flops_per_image(D, F, B, T, 0) - 2 * T * D * F


def bench_config(args, world: int) -> dict:
    """The `config` object of the JSON line -- the SAME for both arms (derived from the arguments alone), so that the
    driver can pair them."""
    per_rank = -(-args.images // world)
    return {"workload": (f"{MODEL_NAMES[args.model]}, random init, 2SSP Stage-1 calibration sweep, {args.sparsity:.1%} sparsity plan, "
                         f"{args.images} synthetic 224x224 images in total, batches of up to {args.batch}"),
            "images_per_step": args.images, "batch": args.batch, "images_per_rank": per_rank, "batch_per_rank": min(args.batch, per_rank),
            "parallelism": f"dp{world}: images sharded over {world} ranks, one all-reduce of the score vector per step" if world > 1 else "single GPU",
            "l2": ("step k gives rank r shard (r + k) mod N of the resident image set: no rank re-reads pixels it has just had in L2, and every "
                   "batch streams > 2 GB of activations through the 126 MB L2" if world > 1 else
                   f"inputs are larger than L2 ({args.images * 3 * 224 * 224 * 4 / 1e6:.0f} MB of pixels per step vs 126 MB)"),
            "graphs": "per-batch launch chains replayed as CUDA graphs (TSSP_GRAPHS=0 for eager launches)"}


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); power.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, power) if p > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"burst": p.get("bf16_tflops"), "sustained": p.get("bf16_tflops_sustained"), "hbm_gbs": p.get("hbm_gbs"), "source": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def ncu_traffic():
    """dram bytes per launch of the fc1 kernel from the committed ncu capture, if any (profiles/fc1_traffic.json)."""
    path = os.path.join(ROOT, "profiles", "fc1_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("dram_bytes_per_launch")
    return None


# ======================================================================================= reference arm (CPU)
def cpu_s1_rate(model_cpu, n_images: int, batch: int, threads: int):
    """images/s of the oracle port of the reference's Stage-1 sweep (CPU autocast = bf16, as the reference runs)."""
    from oracle import synth
    from oracle import twossp_oracle as O
    px = synth.make_pixels(n_images, 224, seed=4321)
    batches = synth.make_batches(px, None, batch)
    t0 = time.perf_counter()
    O.s1_scores(model_cpu, batches, "cpu", None, autocast=True)
    dt = time.perf_counter() - t0
    return n_images / dt, dt


def cpu_batch(n: int, bench_batch: int) -> int:
    """The reference arm runs the bench arm's batch size whenever the bounded sample holds a whole batch; the fp32
    activations of one ViT-B batch of 256 are 2.5 GB on the host, well inside the box."""
    return bench_batch if n >= bench_batch else n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import synth
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    model = synth.make_vit(args.model, seed=0)
    probe_rate, _ = cpu_s1_rate(model, 8, 8, threads)
    budget = 170.0 / max(1, args.steps + args.warmup)                 # whole run within a few minutes
    n = int(max(8, min(args.ref_images, probe_rate * min(budget, 12.0))))
    n = n - n % args.batch if n >= args.batch else n - n % 8
    bs = cpu_batch(n, args.batch)
    for _ in range(args.warmup):
        cpu_s1_rate(model, n, bs, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_s1_rate(model, n, bs, threads)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = (f"{n} images per step in batches of {bs} (bounded sample of the {args.images}-image workload; the bench arm's batch is "
              f"{args.batch}), CPU autocast bf16, {threads} threads")
    line = {
        "impl": "reference", "metric": "calibration_images_per_s", "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": bench_config(args, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ======================================================================================= this repository's arm
class Ctx:
    """What every measurement below needs: process group, device, library handles."""

    def __init__(self):
        import torch.distributed as dist
        from twossp_b200 import _lib as L
        from twossp_b200 import api
        self.dist, self.L, self.api = dist, L, api
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.group = None
        self.host_binding = None
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD
            # one process per GPU: keep it (and the pinned batches it allocates from here on) on the GPU's own NUMA node;
            # a no-op on single-node hosts. Not at N=1, where the cpu_baseline leg wants every core.
            from twossp_b200 import distributed as D
            self.host_binding = D.bind_host_to_gpu(self.local)
        if self.rank == 0:
            import __graft_entry__ as g
            g.build()
        self.barrier()
        self.lib = L.load()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, ms: float) -> float:
        if self.world == 1:
            return ms
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        """W untimed calls, then K calls between barrier + synchronize, CUDA events on the launching stream, max over ranks.
        Returns (ms, launches, what the last timed call returned)."""
        for i in range(warmup):
            fn(i)
        self.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = self.lib.tssp_launch_count()
        e0.record()
        for i in range(steps):
            last = fn(warmup + i)
        e1.record()
        torch.cuda.synchronize()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)), int(self.lib.tssp_launch_count() - l0), last


def shard(n: int, rank: int, world: int) -> slice:
    from twossp_b200 import distributed as D
    return D.shard_slice(n, rank, world)


def measure_sweep(cx: Ctx, model_name: str, model, px_dev, px_host, bs: int, steps: int, warmup: int, profile: bool, weak: bool,
                  outputs: bool = False):
    """Stage-1 sweep of the whole calibration set, sharded over the ranks (strong scaling): device-timed value, the
    end-to-end API arm, optionally the weak-scaling line and the per-kernel-class profile."""
    api, L, lib, world, rank, dev = cx.api, cx.L, cx.lib, cx.world, cx.rank, cx.dev
    n_total = px_dev.shape[0]
    shards = [shard(n_total, r, world) for r in range(world)]
    n_local = shards[rank].stop - shards[rank].start
    bs_local = max(1, min(bs, max(s.stop - s.start for s in shards)))
    eng = api.engine_for(model, dev, batch_hint=bs_local)
    sum_f = sum(eng.ffn_dims)

    def batches_of(sl: slice, src):
        return [src[s:min(s + bs_local, sl.stop)] for s in range(sl.start, sl.stop, bs_local)]

    # Strong scaling: step k gives rank r the shard (r + k) mod N of the resident set, so the 1024 images are swept
    # exactly once per step by the N ranks together and no rank re-reads the pixels it has just had in L2.
    dev_shards = [batches_of(sl, px_dev) for sl in shards]
    host_batches = [{"pixel_values": b} for b in batches_of(shards[rank], px_host)]

    def sweep(batches):
        eng.s1_reset()
        for b in batches:
            eng.s1_batch(b)
        sums = eng.s1_score_sums(on_device=True)
        if world > 1:
            cx.dist.all_reduce(sums, group=cx.group)
        return sums

    def step_resident(k):
        return sweep(dev_shards[(rank + k) % world])

    def step_weak(k):
        return sweep([b for sh in dev_shards for b in sh])

    def step_e2e(k):
        return api._compute_ffn_activation_importance(model, host_batches, device=dev, group=cx.group)

    out = {"images": n_total, "batch": bs_local, "images_per_rank": n_local}
    ms, launches, sums = cx.timed(step_resident, steps, warmup)
    out.update(ms_total=ms, launches=launches, value=n_total * steps / (ms * 1e-3), ms_per_step=ms / steps)
    # the host-batch path settles over its first ~7 calls (tools/e2e_scaling_probe.py: 13.9 -> 11.5 ms per call at 4 ranks
    # right after the resident loop), so it gets its own warm-up of at least 8 calls
    e2e_warmup = max(warmup, 8)
    ms_e, _, importance = cx.timed(step_e2e, steps, e2e_warmup)
    if outputs:
        # what each timed path hands its caller in the last step: the engine's score sums over all images (device, flat)
        # and the API's per-block importance (host, sums / images)
        out["outputs"] = {"s1_score_sums": sums.cpu().numpy(), "ffn_importance": torch.stack(importance).numpy()}
    out["e2e"] = {"value": n_total * steps / (ms_e * 1e-3), "unit": "images/s", "ms_per_step": ms_e / steps, "warmup": e2e_warmup,
                  "h2d_bytes_per_step": int(n_total * 3 * 224 * 224 * 4), "d2h_bytes_per_step": int(sum_f * 4 * world),
                  "api": "twossp_b200.api._compute_ffn_activation_importance(model, pinned host batches of the rank's shard, device='cuda', group=...)"}
    if weak and world > 1:
        ms_w, _, _ = cx.timed(step_weak, max(2, steps // 2), 2)
        out["weak"] = {"value": n_total * world * max(2, steps // 2) / (ms_w * 1e-3), "unit": "images/s", "ms_per_step": ms_w / max(2, steps // 2),
                       "images_per_gpu_per_step": n_total, "note": "every rank sweeps the whole set (last round's headline): work grows with N"}
    D_, F_, B_ = SHAPE[model_name]
    out["step_tflops"] = s1_flops_per_image(D_, F_, B_) * n_total / (out["ms_per_step"] * 1e-3) / 1e12
    out["sum_f"] = sum_f
    if profile:
        # per-kernel device times, CUDA events on the launching stream, over the same steps re-run with instrumentation
        # (eager launches: a captured chain cannot carry the events)
        prof_steps = max(2, min(steps, 5))
        torch.cuda.synchronize()
        lib.tssp_profile_begin()
        t0 = time.perf_counter()
        for k in range(prof_steps):
            step_resident(k)
        ms_arr = (C.c_double * len(L.PROFILE_CLASSES))()
        n_arr = (C.c_uint64 * len(L.PROFILE_CLASSES))()
        L.check(lib.tssp_profile_end(ms_arr, n_arr, len(L.PROFILE_CLASSES)))
        out["ms_per_step_instrumented"] = 1e3 * (time.perf_counter() - t0) / prof_steps
        kernels = {name: {"ms_per_step": ms_arr[i] / prof_steps, "launches_per_step": int(n_arr[i]) // prof_steps}
                   for i, name in enumerate(L.PROFILE_CLASSES) if n_arr[i] > 0}
        out["kernels"] = kernels
        peaks = measured_peaks()
        fc1 = kernels.get("fc1_gelu_score")
        if fc1:
            M, N, K = bs_local * T_TOKENS, F_, D_
            flop = 2.0 * M * N * K                                   # algorithmic FLOPs of one fused fc1 launch (one batch, one block)
            avg_ms = fc1["ms_per_step"] / fc1["launches_per_step"]
            achieved = flop / (avg_ms * 1e-3) / 1e12
            out["roofline"] = {"kernel": "gemm_bf16_tn_kernel<EPI_BF16_GELU_SCORE> (fc1 + bias + GELU + per-image sum of squares)",
                               "bound": "tensor", "achieved": achieved, "peak": peaks["sustained"], "unit": "TFLOP/s",
                               "frac": achieved / peaks["sustained"], "peak_kind": f"{peaks['source']} cuBLAS bf16, sustained",
                               "frac_of_burst_peak": achieved / peaks["burst"], "frac_of_nominal_2250": achieved / 2250.0,
                               "flop_per_launch": flop, "avg_launch_ms": avg_ms, "launches_per_step": fc1["launches_per_step"],
                               "share_of_step": fc1["ms_per_step"] / max(1e-9, sum(k["ms_per_step"] for k in kernels.values())),
                               "traffic": ncu_traffic() if (model_name == "base" and bs_local == 256) else None}
        hbm_peak = peaks.get("hbm_gbs") or 6555.2
        hbm = {"peak_gbs": hbm_peak, "peak_kind": f"{peaks['source']} copy bandwidth"}
        M_rows = bs_local * T_TOKENS
        ln = kernels.get("layernorm")
        if ln:
            us = 1e3 * ln["ms_per_step"] / ln["launches_per_step"]
            byt = M_rows * D_ * 6                                    # fp32 row read + bf16 row written
            hbm["layernorm"] = {"bytes_per_launch": byt, "us_per_launch": us, "achieved_gbs": byt / us / 1e3, "frac": byt / us / 1e3 / hbm_peak}
        sf = kernels.get("score_finish")
        if sf:
            pairs = sum(((i + 1) * T_TOKENS - 1) // 32 - (i * T_TOKENS) // 32 + 1 for i in range(bs_local))   # (image, 32-row sub-tile) pairs
            byt = B_ * (pairs * F_ * 4 + bs_local * F_ * 4) + bs_local * B_ * F_ * 4   # partials read + norms written, norms read again
            us = 1e3 * sf["ms_per_step"] / (sf["launches_per_step"] / 2)               # the two finisher kernels of one batch together
            hbm["score_finish"] = {"bytes_per_batch": byt, "us_per_batch": us, "achieved_gbs": byt / us / 1e3, "frac": byt / us / 1e3 / hbm_peak}
        out["hbm_kernels"] = hbm
    return out


def gather_bandwidth(cx: Ctx, model, model_name: str, sparsity: float, hbm_peak: float):
    """The batched neuron gather against the measured copy bandwidth (north_star subsystem 2)."""
    from twossp_b200 import ops
    api, L, lib, dev = cx.api, cx.L, cx.lib, cx.dev
    D_m, F_m, B_m = SHAPE[model_name]
    pairs_mlp = api.gather_mlp_pairs(model)
    keep_n = F_m - PLAN_T.get((model_name, sparsity), F_m * 3 // 8)
    gen_k = torch.Generator(device=dev).manual_seed(7)
    blocks = [(a.weight.detach(), a.bias.detach(), b.weight.detach(),
               torch.sort(torch.randperm(F_m, device=dev, generator=gen_k)[:keep_n])[0]) for a, b in pairs_mlp]
    g_args, g_outs, g_hold = ops.ffn_gather_batch_plan(blocks)
    flush = torch.empty(64 << 20, device=dev)
    stream = L.current_stream()
    times = []
    for _ in range(7):
        flush.fill_(0.0)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        L.check(lib.tssp_ffn_gather_batch(*g_args, stream))
        a1.record()
        torch.cuda.synchronize()
        times.append(a0.elapsed_time(a1) * 1e3)
    us = sorted(times)[len(times) // 2]
    alg = B_m * 2 * (keep_n * D_m + keep_n + D_m * keep_n) * 4
    moved = B_m * ((keep_n * D_m + keep_n + D_m * F_m) * 4 + (keep_n * D_m + keep_n + D_m * keep_n) * 4)
    return {"blocks": B_m, "keep": keep_n, "algorithmic_bytes": alg, "moved_bytes": moved, "us_per_launch": us,
            "achieved_gbs": alg / us / 1e3, "moved_gbs": moved / us / 1e3, "frac": moved / us / 1e3 / hbm_peak,
            "note": "all blocks in one launch, L2 flushed before each; moved = algorithmic + the dropped W2 columns (same sectors)"}


def s2_shard_mode(n_total: int, world: int) -> str:
    """Image shards as soon as every rank gets a workable batch: no rank then repeats the baseline pass on images it does not
    own (B + B(B+1)/2 block-forwards on n/N images each, against B on ALL images + B(B+1)/2N with candidate sharding)."""
    return "images" if world > 1 and n_total // world >= 32 else "candidates"


def end_to_end_prune(cx: Ctx, model, px_host, bs: int, sparsity: float, shard_mode=None, inference: bool = True):
    """plan -> fit (Stage-2 search + Stage-1 scores) -> select+gather -> bypass install -> masks/JSON, wall clock, on a copy."""
    api, dev, group, rank, world = cx.api, cx.dev, cx.group, cx.rank, cx.world
    n = px_host.shape[0]
    mode = shard_mode or s2_shard_mode(n, world)
    eng = api.engine_for(model, dev, batch_hint=bs)
    with torch.no_grad():
        labels = torch.cat([eng.logits(px_host[s:s + bs]).argmax(-1) for s in range(0, n, bs)]).cpu()   # self-labels
    api.release_engine(model)
    mine = shard(n, rank, world) if mode == "images" else slice(0, n)
    bs_local = max(1, min(bs, mine.stop - mine.start))
    batches = [{"pixel_values": px_host[s:min(s + bs_local, mine.stop)], "labels": labels[s:min(s + bs_local, mine.stop)]}
               for s in range(mine.start, mine.stop, bs_local)]
    quiet = io.StringIO()
    runs = []
    # Three complete runs, each on a fresh copy of the model. The first also pays one-time costs that are not the pruning
    # flow's (torch's sort / nonzero kernels being paged in on a fresh box, cudaMalloc of the allocator's first segments)
    # and is kept as `first_run_seconds`; the faster of the two warm runs is reported and both are listed (`warm_runs`):
    # with several ranks on one node a single cudaMalloc inside torch's allocator occasionally stalls a run by 0.2 s.
    work = None
    phases = []
    for attempt in range(3):
        if work is not None:
            api.release_engine(work)
        work = copy.deepcopy(model)
        cx.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(quiet):
            plan = api.plan_2ssp_allocation(work, sparsity, min_remaining=512)
            iface = api.B200Auto2SSPInterface(work, batches, device=dev, batch_limit=None, min_remaining=512, group=group, s2_shard=mode)
            api.engine_for(work, dev, batch_hint=bs_local, need_cache=True)   # engine build (HBM allocation, weight packing) timed here
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            att, mlp = iface.fit()   # Stage-2 search; its baseline pass also yields the Stage-1 scores (fuse_passes)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            res = api.prune_vit_mlp_width(work, n_to_prune_per_block=[plan.per_block_neurons_to_prune] * plan.num_blocks_total, strategy="act_l2",
                                          precomputed_importance=[m.float() for m in mlp], collect_masks=True, min_remaining=512)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            sel = torch.argsort(att)[: plan.blocks_to_prune].tolist()
            out = api.prune_vit_attention_blocks(work, 0.0, dataloader=None, device=dev, num_to_prune=plan.blocks_to_prune, selected_indices=sel)
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            if rank == 0:
                with tempfile.TemporaryDirectory() as d:
                    api.save_ffn_importances(mlp, os.path.join(d, "ffn_importances.json"))
                    api.save_ffn_masks(res["ffn_prune_masks"], res["ffn_pruned_indices"], os.path.join(d, "ffn_prune_masks.json"), min_remaining=512)
                    api.save_attention_indices(out["pruned_indices"], os.path.join(d, "attention_pruned_indices.json"))
        t5 = time.perf_counter()
        runs.append(cx.max_over_ranks(1e3 * (t5 - t0)) / 1e3)
        phases.append((t0, t1, t2, t3, t4, t5))
    best = 1 if runs[1] <= runs[2] else 2
    t0, t1, t2, t3, t4, t5 = phases[best]
    before = api.count_total_params(model)
    after = api.count_total_params(work)
    result = {"seconds": runs[best], "first_run_seconds": runs[0], "warm_runs": runs[1:], "plan_engine_s": t1 - t0, "fit_s": t2 - t1,
              "fit": "Stage-2 search with the Stage-1 scores taken from its baseline pass (one sweep fewer)",
              "select_gather_s": t3 - t2, "bypass_install_s": t4 - t3, "json_s": t5 - t4,
              "stage2_sharding": mode, "images": int(n), "images_per_rank": mine.stop - mine.start, "K": plan.blocks_to_prune,
              "t": plan.per_block_neurons_to_prune, "pruned_attention_blocks": out["pruned_indices"],
              "achieved_sparsity": api.compute_actual_sparsity(before, after),
              "stage2_block_forwards_per_batch": sum(plan.num_blocks_total - i for i in range(plan.num_blocks_total)) + plan.num_blocks_total}
    if inference:
        # BASELINE configs[4]: inference throughput of the pruned model (odd FFN widths, bypassed attention) at batch 256
        infer = {}
        try:
            eng_p = api.engine_for(work, dev, batch_hint=256)
            eng_d = api.engine_for(model, dev, batch_hint=256)
            px256 = px_host[:256].to(dev)
            for name, e_ in (("dense", eng_d), ("pruned", eng_p)):
                for _ in range(2):
                    e_.logits(px256)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    e_.logits(px256)
                e1.record()
                torch.cuda.synchronize()
                infer[f"{name}_images_per_s_batch256"] = 5 * 256 / (e0.elapsed_time(e1) * 1e-3)
        except Exception as exc:  # never let the secondary number take the headline down
            infer["error"] = repr(exc)
        result["inference"] = infer
        api.release_engine(model)
    api.release_engine(work)
    return result


def torch_cuda_baseline(cx: Ctx, model_name: str, px_dev, bs: int, ours_value: float, ours_model):
    """The like-for-like GPU baseline (SURVEY 2a / 8c, oracle mode O-cuda-asis): the reference's algorithm as it runs with
    device="cuda" -- HF module + forward hooks under CUDA autocast (fp16 GEMMs through cuBLASLt, eager GELU, fp32
    vector_norm / sum, one .to("cpu") per block per batch) -- on THIS GPU, same images, same batch size. The oracle port
    restates src/vit_pruning.py:143-158,173-185 (the reference itself is not on the GPU box). Stage 2 the reference's way
    (deepcopy + bypass + full evaluation per candidate, mask_conjunction.py:327-357) on one batch of 256, next to ours."""
    from oracle import synth
    from oracle import twossp_oracle as O
    dev = cx.dev
    out = {}
    model = synth.make_vit(model_name, seed=0).to(dev)
    n = px_dev.shape[0]
    batches = [{"pixel_values": px_dev[s:s + bs]} for s in range(0, n, bs)]
    O.s1_scores(model, batches[:1], str(dev), None, autocast=True)             # warm-up (cuBLAS handles, autotuning)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    e0.record()
    for _ in range(reps):
        ref_scores = O.s1_scores(model, batches, str(dev), None, autocast=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    out.update(value=n / (ms * 1e-3), unit="images/s", ms_per_step=ms, images=n, batch=bs,
               what="oracle port of _compute_ffn_activation_importance on model.cuda() under torch.autocast('cuda') (fp16), hooks + vector_norm + per-block .to('cpu')",
               speedup_of_this_repo=ours_value / (n / (ms * 1e-3)))
    # agreement of the two GPU paths (both low-precision forwards of the same fp32 model)
    ours = torch.stack(cx.api._compute_ffn_activation_importance(ours_model, batches, device=dev))
    theirs = torch.stack([s.float() for s in ref_scores])
    out["max_rel_diff_vs_this_repo"] = float(((ours - theirs).abs() / theirs.abs().clamp_min(1e-12)).max())
    # Stage 2 on one batch of 256 self-labelled images
    px = px_dev[:256]
    with torch.no_grad(), torch.autocast("cuda"):
        labels = model(pixel_values=px).logits.float().argmax(-1)
    b256 = [{"pixel_values": px, "labels": labels}]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rb, rc, rt = O.s2_candidate_scores(model, b256, str(dev), None, autocast=True)
    torch.cuda.synchronize()
    t_ref = time.perf_counter() - t0
    cx.api.attention_removal_counts(ours_model, b256, dev, None)                  # builds the cached engine, captures the chain
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ob, oc, ot = cx.api.attention_removal_counts(ours_model, b256, dev, None)
    torch.cuda.synchronize()
    t_ours = time.perf_counter() - t0
    out["stage2_256_images"] = {"reference_style_seconds": t_ref, "this_repo_seconds": t_ours, "speedup": t_ref / t_ours,
                                "reference_counts": [rb] + list(rc), "this_repo_counts": [ob] + list(oc),
                                "what": "reference: baseline + 12 x (deepcopy, bypass, full evaluation); here: cached-prefix suffix recompute in one captured chain"}
    del model
    torch.cuda.empty_cache()
    return out


def other_config(cx: Ctx, name: str, n_img: int, sparsity: float, steps: int, with_sweep: bool, both_s2_modes: bool):
    """One of the other BASELINE configs as a sub-object: Stage-1 sweep + fc1 roofline (optional) and the prune seconds."""
    from oracle import synth
    dev = cx.dev
    model = synth.make_vit(name, seed=0).to(dev)
    gen = torch.Generator(device=dev).manual_seed(1234)
    px_dev = torch.randn(n_img, 3, 224, 224, generator=gen, device=dev, dtype=torch.float32)
    px_host = torch.empty(px_dev.shape, dtype=torch.float32).pin_memory()
    px_host.copy_(px_dev)
    out = {"model": MODEL_NAMES[name], "images": n_img, "sparsity": sparsity}
    if with_sweep:
        m = measure_sweep(cx, name, model, px_dev, px_host, 256, steps, 3, profile=True, weak=False)
        out.update(value=m["value"], unit="images/s", ms_per_step=m["ms_per_step"], e2e_value=m["e2e"]["value"], step_tflops=m["step_tflops"],
                   roofline=m.get("roofline"), batch=m["batch"])
    del px_dev
    cx.api.release_engine(model)
    p = end_to_end_prune(cx, model, px_host, 256, sparsity, inference=(cx.world == 1))
    out.update(prune_seconds=p["seconds"], prune=p)
    if both_s2_modes and cx.world > 1 and p["stage2_sharding"] != "candidates":
        pc = end_to_end_prune(cx, model, px_host, 256, sparsity, shard_mode="candidates", inference=False)
        out["prune_seconds_candidate_sharded"] = pc["seconds"]
    del model, px_host
    cx.api.trim_pool()
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    from oracle import synth                      # synthetic model/data generators only (measurement infrastructure)
    cx = Ctx()
    api, dev, rank, world = cx.api, cx.dev, cx.rank, cx.world
    n_img, bs = args.images, args.batch
    model = synth.make_vit(args.model, seed=0).to(dev)
    gen = torch.Generator(device=dev).manual_seed(1234)   # every rank generates the same set and sweeps its share of it
    px_dev = torch.randn(n_img, 3, 224, 224, generator=gen, device=dev, dtype=torch.float32)
    px_host = torch.empty(px_dev.shape, dtype=torch.float32).pin_memory()
    px_host.copy_(px_dev)

    sampler = ClockSampler(cx.local) if rank == 0 and not args.no_clocks else None
    main = measure_sweep(cx, args.model, model, px_dev, px_host, bs, args.steps, args.warmup, profile=True, weak=not args.no_extra,
                         outputs=rank == 0 and bool(args.dump_outputs))
    clocks = sampler.stop() if sampler is not None else None
    if rank == 0 and args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in main.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)

    peaks = measured_peaks()
    # everything below is secondary to the line's headline numbers: a failure there is reported inside the line, not instead of it
    if rank == 0:
        try:
            main["hbm_kernels"]["ffn_gather_batch"] = gather_bandwidth(cx, model, args.model, args.sparsity, main["hbm_kernels"]["peak_gbs"])
        except Exception as exc:
            main["hbm_kernels"]["ffn_gather_batch"] = {"error": repr(exc)}

    extra = {}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        try:
            cpu_model = synth.make_vit(args.model, seed=0)
            probe, _ = cpu_s1_rate(cpu_model, 8, 8, threads)
            n_cpu = int(max(8, min(512, probe * args.cpu_seconds)))
            n_cpu = n_cpu - n_cpu % bs if n_cpu >= bs else n_cpu - n_cpu % 8
            bs_cpu = cpu_batch(n_cpu, bs)
            rate, dt = cpu_s1_rate(cpu_model, n_cpu, bs_cpu, threads)
            extra["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                                     "sample": f"{n_cpu} images in batches of {bs_cpu} ({dt:.1f} s), oracle port of the reference sweep, CPU autocast bf16"}
            del cpu_model
        except Exception as exc:
            extra["cpu_baseline"] = {"value": None, "unit": "images/s", "cores": threads, "kind": "port", "sample": f"failed: {exc!r}"}
    if world == 1 and not args.no_extra:
        try:
            extra["torch_cuda_baseline"] = torch_cuda_baseline(cx, args.model, px_dev, bs, main["value"], model)
        except Exception as exc:
            extra["torch_cuda_baseline"] = {"error": repr(exc)}

    prune = None
    if not args.no_prune:
        try:
            api.release_engine(model)
            prune = end_to_end_prune(cx, model, px_host, bs, args.sparsity)
        except Exception as exc:
            prune = {"seconds": None, "error": repr(exc)}

    configs = {}
    if not args.no_extra and not args.no_prune and args.model == "base" and "error" not in prune:
        del px_dev
        api.release_engine(model)
        torch.cuda.empty_cache()
        try:
            if world == 1:
                configs["vit_s16_512_37.5pct"] = other_config(cx, "small", 512, 0.375, args.steps, with_sweep=True, both_s2_modes=False)
                sweep = []
                for sp in (0.25, 0.375, 0.5):          # BASELINE configs[4]: sparsity_rate=-2
                    p = end_to_end_prune(cx, model, px_host, bs, sp) if sp != args.sparsity else prune
                    sweep.append({"sparsity": sp, "K": p["K"], "t": p["t"], "prune_seconds": p["seconds"], "achieved_sparsity": p["achieved_sparsity"],
                                  "inference": p.get("inference")})
                configs["vit_b16_sparsity_sweep"] = sweep
            configs["vit_l16_2048_50pct"] = other_config(cx, "large", 2048, 0.5, max(2, args.steps // 4), with_sweep=(world == 1), both_s2_modes=True)
        except Exception as exc:
            configs["error"] = repr(exc)

    if rank == 0:
        cfg = bench_config(args, world)
        line = {
            "metric": "calibration_images_per_s", "value": main["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg,
            "e2e": main["e2e"], "gpu_launches": main["launches"], "clocks": clocks, "roofline": main.get("roofline"),
            "step_tflops": main["step_tflops"], "kernels": main.get("kernels"), "ms_per_step_instrumented": main.get("ms_per_step_instrumented"),
            "hbm_kernels": main.get("hbm_kernels"), "weak": main.get("weak"),
            "prune_e2e_seconds": prune["seconds"] if prune else None, "prune_e2e": prune, "configs": configs or None,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
