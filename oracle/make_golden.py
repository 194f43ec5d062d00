"""Generates tests/golden/*.npz|json by running the UNMODIFIED reference (zvezdvv/2ssp-X-vit, mounted at
/root/reference in the build container) on seeded synthetic inputs. TEST INFRASTRUCTURE.

    python oracle/make_golden.py            # needs /root/reference; the GPU box only uses the committed fixtures

What is recorded (all produced by reference functions, none by this repository's code):
  * src/vit_pruning.py:_compute_ffn_activation_importance  -- Stage-1 scores, in the two oracle modes of
    SURVEY.md section 8c: "fp32" (torch.autocast patched to disabled, harness side) and "asis" (CPU autocast = bf16);
  * src/vit_pruning.py:prune_vit_mlp_width(precomputed_importance=fp32 scores) -- masks, indices, gathered weights;
  * src/vit_pruning.py:evaluate_top1 / prune_vit_attention_blocks and
    pruning_srp-main/mask_conjunction.py:Auto2SSPInterface.fit() -- Stage-2 impacts, selection, accuracies;
  * src/vit_pruning.py:plan_2ssp_allocation -- (K, t) for ViT-S/B/L at 25 / 37.5 / 50 % and for the tiny model.

Harness-side shim (reference source untouched): transformers >= 5 `ViTLayer.forward` adds the attention
module's output directly, while the reference's HFAttentionBypass returns a tuple (src/vit_pruning.py:419-423);
the shim restores the 4.x behaviour of taking element [0].
"""
from __future__ import annotations

import contextlib
import copy
import hashlib
import importlib.util
import io
import json
import os
import sys
from pathlib import Path
from unittest import mock

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ.get("TSSP_REFERENCE", "/root/reference"))
sys.path.insert(0, str(ROOT))
from oracle import synth  # noqa: E402

GOLDEN = ROOT / "tests" / "golden"


def load_reference():
    if not (REF / "src" / "vit_pruning.py").exists():
        raise SystemExit(f"{REF} not found: golden vectors can only be regenerated where the reference is mounted")
    sys.path.insert(0, str(REF))
    import src.vit_pruning as vp  # the reference module, unmodified
    spec = importlib.util.spec_from_file_location("ref_mask_conjunction", REF / "pruning_srp-main" / "mask_conjunction.py")
    mc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mc)
    return vp, mc


def install_tuple_shim():
    from transformers.models.vit import modeling_vit as mv

    def forward(self, hidden_states, **kwargs):
        attn = self.attention(self.layernorm_before(hidden_states), **kwargs)
        if isinstance(attn, (tuple, list)):
            attn = attn[0]
        hidden_states = attn + hidden_states
        out = self.intermediate(self.layernorm_after(hidden_states))
        return self.output(out, hidden_states)

    mv.ViTLayer.forward = forward


@contextlib.contextmanager
def autocast_disabled():
    """O-fp32 oracle mode: every torch.autocast(...) the reference opens becomes a no-op."""
    real = torch.autocast

    class Off(real):
        def __init__(self, device_type, *a, **k):
            k["enabled"] = False
            super().__init__(device_type, *a, **k)

    with mock.patch.object(torch, "autocast", Off):
        yield


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        return fn(*a, **k)


def pack_bits(mask_lists):
    return np.packbits(np.asarray(mask_lists, dtype=np.uint8), axis=-1)


WEIGHT_SAMPLE = 512


def weight_fixture(state):
    """The seeded init in a file well under 1 MB: per tensor its shape, the SHA-256 of its bytes and a fixed sample of
    its entries (all of them for tensors of at most WEIGHT_SAMPLE entries) at the stored flat positions."""
    out = {}
    rng = np.random.default_rng(0)
    for k, v in state.items():
        v = np.ascontiguousarray(v, dtype=np.float32)
        idx = np.arange(v.size) if v.size <= WEIGHT_SAMPLE else np.sort(rng.choice(v.size, WEIGHT_SAMPLE, replace=False))
        out[k] = v.reshape(-1)[idx]
        out[f"{k}:index"] = idx.astype(np.int64)
        out[f"{k}:shape"] = np.asarray(v.shape, dtype=np.int64)
        out[f"{k}:sha256"] = np.array(hashlib.sha256(v.tobytes()).hexdigest())
    return out


def golden_for(vp, mc, name: str, n_img: int, batch: int, t_prune: int, store_weights: bool, s2: bool):
    model = synth.make_vit(name, seed=0)
    image = synth.SHAPES[name][0]
    pixels = synth.make_pixels(n_img, image, seed=1234)
    with autocast_disabled():
        labels = synth.self_labels(model, pixels, batch)
    batches = synth.make_batches(pixels, labels, batch)
    out = {}
    meta = {"model": name, "n_img": n_img, "batch": batch, "t_prune": t_prune, "state_sha": synth.state_sha(model),
            "pixels_sha": synth.sha256_tensors([pixels]), "torch": torch.__version__}
    import transformers
    meta["transformers"] = transformers.__version__
    meta["cpu_threads"] = torch.get_num_threads()   # oneDNN's bf16 GEMMs split work by thread count: the as-is bits follow

    with autocast_disabled():
        s_fp32 = quiet(vp._compute_ffn_activation_importance, model, batches, device="cpu", batch_limit=None)
        logits = torch.cat([model(pixel_values=b["pixel_values"]).logits for b in batches]).detach()
    s_asis = quiet(vp._compute_ffn_activation_importance, model, batches, device="cpu", batch_limit=None)
    out["scores_fp32"] = torch.stack(s_fp32).numpy()
    out["scores_asis"] = torch.stack([s.float() for s in s_asis]).numpy()
    out["scores_asis_dtype"] = np.array(str(s_asis[0].dtype))
    out["logits_fp32"] = logits.numpy()
    out["labels"] = labels.numpy()

    # Stage-1 select + gather on the fp32 scores (the auto_2ssp.py flow: precomputed_importance=fp32 scores)
    pruned = copy.deepcopy(model)
    nb = len(s_fp32)
    res = quiet(vp.prune_vit_mlp_width, pruned, n_to_prune_per_block=[t_prune] * nb, strategy="act_l2",
                precomputed_importance=[s.float() for s in s_fp32], collect_masks=True, min_remaining=8)
    out["masks_bits"] = pack_bits(res["ffn_prune_masks"])
    out["mask_width"] = np.array(len(res["ffn_prune_masks"][0]))
    pairs = vp._gather_mlp_pairs(pruned)
    meta["gathered_sha"] = synth.sha256_tensors([t for fc1, fc2 in pairs for t in (fc1.weight, fc1.bias, fc2.weight)])
    meta["pruned_widths"] = [int(fc1.weight.shape[0]) for fc1, _ in pairs]
    # with massively tied scores (apply_mask_prune.py flow: +/-1 importances)
    tied = copy.deepcopy(model)
    g = torch.Generator().manual_seed(7)
    width = s_fp32[0].numel()
    pm = [(torch.rand(width, generator=g) < 0.3) for _ in range(nb)]
    imp_tied = [torch.where(m, torch.tensor(-1.0), torch.tensor(1.0)) for m in pm]
    res_t = quiet(vp.prune_vit_mlp_width, tied, n_to_prune_per_block=[int(m.sum()) for m in pm], strategy="act_l2",
                  precomputed_importance=imp_tied, collect_masks=True, min_remaining=8)
    same = all(torch.equal(torch.tensor(a, dtype=torch.bool), m) for a, m in zip(res_t["ffn_prune_masks"], pm))
    meta["tied_masks_reproduce_input"] = bool(same)

    if s2:
        with autocast_disabled():
            iface = mc.Auto2SSPInterface(copy.deepcopy(model), batches, device="cpu", importance_mode="copy", batch_limit=None)
            att_imp, mlp_imp = quiet(iface.fit)
            base_acc = quiet(vp.evaluate_top1, model, batches, "cpu")
            sel = quiet(vp.prune_vit_attention_blocks, copy.deepcopy(model), 0.0, dataloader=batches, device="cpu",
                        batch_limit=None, importance_mode="copy", show_progress=False, num_to_prune=max(1, nb // 3))
        out["att_importance_fp32"] = att_imp.numpy()
        out["iface_mlp_importance_fp32"] = torch.stack(mlp_imp).numpy()
        meta["s2"] = {"baseline_acc": float(base_acc), "pruned_indices": sel["pruned_indices"],
                      "original_metrics": sel["original_metrics"], "final_metrics": sel["final_metrics"],
                      "num_to_prune": max(1, nb // 3)}
    if store_weights:
        sd = model.state_dict()
        np.savez_compressed(GOLDEN / f"{name}_weights.npz", **weight_fixture({k: v.numpy() for k, v in sd.items()}))
    np.savez_compressed(GOLDEN / f"{name}_ref.npz", **out)
    return meta


def planner_golden(vp):
    rows = []
    for name in ("tiny", "small", "base", "large"):
        model = synth.make_vit(name, seed=0)
        for target in (0.25, 0.375, 0.5, 0.1, 0.02):
            for mr in (256, 512) if name != "tiny" else (8, 64):
                p = quiet(vp.plan_2ssp_allocation, model, target, min_remaining=mr)
                rows.append({"model": name, "target": target, "min_remaining": mr, "K": p.blocks_to_prune,
                             "t": p.per_block_neurons_to_prune, "removed": p.estimated_total_removed_params,
                             "err": p.est_error_params})
        p = quiet(vp.plan_2ssp_allocation, model, 0.3, min_remaining=8, forced_blocks=1)
        rows.append({"model": name, "target": 0.3, "min_remaining": 8, "forced_blocks": 1, "K": p.blocks_to_prune,
                     "t": p.per_block_neurons_to_prune, "removed": p.estimated_total_removed_params, "err": p.est_error_params})
        del model
    return rows


def main():
    GOLDEN.mkdir(parents=True, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    vp, mc = load_reference()
    install_tuple_shim()
    meta = {"tiny": golden_for(vp, mc, "tiny", n_img=12, batch=4, t_prune=96, store_weights=True, s2=True),
            "base": golden_for(vp, mc, "base", n_img=8, batch=4, t_prune=1120, store_weights=False, s2=True),
            "planner": planner_golden(vp)}
    with open(GOLDEN / "meta.json", "w") as f:
        json.dump(meta, f, indent=1)
    print("wrote", sorted(p.name for p in GOLDEN.iterdir()))


if __name__ == "__main__":
    main()
