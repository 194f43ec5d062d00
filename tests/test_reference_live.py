"""Differential tests against the UNMODIFIED reference, for the parts of the path that are pure host logic
(planner, parameter accounting, selection + masks given scores). They widen the pinned golden rows of tests/golden/ to a
few hundred random configurations. The reference is not part of this repository: the comparisons with it run when
TSSP_REFERENCE names a checkout of it (zvezdvv/2ssp-X-vit) and skip otherwise. The planner and the parameter accounting
are also compared, on the same random configurations and on every run, with the oracle (oracle/twossp_oracle.py), which
the golden rows pin to the reference."""
import contextlib
import io
import os
import random
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ["TSSP_REFERENCE"]) if os.environ.get("TSSP_REFERENCE") else None
needs_reference = pytest.mark.skipif(REF is None or not (REF / "src" / "vit_pruning.py").exists(),
                                     reason="TSSP_REFERENCE does not name a checkout of the reference")


@pytest.fixture(scope="module")
def ref_vp():
    sys.path.insert(0, str(REF))
    try:
        import src.vit_pruning as vp  # the reference module, unmodified
    finally:
        sys.path.remove(str(REF))
    return vp


def _tiny_vit(hidden, layers, heads, ffn, seed):
    from transformers import ViTConfig, ViTForImageClassification
    torch.manual_seed(seed)
    cfg = ViTConfig(image_size=16, patch_size=8, hidden_size=hidden, num_hidden_layers=layers, num_attention_heads=heads,
                    intermediate_size=ffn, num_labels=7)
    return ViTForImageClassification(cfg).eval()


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _planner_cases():
    """12 random tiny ViTs (heads, widths, depths, odd FFN widths), 25 random (target, min_remaining, forced_blocks) each:
    yields (model, None) once per model, then (model, (target, min_remaining, forced_blocks)) per plan."""
    rng = random.Random(20261018)
    for m in range(12):
        heads = rng.choice([1, 2, 4])
        hidden = heads * rng.choice([8, 16, 32])
        layers = rng.randint(2, 9)
        ffn = rng.choice([hidden, 2 * hidden, 4 * hidden, 4 * hidden + 8, 3 * hidden - 8])
        model = _tiny_vit(hidden, layers, heads, ffn, seed=m)
        yield model, None
        for _ in range(25):
            target = rng.choice([0.02, 0.1, 0.25, 0.375, 0.5, 0.6, 0.75, rng.uniform(0.01, 0.9)])
            mr = rng.choice([1, 8, ffn // 4, ffn // 2, ffn, 2 * ffn])
            forced = rng.choice([None, None, None, 0, 1, layers - 1])
            yield model, (target, mr, forced)


def _plan_key(p):
    return (p.target_sparsity, p.num_blocks_total, p.blocks_to_prune, p.per_block_neurons_to_prune, p.stage2_fraction,
            p.estimated_total_removed_params, p.est_error_params)


def test_planner_and_accounting_match_the_oracle_on_random_shapes():
    from oracle import twossp_oracle as O
    from twossp_b200 import api
    n_cases = 0
    for model, case in _planner_cases():
        if case is None:
            blocks = O.blocks_of(model)[1]
            pairs = O.mlp_pairs(model)
            assert api.count_total_params(model) == O._numel(model)
            assert api.count_block_params(model) == [O._numel(b) for b in blocks]
            assert api._count_attention_params_per_block(model) == [O._numel(b.attention) for b in blocks]
            assert api._count_ffn_params_per_block(model) == [O._numel(a) + O._numel(c) for a, c in pairs]
            continue
        target, mr, forced = case
        ours = _quiet(api.plan_2ssp_allocation, model, target, min_remaining=mr, forced_blocks=forced)
        oracle = O.plan(model, target, min_remaining=mr, forced_blocks=forced)
        assert _plan_key(ours) == _plan_key(oracle), (case, _plan_key(ours), _plan_key(oracle))
        n_cases += 1
    assert n_cases == 300


@needs_reference
def test_planner_and_accounting_match_the_reference_on_random_shapes(ref_vp):
    from twossp_b200 import api
    n_cases = 0
    for model, case in _planner_cases():
        if case is None:
            assert api.count_total_params(model) == ref_vp.count_total_params(model)
            assert api.count_block_params(model) == ref_vp.count_block_params(model)
            assert api._count_attention_params_per_block(model) == ref_vp._count_attention_params_per_block(model)
            assert api._count_ffn_params_per_block(model) == ref_vp._count_ffn_params_per_block(model)
            continue
        target, mr, forced = case
        ours = _quiet(api.plan_2ssp_allocation, model, target, min_remaining=mr, forced_blocks=forced)
        theirs = _quiet(ref_vp.plan_2ssp_allocation, model, target, min_remaining=mr, forced_blocks=forced)
        assert _plan_key(ours) == _plan_key(theirs), (case, _plan_key(ours), _plan_key(theirs))
        n_cases += 1
    assert n_cases == 300


@needs_reference
def test_selection_and_masks_given_scores_match_the_reference_on_cpu_tensors(ref_vp):
    # the selection arithmetic of prune_vit_mlp_width (n_prune truncation, min_remaining clamp, argsort / sort, mask layout,
    # skipped blocks) restated by the oracle, against the reference itself, on random widths and score vectors with ties
    from oracle import twossp_oracle as O
    import copy
    rng = random.Random(7)
    for m in range(6):
        heads = rng.choice([1, 2])
        hidden = heads * 16
        layers = rng.randint(2, 5)
        ffn = rng.choice([32, 40, 64, 72])
        model = _tiny_vit(hidden, layers, heads, ffn, seed=100 + m)
        g = torch.Generator().manual_seed(m)
        scores = [torch.randint(0, 9, (ffn,), generator=g).float() + torch.rand(ffn, generator=g) * (m % 2) for _ in range(layers)]
        n_prune = [rng.choice([0, 1, ffn // 3, ffn - 8, ffn]) for _ in range(layers)]
        mr = rng.choice([1, 8, ffn // 2])
        ref = _quiet(ref_vp.prune_vit_mlp_width, copy.deepcopy(model), n_to_prune_per_block=n_prune, strategy="act_l2",
                     precomputed_importance=[s.clone() for s in scores], collect_masks=True, min_remaining=mr, device="cpu")
        ours = _quiet(O.s1_prune, copy.deepcopy(model), n_to_prune_per_block=n_prune, importance=[s.clone() for s in scores], min_remaining=mr)
        assert ours["ffn_prune_masks"] == ref["ffn_prune_masks"] and ours["ffn_pruned_indices"] == ref["ffn_pruned_indices"]
        for (a1, a2), (b1, b2) in zip(O.mlp_pairs(ours["model"]), ref_vp._gather_mlp_pairs(ref["model"])):
            assert torch.equal(a1.weight, b1.weight) and torch.equal(a1.bias, b1.bias) and torch.equal(a2.weight, b2.weight)
            assert a1.out_features == b1.out_features and a2.in_features == b2.in_features


def _load_script(name, file):
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, REF / "manual-experiments" / file)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@needs_reference
@pytest.mark.skipif(REF is None or not (REF / "manual-experiments" / "consensus_mask.py").exists(),
                    reason="TSSP_REFERENCE does not name a checkout of the reference with its manual-experiments scripts")
def test_mask_builder_oracle_matches_the_reference_scripts_on_random_inputs():
    # consensus (growing-t intersection), summation masks and min-max normalisation: the oracle restatement against the
    # unmodified scripts on 40 random configurations (files, ragged widths, heavy ties, every rounding mode, tiny fractions)
    import re
    from oracle import mask_builders_oracle as MO
    cons = _load_script("ref_consensus_mask_live", "consensus_mask.py")
    summ = _load_script("ref_summation_live", "aggregate_and_mask-summation.py")
    norm = _load_script("ref_normalize_live", "normalize_scores.py")
    rng = random.Random(99)
    for case in range(40):
        n_files = rng.randint(1, 4)
        widths = [rng.choice([7, 16, 33, 64, 100]) + rng.randint(0, 5) for _ in range(rng.randint(1, 5))]
        quant = rng.choice([0, 0, 4, 16])
        frac = rng.choice([0.0, 0.004, 0.1, 0.25, 0.35, 0.5, 0.9, rng.random()])
        rounding = rng.choice(["round", "floor", "ceil"])
        leaves = [MO.make_leaf(1000 * case + f, widths, quant) for f in range(n_files)]
        if n_files > 1 and case % 3 == 0:   # an anti-correlated file forces the selection fraction t to grow
            leaves[1] = {k: 1.0 - v for k, v in leaves[0].items()}
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            ref_mask = cons.consensus_for_path(leaves, frac, rounding, verbose=True)
        ours, info = MO.consensus(leaves, frac, rounding)
        assert ours == ref_mask and list(ours) == list(ref_mask), (case, n_files, widths, quant, frac, rounding)
        m = re.search(r"t_final=([0-9.]+), min_intersection=(\d+), K_common=(\d+), iters=(\d+)", buf.getvalue())
        if m and info:
            assert (int(m.group(2)), int(m.group(3)), int(m.group(4))) == (info["min_intersection"], info["K_common"], info["iters"])
        sums = MO.aggregate(leaves)
        ref_sums = {}
        for leaf in leaves:
            for k, v in leaf.items():
                ref_sums[k] = ref_sums.get(k, 0.0) + float(v)
        assert sums == ref_sums
        with contextlib.redirect_stdout(io.StringIO()):
            assert MO.summation_mask(sums, frac, rounding) == summ.make_mask_for_leaf(ref_sums, frac, rounding)
            k = rng.randint(0, max(widths) + 3)
            assert MO.summation_mask(sums, 0.0, rounding, per_block_k=k) == summ.make_mask_for_leaf(ref_sums, 0.0, rounding, per_block_k=k)
        tree = {"ffn": leaves[0], "meta": {"alpha": rng.random() * 10 - 5, "flag": True, "name": "x", "list": [3, -2.5, {"z": 7}]}}
        lo, hi = norm.scan_min_max_raw(tree)
        assert MO.normalize(tree) == norm.normalize_structure(tree, lo, hi)


@pytest.fixture(scope="module")
def ref_iface():
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_mask_conjunction_live", REF / "pruning_srp-main" / "mask_conjunction.py")
    mc = importlib.util.module_from_spec(spec)
    sys.path.insert(0, str(REF))
    try:
        spec.loader.exec_module(mc)
    finally:
        sys.path.remove(str(REF))
    return mc


@pytest.fixture()
def hf_tuple_shim():
    """transformers >= 5 ViTLayer.forward adds the attention output directly, the reference bypass returns a tuple
    (src/vit_pruning.py:419-423): restore the 4.x behaviour for the duration of a test (harness-side, reference untouched)."""
    from transformers.models.vit import modeling_vit as mv
    saved = mv.ViTLayer.forward

    def forward(self, hidden_states, **kwargs):
        attn = self.attention(self.layernorm_before(hidden_states), **kwargs)
        if isinstance(attn, (tuple, list)):
            attn = attn[0]
        hidden_states = attn + hidden_states
        return self.output(self.intermediate(self.layernorm_after(hidden_states)), hidden_states)

    mv.ViTLayer.forward = forward
    yield
    mv.ViTLayer.forward = saved


@needs_reference
@pytest.mark.parametrize("autocast", [True, False])
def test_stage1_and_stage2_oracle_match_the_reference_live(ref_vp, ref_iface, hf_tuple_shim, autocast):
    # random tiny ViTs and inputs beyond the committed fixtures: Stage-1 scores bit for bit (as-is = CPU autocast bf16, and
    # fp32 with autocast disabled), Stage-2 impacts, the selected blocks and the final metric of prune_vit_attention_blocks
    import copy
    from unittest import mock
    from oracle import synth
    from oracle import twossp_oracle as O

    class Off(torch.autocast):
        def __init__(self, device_type, *a, **k):
            k["enabled"] = False
            super().__init__(device_type, *a, **k)

    ctx = contextlib.nullcontext() if autocast else mock.patch.object(torch, "autocast", Off)
    rng = random.Random(5 + int(autocast))
    for m in range(3):
        heads = rng.choice([1, 2])
        layers = rng.randint(2, 4)
        model = _tiny_vit(heads * 16, layers, heads, rng.choice([48, 64]), seed=200 + m)
        with torch.no_grad():   # non-trivial biases / LayerNorm affines, as in oracle/synth.py
            for p in model.parameters():
                if p.dim() == 1:
                    p.add_(torch.randn(p.shape, generator=torch.Generator().manual_seed(m)) * 0.05)
        px = synth.make_pixels(10, 16, seed=300 + m)
        labels = synth.self_labels(model, px, 4)
        batches = synth.make_batches(px, labels, 4)
        limit = rng.choice([None, 2])
        with ctx:
            ref_s = _quiet(ref_vp._compute_ffn_activation_importance, model, batches, device="cpu", batch_limit=limit)
            iface = ref_iface.Auto2SSPInterface(copy.deepcopy(model), batches, device="cpu", importance_mode="copy", batch_limit=limit)
            ref_att, ref_mlp = _quiet(iface.fit)
            ref_sel = _quiet(ref_vp.prune_vit_attention_blocks, copy.deepcopy(model), 0.0, dataloader=batches, device="cpu",
                             batch_limit=limit if limit is not None else 10 ** 9, importance_mode="copy", show_progress=False, num_to_prune=1)
        ours_s = O.s1_scores(model, batches, "cpu", limit, autocast=autocast)
        assert all(a.dtype == b.dtype and torch.equal(a, b) for a, b in zip(ours_s, ref_s))
        assert all(torch.equal(a.float(), b.float()) for a, b in zip(ours_s, ref_mlp))
        base, cand, seen = O.s2_candidate_scores(model, batches, "cpu", limit, autocast=autocast)
        assert torch.equal(torch.tensor(O.s2_impacts(base, cand, seen), dtype=torch.float32), ref_att)
        ours_sel = O.s2_prune(copy.deepcopy(model), 0.0, batches, "cpu", limit if limit is not None else 10 ** 9, "copy", num_to_prune=1, autocast=autocast)
        assert ours_sel["pruned_indices"] == ref_sel["pruned_indices"]
        assert ours_sel["original_metrics"] == ref_sel["original_metrics"] and ours_sel["final_metrics"] == ref_sel["final_metrics"]


@needs_reference
def test_api_surface_mirrors_the_reference(ref_vp):
    """Every function of the path that the reference exports has a counterpart with the same parameter names in the same
    order (extra keyword-only / trailing parameters allowed), and the plugin class has the same constructor and methods.
    The checkpoint / report file I/O of the fine-tuning flow is deliberately not mirrored (DESIGN.md section 8)."""
    import importlib.util
    import inspect

    from twossp_b200 import api
    not_mirrored = {"save_cifar_adapter", "load_cifar_adapter", "save_report"}
    names = [n for n in ref_vp.__all__ if n not in not_mirrored]
    names += ["_compute_ffn_activation_importance", "_count_attention_params_per_block", "_count_ffn_params_per_block",
              "_get_hidden_and_inter_sizes"]
    assert set(ref_vp.__all__) - not_mirrored <= set(api.__all__)
    for name in names:
        ref_params = list(inspect.signature(getattr(ref_vp, name)).parameters.values())
        our_params = list(inspect.signature(getattr(api, name)).parameters.values())
        assert [p.name for p in our_params[:len(ref_params)]] == [p.name for p in ref_params], name
        for rp, op in zip(ref_params, our_params):
            assert rp.default == op.default or (rp.default is inspect.Parameter.empty) == (op.default is inspect.Parameter.empty), (name, rp.name)
        assert all(p.default is not inspect.Parameter.empty or p.kind is p.KEYWORD_ONLY for p in our_params[len(ref_params):]), name

    spec = importlib.util.spec_from_file_location("ref_mask_conjunction_live", REF / "pruning_srp-main" / "mask_conjunction.py")
    mc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mc)
    ref_cls, our_cls = mc.Auto2SSPInterface, api.B200Auto2SSPInterface
    ref_init = list(inspect.signature(ref_cls.__init__).parameters.values())
    our_init = list(inspect.signature(our_cls.__init__).parameters.values())
    assert [(p.name, p.default) for p in our_init[:len(ref_init)]] == [(p.name, p.default) for p in ref_init]
    assert all(p.default is not inspect.Parameter.empty for p in our_init[len(ref_init):])
    ref_methods = {m for m in vars(ref_cls) if not m.startswith("__")}
    assert ref_methods <= {m for m in vars(our_cls) if not m.startswith("__")}
    assert {t.name for t in mc.PruningTypes} == {t.name for t in api.PruningTypes}
