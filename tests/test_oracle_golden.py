"""The oracle (oracle/twossp_oracle.py) against the golden vectors recorded from the UNMODIFIED reference by
oracle/make_golden.py. CPU only. Integer/index results must be identical; float results are produced by the same
torch ops in the same order, so they are compared bit-for-bit too."""
import contextlib
import copy
import hashlib

import numpy as np
import pytest
import torch

from oracle import synth
from oracle import twossp_oracle as O


def _load(golden_dir, name):
    return np.load(f"{golden_dir}/{name}_ref.npz")


def _setup(name, meta):
    m = meta[name]
    model = synth.make_vit(name, seed=0)
    assert synth.state_sha(model) == m["state_sha"], "seeded init drifted from the fixture"
    pixels = synth.make_pixels(m["n_img"], synth.SHAPES[name][0], seed=1234)
    assert synth.sha256_tensors([pixels]) == m["pixels_sha"]
    return model, pixels, m


def _unpack(bits, width):
    return np.unpackbits(bits, axis=-1)[..., :width]


@contextlib.contextmanager
def _cpu_threads(n):
    saved = torch.get_num_threads()
    torch.set_num_threads(n)
    try:
        yield
    finally:
        torch.set_num_threads(saved)


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_s1_scores_match_reference(name, golden_dir, golden_meta):
    model, pixels, m = _setup(name, golden_meta)
    g = _load(golden_dir, name)
    batches = synth.make_batches(pixels, None, m["batch"])
    # CPU autocast runs oneDNN's bf16 GEMMs, which split their work by the intra-op thread count: the recorded bits are
    # those of the recording's thread count, whatever the cores of the machine running the test
    with _cpu_threads(m["cpu_threads"]):
        fp32 = torch.stack(O.s1_scores(model, batches, "cpu", None, autocast=False)).numpy()
        asis = O.s1_scores(model, batches, "cpu", None, autocast=True)
    assert np.array_equal(fp32, g["scores_fp32"])
    assert str(asis[0].dtype) == str(g["scores_asis_dtype"])
    assert np.array_equal(torch.stack([s.float() for s in asis]).numpy(), g["scores_asis"])


def test_tiny_weights_fixture_matches_seeded_init(golden_dir, golden_meta):
    # the fixture holds, per tensor, its shape, the SHA-256 of all its bytes and a sample of its entries
    # (oracle/make_golden.py: weight_fixture)
    model, _, _ = _setup("tiny", golden_meta)
    w = np.load(f"{golden_dir}/tiny_weights.npz")
    sd = model.state_dict()
    keys = {f for f in w.files if ":" not in f}
    assert keys == set(sd.keys())
    for k in keys:
        v = np.ascontiguousarray(sd[k].numpy(), dtype=np.float32)
        assert list(v.shape) == w[f"{k}:shape"].tolist(), k
        assert np.array_equal(v.reshape(-1)[w[f"{k}:index"]], w[k]), k
        assert hashlib.sha256(v.tobytes()).hexdigest() == str(w[f"{k}:sha256"]), k


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_s1_select_and_gather_match_reference(name, golden_dir, golden_meta):
    model, pixels, m = _setup(name, golden_meta)
    g = _load(golden_dir, name)
    scores = [torch.from_numpy(s.copy()) for s in g["scores_fp32"]]
    res = O.s1_prune(copy.deepcopy(model), n_to_prune_per_block=[m["t_prune"]] * len(scores), strategy="act_l2",
                     importance=scores, min_remaining=8)
    want = _unpack(g["masks_bits"], int(g["mask_width"]))
    assert np.array_equal(np.asarray(res["ffn_prune_masks"], dtype=np.uint8), want)
    assert [int(np.sum(r)) for r in want] == [m["t_prune"]] * len(scores)
    for row, idx in zip(want, res["ffn_pruned_indices"]):
        assert np.array_equal(np.nonzero(row)[0], np.asarray(idx))
    pairs = O.mlp_pairs(res["model"])
    assert [int(a.weight.shape[0]) for a, _ in pairs] == m["pruned_widths"]
    assert synth.sha256_tensors([t for a, b in pairs for t in (a.weight, a.bias, b.weight)]) == m["gathered_sha"]


def test_s1_prune_edge_cases():
    model = synth.make_vit("tiny", seed=0)
    with pytest.raises(ValueError):
        O.s1_prune(copy.deepcopy(model), n_to_prune_per_block=[1, 2])
    with pytest.raises(ValueError):
        O.s1_prune(copy.deepcopy(model))
    with pytest.raises(AssertionError):
        O.s1_prune(copy.deepcopy(model), sparsity=1.0)
    # blocks with nothing to prune are skipped: no mask entry (src/vit_pruning.py:283-284)
    res = O.s1_prune(copy.deepcopy(model), n_to_prune_per_block=[0, 5, 0], min_remaining=8)
    assert len(res["ffn_prune_masks"]) == 1 and sum(res["ffn_prune_masks"][0]) == 5
    # min_remaining clamps
    res = O.s1_prune(copy.deepcopy(model), sparsity=0.9, min_remaining=200)
    assert all(a.weight.shape[0] == 200 for a, _ in O.mlp_pairs(res["model"]))


@pytest.mark.parametrize("name", ["tiny", "base"])
def test_s2_matches_reference(name, golden_dir, golden_meta):
    model, pixels, m = _setup(name, golden_meta)
    g = _load(golden_dir, name)
    labels = torch.from_numpy(g["labels"].copy())
    batches = synth.make_batches(pixels, labels, m["batch"])
    base, cand, seen = O.s2_candidate_scores(model, batches, "cpu", None, autocast=False)
    assert base / seen == m["s2"]["baseline_acc"]
    impacts = torch.tensor(O.s2_impacts(base, cand, seen), dtype=torch.float32).numpy()
    assert np.array_equal(impacts, g["att_importance_fp32"])
    res = O.s2_prune(copy.deepcopy(model), 0.0, batches, "cpu", None, "copy", num_to_prune=m["s2"]["num_to_prune"], autocast=False)
    assert res["pruned_indices"] == m["s2"]["pruned_indices"]
    assert res["original_metrics"] == m["s2"]["original_metrics"]
    assert res["final_metrics"] == m["s2"]["final_metrics"]


def test_interface_oracle_matches_reference(golden_dir, golden_meta):
    model, pixels, m = _setup("tiny", golden_meta)
    g = _load(golden_dir, "tiny")
    batches = synth.make_batches(pixels, torch.from_numpy(g["labels"].copy()), m["batch"])
    att, mlp = O.Auto2SSPOracle(model, batches, "cpu", "copy", None, autocast=False).fit()
    assert np.array_equal(att.numpy(), g["att_importance_fp32"])
    assert np.array_equal(torch.stack(mlp).numpy(), g["iface_mlp_importance_fp32"])


def test_functional_forward_agrees_with_reference_outputs(golden_dir, golden_meta):
    model, pixels, m = _setup("tiny", golden_meta)
    g = _load(golden_dir, "tiny")
    out = O.vit_forward(O.extract_weights(model), pixels)
    assert np.allclose(out["logits"].numpy(), g["logits_fp32"], rtol=1e-4, atol=1e-5)
    scores = torch.stack([n.sum(0) / pixels.shape[0] for n in out["norms"]]).numpy()
    assert np.allclose(scores, g["scores_fp32"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", ["tiny", "small", "base", "large"])
def test_planner_matches_reference(name, golden_meta):
    model = synth.make_vit(name, seed=0)
    rows = [r for r in golden_meta["planner"] if r["model"] == name]
    assert rows
    for r in rows:
        p = O.plan(model, r["target"], min_remaining=r["min_remaining"], forced_blocks=r.get("forced_blocks"))
        assert (p.blocks_to_prune, p.per_block_neurons_to_prune, p.estimated_total_removed_params, p.est_error_params) == \
            (r["K"], r["t"], r["removed"], r["err"]), r


def test_planner_pins_survey_table(golden_meta):
    # SURVEY.md section 8a: (K, t) at 25 / 37.5 / 50 % with min_remaining=512
    want = {"small": [(4, 341), (5, 576), (7, 746)], "base": [(4, 661), (5, 1120), (7, 1450)], "large": [(6, 1035), (8, 1638), (12, 2070)]}
    for name, kts in want.items():
        for target, kt in zip((0.25, 0.375, 0.5), kts):
            row = next(r for r in golden_meta["planner"] if r["model"] == name and r["target"] == target and r["min_remaining"] == 512 and "forced_blocks" not in r)
            assert (row["K"], row["t"]) == kt


# ----------------------------------------------------------------------------------------------- full-size fixtures
def _full(golden_dir, key):
    import json
    import os
    path = os.path.join(golden_dir, f"full_{key}.npz")
    meta_path = os.path.join(golden_dir, "full_meta.json")
    if not (os.path.exists(path) and os.path.exists(meta_path)):
        pytest.skip(f"no full-size fixture for {key}")
    with open(meta_path) as f:
        meta = json.load(f)
    if key not in meta:
        pytest.skip(f"no full-size fixture for {key}")
    return np.load(path), meta[key]


@pytest.mark.parametrize("key", ["small512", "base1024", "large2048"])
def test_full_size_masks_follow_from_the_recorded_scores(key, golden_dir):
    """oracle/make_golden_full.py fixtures (the unmodified reference at the benchmarked sizes): the oracle's selection
    rule applied to the recorded fp32 scores gives the recorded masks bit for bit, t ones per block; the recorded Stage-2
    impacts are whole image counts over the recorded number of images."""
    g, m = _full(golden_dir, key)
    want = _unpack(g["masks_bits"], int(g["mask_width"]))
    t = m["t_prune"]
    for b in range(want.shape[0]):
        scores = torch.from_numpy(g["scores_fp32"][b].copy())
        keep = O.s1_keep_indices(scores, t)
        mask = np.ones(scores.numel(), dtype=np.uint8)
        mask[keep.numpy()] = 0
        assert np.array_equal(mask, want[b]) and int(mask.sum()) == t
    counts = g["att_importance_fp32"].astype(np.float64) * m["s2_images"]
    assert np.allclose(counts, np.round(counts), atol=1e-6) and g["labels"].shape == (m["n_img"],)
    assert np.array_equal(g["logits_fp16"].astype(np.float32).argmax(-1)[g["label_margin"][:256] > 2e-3],
                          g["labels"][:256].astype(np.int64)[g["label_margin"][:256] > 2e-3])


@pytest.mark.parametrize("key", ["small512"])
def test_full_size_fixture_is_reproduced_by_the_oracle_forward(key, golden_dir):
    """The oracle's fp32 forward of the first images of the full-size set reproduces the recorded logits (stored as fp16)
    and labels: the fixture and the GPU box's synthetic model / images are the same objects."""
    g, m = _full(golden_dir, key)
    model = synth.make_vit(m["model"], seed=0)
    assert synth.state_sha(model) == m["state_sha"]
    pixels = synth.make_pixels(m["n_img"], 224, seed=1234)
    assert synth.sha256_tensors([pixels]) == m["pixels_sha"]
    out = O.vit_forward(O.extract_weights(model), pixels[:8])
    ref = g["logits_fp16"][:8].astype(np.float32)
    assert np.abs(out["logits"].numpy() - ref).max() <= 2e-3
    assert np.array_equal(out["logits"].argmax(-1).numpy(), g["labels"][:8].astype(np.int64))
