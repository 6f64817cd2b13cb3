"""
Differential tests: the host-side mirror (foldingdiff_b200.{beta_schedules,utils,datasets,sampling}) against what the
STOCK reference package computed on the same inputs (tests/golden/ref_host.npz, written by
tests/golden/make_golden_reference.py from the package installed in baseline/_ref; digests where the comparison is
bit for bit).
Rows a9 - a12 of SURVEY.md section 8: schedules, wrap, noise sampling, the dataset metadata loader, forward noising.
"""
import json

import numpy as np
import pytest
import torch

from conftest import load_golden
from foldingdiff_b200 import beta_schedules, datasets, utils
from oracle.replay import digest

# the inputs: make_golden_reference.py builds the reference's answers from these same definitions
WRAP_RANGES = [(-2.0, 2.0), (0.0, 1.0), (-np.pi, np.pi)]
NOISE_KWARGS = ({}, {"nonangular_variance": 2.0, "angular_variance": 0.5})
ITEMS = [(0, None), (3, 10), (4, 49), (1, 0)]
SAMPLE_T = 3
SAMPLE_KWARGS = (dict(n=2, sweep_lengths=(10, 14), batch_size=3), dict(n=1, sweep_lengths=(20, 23), batch_size=512))


def wrap_inputs():
    g = torch.Generator().manual_seed(0)
    return torch.cat([torch.randn(4096, generator=g) * 10, torch.tensor([0.0, -0.0, np.pi, -np.pi, 2 * np.pi, -2 * np.pi, 1e-30, 1e6, -1e6]),
                      torch.nextafter(torch.tensor([np.pi, -np.pi], dtype=torch.float32), torch.tensor([0.0, 0.0]))])


def write_dataset_dir(d):
    with open(f"{d}/training_args.json", "w") as f:
        json.dump({"angles_definitions": "canonical-full-angles", "max_seq_len": 128}, f)
    np.save(f"{d}/training_mean_offset.npy", np.linspace(-1, 1, 6))


def write_sample_dir(d):
    with open(f"{d}/training_args.json", "w") as f:
        json.dump({"angles_definitions": "canonical-full-angles", "max_seq_len": 128}, f)
    np.save(f"{d}/training_mean_offset.npy", np.array([-1.47, 0.75, 3.1, 1.94, 2.03, 2.12]))  # the shift crosses +-pi for omega


@pytest.fixture(scope="module")
def ref():
    return load_golden("ref_host.npz")


def assert_same(ours, theirs, what):
    """Bit-identical, same dtype and shape: `theirs` is the digest of the reference's array."""
    assert digest(ours) == str(theirs), what


@pytest.mark.parametrize("kind", ["linear", "cosine", "quadratic"])
@pytest.mark.parametrize("T", [2, 100, 250, 1000])
def test_schedules_and_alpha_tables_bit_identical(ref, kind, T):
    key = f"sched_{kind}_{T}"
    ours = beta_schedules.get_variance_schedule(kind, T)
    assert_same(ours, ref[f"{key}_betas"], "betas")
    a = beta_schedules.compute_alphas(ours)
    assert list(a) == ref[f"{key}_keys"].tolist()
    for k in a:
        assert_same(a[k], ref[f"{key}_{k}"], k)


def test_wrap_bit_identical_on_random_and_edge_values(ref):
    x = wrap_inputs()
    assert_same(utils.modulo_with_wrapped_range(x), ref["wrap_default"], "default range")
    for i, (lo, hi) in enumerate(WRAP_RANGES):
        assert_same(utils.modulo_with_wrapped_range(x, lo, hi), ref[f"wrap_range{i}"], (lo, hi))
    arr = x.numpy().astype(np.float64)
    assert_same(utils.modulo_with_wrapped_range(arr, -2, 2), ref["wrap_np64"], "float64 array")


def test_empty_dataset_and_noise_source_agree(ref, tmp_path):
    write_dataset_dir(str(tmp_path))
    ours = datasets.AnglesEmptyDataset.from_dir(str(tmp_path))
    assert ours.feature_names == json.loads(str(ref["dset_feature_names"]))
    assert ours.feature_is_angular == json.loads(str(ref["dset_feature_is_angular"]))
    assert ours.pad == int(ref["dset_pad"])
    assert_same(ours.get_masked_means(), ref["dset_masked_means"], "masked means")
    for i, kw in enumerate(NOISE_KWARGS):
        no = datasets.NoisedAnglesDataset(ours, timesteps=100, beta_schedule="cosine", **kw)
        assert list(no.alpha_beta_terms) == ref[f"dset{i}_terms_keys"].tolist()
        for k in no.alpha_beta_terms:
            assert_same(no.alpha_beta_terms[k], ref[f"dset{i}_terms_{k}"], k)
        torch.manual_seed(7344)
        assert_same(no.sample_noise(torch.zeros(7, 128, 6)), ref[f"dset{i}_noise"], ("noise", kw))


class _Inner:
    """Minimal inner dataset with the attributes NoisedAnglesDataset reads (both implementations)."""
    feature_names = {"angles": ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"]}
    feature_is_angular = {"angles": [True] * 6}
    pad = 32

    def __init__(self):
        g = torch.Generator().manual_seed(3)
        self.x = utils.modulo_with_wrapped_range(torch.randn(5, 32, 6, generator=g))

    def __len__(self):
        return 5

    def __getitem__(self, index, ignore_zero_center=False):
        mask = torch.zeros(32); mask[:20] = 1
        return {"angles": self.x[index].clone(), "attn_mask": mask, "position_ids": torch.arange(32)}


@pytest.mark.parametrize("schedule", ["linear", "cosine"])
def test_forward_noising_item_equals_the_reference_item(ref, schedule):
    no = datasets.NoisedAnglesDataset(_Inner(), timesteps=50, beta_schedule=schedule)
    for idx, tval in ITEMS:
        key = f"item_{schedule}_{idx}_{tval}"
        torch.manual_seed(100 + idx)
        a = no.__getitem__(idx, use_t_val=tval)
        assert set(a.keys()) == set(ref[key + "_keys"].tolist())
        for k in a:
            assert_same(torch.as_tensor(a[k]), ref[f"{key}_{k}"], (k, idx, tval))


def test_sample_orchestration_equals_stock_sample(ref, tmp_path, monkeypatch):
    """
    Row a1 (sampling.sample, sampling.py:135-224): length list, chunking, per-chunk noise draws, trimming, per-chain
    slicing, mean-offset shift + re-wrap.  The stored answer is the stock sample() around the stock p_sample_loop and
    the reference-assembled model (baseline/reference_arm.py).  Here the same loop arithmetic (the oracle's restatement,
    bit-identical to the stock loop: tests/test_oracle_golden.py) is handed the predictions that model made, in the
    same order, for the same inputs (oracle/replay.py), so any difference comes from the orchestration: must be
    bit-identical.
    """
    from foldingdiff_b200 import sampling as ours
    from oracle import loop as oloop
    from oracle.replay import Replay

    write_sample_dir(str(tmp_path))
    o_dset = datasets.NoisedAnglesDataset(datasets.AnglesEmptyDataset.from_dir(str(tmp_path)), timesteps=SAMPLE_T,
                                          beta_schedule="cosine")

    def restated_loop(model, lengths, noise, timesteps, betas, is_angle, disable_pbar=False, history="full"):
        return oloop.p_sample_loop(model, lengths, noise, timesteps, betas, is_angle)
    monkeypatch.setattr(ours, "p_sample_loop", restated_loop)
    for i, kw in enumerate(SAMPLE_KWARGS):
        model = Replay(ref, f"sample{i}")
        torch.manual_seed(77)
        a = ours.sample(model, o_dset, **kw)
        assert model.calls == model.total
        assert len(a) == int(ref[f"sample{i}_n"]) == kw["n"] * (kw["sweep_lengths"][1] - kw["sweep_lengths"][0])
        for j, x in enumerate(a):
            assert x.shape == (SAMPLE_T, x.shape[1], 6)
            assert_same(x, ref[f"sample{i}_out_{j}"], (i, j))
    with pytest.raises(ValueError):  # the stock sample() raises here too (asserted when the answers were stored)
        ours.sample(Replay(ref, "sample0"), o_dset, n=1, sweep_lengths=(30, 30))
