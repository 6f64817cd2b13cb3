"""
CPU side of the training-objective feature: AnglesTableDataset items, the batch layout _get_loss_terms consumes, the
BertForDiffusion constructor surface, bin/eval_loss.py's argument handling and the pdist restatement against the
reference's stored answers (tests/golden/ref_pdist.npz).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from torch.utils.data import default_collate

import loss_oracle
from conftest import GOLDEN, ROOT, load_golden, mini_state_dict
from foldingdiff_b200 import losses, modelling, utils, writers
from foldingdiff_b200.datasets import FEATURE_SET_NAMES_TO_FEATURE_NAMES, AnglesTableDataset, NoisedAnglesDataset

NAMES = FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"]


def _table(l, seed=0):
    return np.random.default_rng(seed).uniform(-np.pi, np.pi, size=(l, 6))


def test_item_centring_wrap_nan_and_pad():
    t = _table(30)
    t[4, 2] = np.nan
    off = np.array([0.5, -3.0, 2.0, 0.1, 0.0, -0.2])
    item = AnglesTableDataset([t], pad=40, mean_offset=off)[0]
    want = utils.modulo_with_wrapped_range(t - off, -np.pi, np.pi)
    want = np.nan_to_num(want, nan=0)
    assert item["angles"].shape == (40, 6) and item["angles"].dtype == torch.float32
    assert torch.equal(item["angles"][:30], torch.from_numpy(want).float())
    assert float(item["angles"][4, 2]) == 0.0  # NaN after centring -> 0
    assert torch.equal(item["angles"][30:], torch.zeros(10, 6))
    assert item["attn_mask"].tolist() == [1.0] * 30 + [0.0] * 10
    assert int(item["lengths"]) == 30 and torch.equal(item["position_ids"], torch.arange(40))
    raw = AnglesTableDataset([t], pad=40, mean_offset=off).__getitem__(0, ignore_zero_center=True)
    assert float(raw["angles"][0, 0]) == pytest.approx(t[0, 0], abs=1e-6)


def test_trim_strategies():
    t = _table(50, 1)
    left = AnglesTableDataset([t], pad=32, trim_strategy="leftalign")[0]
    assert torch.equal(left["angles"], torch.from_numpy(t[:32]).float()) and int(left["lengths"]) == 32
    crop = AnglesTableDataset([t], pad=32, trim_strategy="randomcrop")[0]
    start = np.random.default_rng(seed=6489).integers(0, 50 - 32)  # the reference's crop rng (datasets.py:111)
    assert torch.equal(crop["angles"], torch.from_numpy(t[start:start + 32]).float())
    kept = AnglesTableDataset([t, _table(20), _table(32)], pad=32, trim_strategy="discard")
    assert len(kept) == 2 and int(kept[0]["lengths"]) == 20 and int(kept[1]["lengths"]) == 32
    with pytest.raises(ValueError):
        AnglesTableDataset([t], trim_strategy="middle")


def test_reads_writers_tables(tmp_path):
    tabs = [_table(l, l).astype(np.float32) for l in (12, 40)]
    for i, t in enumerate(tabs):
        writers.write_angles_csv_gz(t, NAMES, str(tmp_path / f"generated_{i}.csv.gz"))
    ds = AnglesTableDataset(str(tmp_path), pad=64)
    assert len(ds) == 2 and ds.filenames[0].endswith("generated_0.csv.gz")
    for i, t in enumerate(tabs):
        assert torch.equal(ds[i]["angles"][: t.shape[0]], torch.from_numpy(t))
    with pytest.raises(FileNotFoundError):
        AnglesTableDataset(str(tmp_path / "nothing"))


def test_collated_batch_layout():
    nd = NoisedAnglesDataset(AnglesTableDataset([_table(l, l) for l in (5, 17, 9)], pad=24), timesteps=50)
    torch.manual_seed(0)
    b = default_collate([nd[i] for i in range(3)])
    assert b["corrupted"].shape == b["known_noise"].shape == b["angles"].shape == (3, 24, 6)
    assert b["t"].shape == (3, 1) and b["t"].dtype == torch.long
    assert b["attn_mask"].shape == (3, 24) and b["position_ids"].shape == (3, 24)
    assert b["lengths"].tolist() == [5, 17, 9]
    assert b["sqrt_alphas_cumprod_t"].shape == b["sqrt_one_minus_alphas_cumprod_t"].shape == (3,)
    lengths, _, prefix = modelling.mask_layout(b["attn_mask"])
    assert lengths == [5, 17, 9] and prefix


def test_mask_layout_detects_non_prefix():
    m = torch.ones(2, 8)
    m[1, 3] = 0
    assert not modelling.mask_layout(m)[2]
    assert not modelling.mask_layout(torch.zeros(1, 4))[2]


def test_constructor_surface():
    _, cfg, _, _ = mini_state_dict()
    c = modelling.BertConfig(**cfg)
    m = modelling.BertForDiffusion(config=c, loss="radian_l1_smooth", use_pairwise_dist_loss=(0.1, 1.0, 250),
                                   circle_reg=0.2, lr=1e-4, l1=0.0, l2=0.1, epochs=3, steps_per_epoch=7,
                                   lr_scheduler="LinearWarmup")
    assert m.loss == "smooth_l1" and m.pdist_enabled and m.use_pairwise_dist_loss == [0.1, 1.0, 250]
    assert not modelling.BertForDiffusion(config=c).pdist_enabled
    with pytest.raises(NotImplementedError):
        modelling.BertForDiffusion(config=c, loss=torch.nn.functional.l1_loss)
    with pytest.raises(NotImplementedError):
        modelling.BertForDiffusion(config=c, write_preds_to_dir="/nonexistent")
    with pytest.raises(ValueError):
        modelling.BertForDiffusion(config=c, loss="mse")
    with pytest.raises(NotImplementedError, match="backward"):
        m.training_step({}, 0)


def test_pdist_coefficients_follow_reference():
    t = torch.tensor([[0], [100], [249]])
    c = losses.pdist_coefficients([0.5, 2.0, 250], t)
    want = (0.5 + (2.0 - 0.5) * ((250 - t) / 250)).reshape(-1)
    assert torch.equal(c, want)
    assert torch.equal(losses.pdist_coefficients(3.0, t), torch.full((3,), 3.0))


def test_eval_loss_cli_help_and_errors(tmp_path):
    script = os.path.join(ROOT, "bin", "eval_loss.py")
    r = subprocess.run([sys.executable, script, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--exhaustive-t" in r.stdout and "--noise" in r.stdout
    r = subprocess.run([sys.executable, script, "-m", str(tmp_path), "--angles", str(tmp_path), "-o", "x.json"],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "training_args.json" in r.stderr
    r = subprocess.run([sys.executable, script, "-m", str(tmp_path), "--angles", str(tmp_path), "--exhaustive-t",
                        "--t", "3", "-o", "x.json"], capture_output=True, text=True)
    assert r.returncode == 2 and "not allowed" in r.stderr
    r = subprocess.run([sys.executable, script, "-m", str(tmp_path), "--angles", str(tmp_path), "--noise", "numpy",
                        "-o", "x.json"], capture_output=True, text=True)
    assert r.returncode == 2


@pytest.mark.skipif(not os.path.isfile(os.path.join(GOLDEN, "ref_pdist.npz")), reason="ref_pdist.npz not generated")
def test_pdist_oracle_reproduces_reference_answers():
    z = load_golden("ref_pdist.npz")
    names = [str(n) for n in z["names"]]
    # the stock scalar form raises inside losses.pairwise_dist_loss (weights.ndim of a float); the ramp form runs
    assert "AttributeError" in str(z["scalar_raises"])
    for tag in ("ramp",):
        inp = {k: torch.from_numpy(z[f"{tag}_{k}"]) for k in ("corrupted", "pred", "angles", "sa", "s1m", "coef",
                                                              "lengths")}
        got, _ = loss_oracle.pdist_term(inp["corrupted"], inp["pred"], inp["angles"], inp["sa"], inp["s1m"],
                                        inp["coef"], inp["lengths"].tolist(), names, torch.float64)
        want = float(z[f"{tag}_pdist"])
        # the reference mixes fp32 bond terms into fp64 coordinates, the restatement is fp64 throughout: agreement is
        # to the fp32 rounding of those terms, not bit for bit
        assert abs(float(got) - want) <= 1e-5 * abs(want), (tag, float(got), want)
        terms = torch.from_numpy(z[f"{tag}_terms"])
        assert terms.shape == (7,) and float(terms[-1]) == want
