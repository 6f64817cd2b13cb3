"""
The training objective on the device (csrc/loss.cuh through the C ABI): forward noising, the per-feature loss terms, the
pairwise-distance term, BertForDiffusion._get_loss_terms end to end, losses.validation_loss and bin/eval_loss.py.
Compared against the host mirror (bit for bit), the CPU oracle (oracle/loss.py, oracle/forward.py) and the pdist
restatement in tests/loss_oracle.py.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import loss_oracle
from conftest import ROOT, mini_state_dict, write_model_dir
from gpu_util import GEMMS, prefix_mask, prod_state_dict
from foldingdiff_b200 import _native, losses, modelling, synthetic, writers
from foldingdiff_b200.datasets import (FEATURE_SET_NAMES_TO_FEATURE_NAMES, AnglesTableDataset, NoisedAnglesDataset,
                                       SyntheticAnglesDataset)
from oracle import forward as ofwd
from oracle import loss as oloss

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RAGGED = [1, 128, 37, 64, 2, 100, 127, 50]


def _device_q_sample(nd, items, zs):
    key = nd.dset_key
    x0 = torch.stack([it["x0"] for it in items]).to(DEV)
    t = torch.tensor([it["t"] for it in items])
    sa = nd.alpha_beta_terms["sqrt_alphas_cumprod"][t].to(torch.float32)
    s1m = nd.alpha_beta_terms["sqrt_one_minus_alphas_cumprod"][t].to(torch.float32)
    ang = nd.feature_is_angular[key]
    scales = [nd.angular_var_scale if a else nd.nonangular_var_scale for a in ang]
    z = None if zs is None else torch.stack(zs).to(DEV)
    return losses.q_sample(x0, sa.to(DEV), s1m.to(DEV), ang, scales, z=z)


@pytest.mark.parametrize("fset,ang_var,nonang_var", [("canonical-full-angles", 1.0, 1.0),
                                                     ("canonical-full-angles", 0.7, 1.0),
                                                     ("canonical", 1.3, 0.6), ("cart-coords", 1.0, 2.5)])
def test_q_sample_torch_noise_matches_host_mirror(fset, ang_var, nonang_var):
    T = 1000
    base = SyntheticAnglesDataset(8, 90, feature_set_key=fset, scale=1.5, seed=3)
    key = "angles"
    nd = NoisedAnglesDataset(base, dset_key=key, timesteps=T, beta_schedule="cosine", angular_variance=ang_var,
                             nonangular_variance=nonang_var)
    ts = [0, 1, T // 2, T - 1, 0, 999, 250, 1]  # mixed t within one batch
    items, zs, host = [], [], []
    for i, t in enumerate(ts):
        torch.manual_seed(1000 + i)
        host.append(nd.__getitem__(i, use_t_val=t))
        torch.manual_seed(1000 + i)
        zs.append(torch.randn(base.pad, len(nd.feature_is_angular[key])))  # the draw sample_noise makes
        items.append({"x0": base[i]["angles"], "t": t})
    known, corrupted = _device_q_sample(nd, items, zs)
    for i, h in enumerate(host):
        assert torch.equal(known[i].cpu(), h["known_noise"]), (fset, i)
        assert torch.equal(corrupted[i].cpu(), h["corrupted"]), (fset, i)


def test_q_sample_philox_equals_predrawn_fd_randn():
    base = SyntheticAnglesDataset(5, 70, seed=1)
    nd = NoisedAnglesDataset(base, timesteps=100, beta_schedule="linear", angular_variance=0.9)
    items = [{"x0": base[i]["angles"], "t": t} for i, t in enumerate([0, 5, 50, 99, 12])]
    B, N, F = 5, base.pad, 6
    seed, offset = 1234, 7 * N * F + 3
    x0 = torch.stack([it["x0"] for it in items]).to(DEV)
    t = torch.tensor([it["t"] for it in items])
    sa = nd.alpha_beta_terms["sqrt_alphas_cumprod"][t].to(DEV)
    s1m = nd.alpha_beta_terms["sqrt_one_minus_alphas_cumprod"][t].to(DEV)
    z = torch.empty(B, N, F, device=DEV)
    _native.check(_native.lib().fd_randn(z.data_ptr(), z.numel(), seed, offset, torch.cuda.current_stream().cuda_stream),
                  "fd_randn")
    scales = [0.9] * 6
    a = losses.q_sample(x0, sa, s1m, [True] * 6, scales, z=None, seed=seed, offset=offset)
    b = losses.q_sample(x0, sa, s1m, [True] * 6, scales, z=z)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("loss,circle,ang", [("smooth_l1", 0.0, [True] * 6), ("l1", 0.0, [True] * 6),
                                             ("smooth_l1", 0.3, [True] * 6),
                                             ("smooth_l1", 0.0, [False, False, False, True, True, True, True, True, True]),
                                             ("l1", 0.0, [False, False, True])])
def test_loss_terms_match_oracle(loss, circle, ang):
    g = torch.Generator().manual_seed(len(ang) + int(circle * 10))
    B, N, F = len(RAGGED), 128, len(ang)
    pred = torch.randn(B, N, F, generator=g) * 2.5  # |pred| > pi on some entries: the circle term is exercised
    known = torch.randn(B, N, F, generator=g)
    mask = prefix_mask(RAGGED, N)
    want = oloss.loss_terms(pred, known, mask, ang, loss, circle)
    got, chain = losses.loss_terms(pred.to(DEV), known.to(DEV), mask.to(DEV), ang, loss, circle)
    rel = ((got.cpu().double() - want.double()).abs() / want.double().abs()).max().item()
    print(f"loss={loss} circle={circle} F={F}: max rel diff {rel:.2e}")
    assert rel < 2e-6, rel
    assert chain[:, 2 * F].cpu().tolist() == [float(l) for l in RAGGED]


def _mini_bfd(gemm, **kw):
    sd, cfg, _, _ = mini_state_dict()
    m = modelling.BertForDiffusion(config=modelling.BertConfig(**cfg), ft_is_angular=[True] * 6,
                                   ft_names=FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"], **kw)
    m.load_state_dict(sd)
    return m.to(DEV).set_gemm(gemm), ofwd.OracleModel(sd, ofwd.OracleConfig(**cfg), [True] * 6).eval()


def _prod_bfd(gemm, **kw):
    m = modelling.BertForDiffusion(config=modelling.BertConfig(**synthetic.PRODUCTION), ft_is_angular=[True] * 6,
                                   ft_names=FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"], **kw)
    m.load_state_dict(prod_state_dict())
    return m.to(DEV).set_gemm(gemm), ofwd.OracleModel(prod_state_dict(), ofwd.OracleConfig(**synthetic.PRODUCTION),
                                                      [True] * 6).eval()


def _noised_batch(lengths, T=250, seed=0, schedule="cosine"):
    from torch.utils.data import default_collate
    g = torch.Generator().manual_seed(seed)
    tabs = [synthetic_table(l, g) for l in lengths]
    nd = NoisedAnglesDataset(AnglesTableDataset(tabs), timesteps=T, beta_schedule=schedule)
    torch.manual_seed(seed)
    return default_collate([nd[i] for i in range(len(lengths))])


def synthetic_table(l, g):
    return (torch.rand(l, 6, generator=g) * 2 - 1).numpy() * np.pi


@pytest.mark.parametrize("gemm", GEMMS)
@pytest.mark.parametrize("shape", ["mini", "production"])
def test_get_loss_terms_end_to_end(gemm, shape):
    lengths = RAGGED * (1 if shape == "mini" else 4)
    model, oracle = (_mini_bfd if shape == "mini" else _prod_bfd)(gemm)
    batch = _noised_batch(lengths, seed=11)
    got = model._get_loss_terms(batch).cpu()
    with torch.no_grad():
        eps = oracle(batch["corrupted"], batch["t"].reshape(-1), batch["attn_mask"])
    want = oloss.loss_terms(eps, batch["known_noise"], batch["attn_mask"], [True] * 6)
    err = (got - want).abs().max().item()
    print(f"{shape} {gemm}: max |term - oracle| = {err:.2e}")
    assert err < 5e-5, err
    v = model.validation_step(batch, 0)["val_loss"]
    assert torch.equal(v, torch.mean(model._get_loss_terms(batch)))


@pytest.mark.parametrize("t", [0, 100, 500])
def test_pdist_within_rounding_of_fp64_oracle(t):
    T, lengths = 1000, [1, 2, 40, 128, 77, 128]
    g = torch.Generator().manual_seed(t + 5)
    B, N, F = len(lengths), 128, 6
    angles = torch.from_numpy(np.stack([np.pad(synthetic_table(l, g), ((0, N - l), (0, 0))) for l in lengths])).float()
    nd = NoisedAnglesDataset(AnglesTableDataset([a[:l].numpy() for a, l in zip(angles, lengths)]), timesteps=T,
                             beta_schedule="linear")
    sa = nd.alpha_beta_terms["sqrt_alphas_cumprod"][t].repeat(B).float()
    s1m = nd.alpha_beta_terms["sqrt_one_minus_alphas_cumprod"][t].repeat(B).float()
    z = torch.randn(B, N, F, generator=g)
    eps = z + 0.05 * torch.randn(B, N, F, generator=g)
    corrupted = oloss.wrap(sa.reshape(B, 1, 1) * angles + s1m.reshape(B, 1, 1) * z, -np.pi, np.pi)
    names = FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"]
    for coef_form in (2.0, [0.5, 3.0, T]):
        coef = losses.pdist_coefficients(coef_form, torch.full((B, 1), t, dtype=torch.long))
        got, _, den = losses.pdist_loss(corrupted.to(DEV), eps.to(DEV), angles.to(DEV), sa.to(DEV), s1m.to(DEV),
                                        coef.to(DEV), lengths, names, return_denoised=True)
        ref64, den_ref = loss_oracle.pdist_term(corrupted, eps, angles, sa, s1m, coef, lengths, names, torch.float64)
        ref32, _ = loss_oracle.pdist_term(corrupted, eps, angles, sa, s1m, coef, lengths, names, torch.float32)
        assert torch.equal(den.cpu(), den_ref)  # the denoising step is the reference's fp32 op order, bit for bit
        floor = abs(float(ref32) - float(ref64))
        err = abs(float(got) - float(ref64))
        print(f"t={t} coef={coef_form}: pdist {float(got):.6e}; |gpu - fp64| = {err:.2e}, |fp32 - fp64| = {floor:.2e}")
        assert err <= 10 * floor + 1e-6 * abs(float(ref64)), (err, floor)


def _table_dset(n, seed, pad=128):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(40, 128, (n,), generator=g).tolist()
    return AnglesTableDataset([synthetic_table(l, g) for l in lens], pad=pad)


def test_validation_loss_equals_manual_loop_and_per_t_table():
    from torch.utils.data import default_collate
    model, _ = _mini_bfd("tc3x")
    nd = NoisedAnglesDataset(_table_dset(13, 2), timesteps=250, beta_schedule="cosine")
    torch.manual_seed(5)
    res = losses.validation_loss(model, nd, batch_size=4, noise="torch")
    torch.manual_seed(5)
    means, terms = [], []
    for s in range(0, len(nd), 4):
        tt = model._get_loss_terms(default_collate([nd[i] for i in range(s, min(len(nd), s + 4))]))
        means.append(torch.mean(tt))
        terms.append(tt)
    assert res["val_loss"] == float(torch.mean(torch.stack(means)).item())
    assert list(res["terms"].values()) == torch.stack(terms).cpu().mean(dim=0).tolist()

    ex = NoisedAnglesDataset(_table_dset(3, 4), timesteps=250, beta_schedule="cosine", exhaustive_t=True)
    torch.manual_seed(9)
    per = losses.validation_loss(model, ex, batch_size=256, noise="torch")["per_t"]
    torch.manual_seed(9)
    whole = losses.validation_loss(model, ex, batch_size=len(ex), noise="torch")["terms"]
    tab = torch.tensor(per["loss"], dtype=torch.float64)
    tok = torch.tensor(per["tokens"], dtype=torch.float64)
    rew = (tab * tok[:, None]).sum(0) / tok.sum()
    want = torch.tensor(list(whole.values()), dtype=torch.float64)
    rel = ((rew - want).abs() / want.abs()).max().item()
    print(f"per-t table re-weighted vs whole-set token mean: max rel {rel:.2e}")
    assert rel < 1e-6
    assert tab.shape == (250, 6)


@pytest.mark.parametrize("noise", ["torch", "philox"])
def test_runs_are_bit_identical(noise):
    model, _ = _mini_bfd("tc3x", use_pairwise_dist_loss=[0.5, 2.0, 250])
    nd = NoisedAnglesDataset(_table_dset(9, 6), timesteps=250, beta_schedule="cosine")
    out = []
    for _ in range(2):
        torch.manual_seed(1)
        out.append(losses.validation_loss(model, nd, batch_size=4, noise=noise, seed=3))
    assert out[0] == out[1]
    assert len(out[0]["terms"]) == 7 and np.isfinite(out[0]["val_loss"])


def test_eval_loss_cli(tmp_path):
    sd, cfg, targs, ckpt = mini_state_dict()
    mdir = write_model_dir(str(tmp_path / "model"), sd, cfg, targs, ckpt,
                           mean_offset=np.linspace(-0.2, 0.2, 6).astype(np.float64))
    adir = tmp_path / "angles"
    os.makedirs(adir)
    g = torch.Generator().manual_seed(0)
    names = FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"]
    for i, l in enumerate([45, 60, 128, 90]):
        writers.write_angles_csv_gz(synthetic_table(l, g).astype(np.float32), names, str(adir / f"generated_{i}.csv.gz"))
    out = tmp_path / "out.json"
    cmd = [sys.executable, os.path.join(ROOT, "bin", "eval_loss.py"), "-m", mdir, "--angles", str(adir), "-b", "3",
           "--exhaustive-t", "--noise", "philox", "-o", str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.load(open(out))
    assert {"val_loss", "terms", "per_t", "n_structures"} <= set(d)
    assert d["n_structures"] == 4 and len(d["per_t"]["loss"]) == targs["timesteps"]
    res = subprocess.run(cmd[:-5] + ["--t", "0", "100", "-o", str(out)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert set(json.load(open(out))["at_t"]) == {"0", "100"}
