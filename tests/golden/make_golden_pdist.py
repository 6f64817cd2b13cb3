#!/usr/bin/env python
"""
Generate tests/golden/ref_pdist.npz: the STOCK reference's BertForDiffusion._get_loss_terms with the pairwise-distance
term switched on, for tests/test_loss_cpu.py::test_pdist_oracle_reproduces_reference_answers.

    python tests/golden/make_golden_pdist.py

Needs the unmodified reference package in baseline/_ref (see tests/golden/make_golden_reference.py).  The method runs
on a stand-in `self` (forward returns a fixed prediction; ft_names, loss_func, circle_lambda and
use_pairwise_dist_loss as BertForDiffusion.__init__ sets them), once with a scalar coefficient ("scalar") and once
with the [min, max, T] form ("ramp").  Stored per case: the inputs, the per-chain coefficients, the returned terms and
the pairwise term - or, where the stock code raises, the error ("<tag>_raises"): the scalar form does, because
losses.pairwise_dist_loss reads `weights.ndim` of the Python float it is given (losses.py:141-147).
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "baseline")):
    sys.path.insert(0, p)

import reference_arm  # noqa: E402

NAMES = ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"]
T = 250
LENGTHS = [32, 10, 25, 3]


def inputs(seed):
    g = torch.Generator().manual_seed(seed)
    B, N = len(LENGTHS), 32
    angles = torch.zeros(B, N, 6)
    mask = torch.zeros(B, N)
    for b, l in enumerate(LENGTHS):
        angles[b, :l] = (torch.rand(l, 6, generator=g) * 2 - 1) * torch.pi
        mask[b, :l] = 1.0
    t = torch.randint(0, T, (B, 1), generator=g)
    abar = torch.cos(torch.linspace(0.05, 1.5, T)) ** 2  # any decreasing table in (0, 1)
    sa, s1m = abar[t.reshape(-1)].sqrt(), (1 - abar[t.reshape(-1)]).sqrt()
    z = torch.randn(B, N, 6, generator=g)
    corrupted = sa.view(B, 1, 1) * angles + s1m.view(B, 1, 1) * z
    corrupted = (corrupted + torch.pi) % (2 * torch.pi) - torch.pi
    pred = z + 0.1 * torch.randn(B, N, 6, generator=g)
    batch = {"corrupted": corrupted, "t": t, "known_noise": z, "attn_mask": mask,
             "position_ids": torch.arange(N).expand(B, -1), "lengths": torch.tensor(LENGTHS), "angles": angles,
             "sqrt_alphas_cumprod_t": sa, "sqrt_one_minus_alphas_cumprod_t": s1m}
    return batch, pred


def main():
    assert reference_arm.available(), "baseline/_ref is not installed: run __graft_entry__.build() where the reference is"
    _, _, _, rm = reference_arm.load_reference()
    base = rm.BertForDiffusionBase
    out = {"names": np.array(NAMES)}
    for tag, coef, seed in (("scalar", 0.7, 1), ("ramp", [0.2, 1.5, T], 2)):
        batch, pred = inputs(seed)
        me = types.SimpleNamespace(forward=lambda *a, **k: pred, ft_names=NAMES, circle_lambda=0.0,
                                   loss_func=[base.angular_loss_fn_dict["smooth_l1"]] * 6, use_pairwise_dist_loss=coef)
        try:
            terms = rm.BertForDiffusion._get_loss_terms(me, batch)
        except AttributeError as e:  # losses.py:143 reads weights.ndim, which a Python float does not have
            out[f"{tag}_raises"] = np.array(f"AttributeError: {e}")
            continue
        if isinstance(coef, list):
            w = coef[0] + (coef[1] - coef[0]) * ((coef[2] - batch["t"]) / coef[2])
        else:
            w = torch.full((len(LENGTHS),), coef)
        for k, v in (("corrupted", batch["corrupted"]), ("pred", pred), ("angles", batch["angles"]),
                     ("sa", batch["sqrt_alphas_cumprod_t"]), ("s1m", batch["sqrt_one_minus_alphas_cumprod_t"]),
                     ("coef", w.reshape(-1).float()), ("lengths", batch["lengths"]), ("t", batch["t"])):
            out[f"{tag}_{k}"] = v.numpy()
        out[f"{tag}_terms"] = terms.detach().numpy()
        out[f"{tag}_pdist"] = np.array(terms[-1].item())
    path = os.path.join(HERE, "ref_pdist.npz")
    np.savez_compressed(path, **out)
    print(f"wrote ref_pdist.npz: {os.path.getsize(path) / 1e3:.1f} kB; ramp: {float(out['ramp_pdist']):.6e} "
          f"({out['ramp_terms'].dtype}); scalar: {out.get('scalar_raises', 'ok')}")


if __name__ == "__main__":
    main()
