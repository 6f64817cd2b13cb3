#!/usr/bin/env python
"""
Generate the stored answers of the STOCK reference package that the differential tests compare against:

    python tests/golden/make_golden_reference.py

Needs the unmodified reference package in baseline/_ref (installed by __graft_entry__.build() where the reference's
sources are present; see baseline/reference_arm.py).  The tests themselves only read the files written here, so they
run on any machine.  Each output is computed on the same inputs the corresponding test builds:

  ref_host.npz  tests/test_host_vs_installed_reference.py: schedules + alpha tables, modulo_with_wrapped_range,
                AnglesEmptyDataset / NoisedAnglesDataset (metadata, noise, forward-noised items), sampling.sample
                (its output, and the calls its loop made to the model)
  ref_loss.npz  tests/test_oracle_loss.py: losses.radian_smooth_l1_loss / radian_l1_loss, BertForDiffusion
                ._get_loss_terms, and the gradient torch autograd takes through them
  ref_loop.npz  tests/test_oracle_golden.py: sampling.p_sample_loop around the oracle forward (with its model calls);
                tests/test_reference_arm.py: the reference-assembled model's forward and the stock loop around it
Where a test compares bit for bit, the file holds the answer's digest (oracle/replay.py) rather than the array.
"""
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS, os.path.join(ROOT, "baseline")):
    sys.path.insert(0, p)

import reference_arm  # noqa: E402
from conftest import mini_state_dict  # noqa: E402
from oracle import forward as ofwd  # noqa: E402
from oracle.replay import Recorder, digest  # noqa: E402
import test_host_vs_installed_reference as t_host  # noqa: E402  (the tests' own input builders)
import test_oracle_loss as t_loss  # noqa: E402


def save(name, arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}: {os.path.getsize(path) / 1e3:.1f} kB")


def host(ref):
    sampling, rbeta, rutils, rdatasets = ref.sampling, ref.beta_schedules, ref.utils, ref.datasets
    out = {}
    for kind in ("linear", "cosine", "quadratic"):
        for T in (2, 100, 250, 1000):
            tab = rbeta.compute_alphas(rbeta.get_variance_schedule(kind, T))
            out[f"sched_{kind}_{T}_keys"] = np.array(list(tab))
            for k, v in tab.items():
                out[f"sched_{kind}_{T}_{k}"] = np.array(digest(v))

    x = t_host.wrap_inputs()
    out["wrap_default"] = np.array(digest(rutils.modulo_with_wrapped_range(x)))
    for i, (lo, hi) in enumerate(t_host.WRAP_RANGES):
        out[f"wrap_range{i}"] = np.array(digest(rutils.modulo_with_wrapped_range(x, lo, hi)))
    out["wrap_np64"] = np.array(digest(rutils.modulo_with_wrapped_range(x.numpy().astype(np.float64), -2, 2)))

    with tempfile.TemporaryDirectory() as d:
        t_host.write_dataset_dir(d)
        theirs = rdatasets.AnglesEmptyDataset.from_dir(d)
        out["dset_feature_names"] = np.array(json.dumps(theirs.feature_names))
        out["dset_feature_is_angular"] = np.array(json.dumps(theirs.feature_is_angular))
        out["dset_pad"] = np.array(theirs.pad)
        out["dset_masked_means"] = np.array(digest(theirs.get_masked_means()))
        for i, kw in enumerate(t_host.NOISE_KWARGS):
            nt = rdatasets.NoisedAnglesDataset(theirs, timesteps=100, beta_schedule="cosine", **kw)
            for k, v in nt.alpha_beta_terms.items():
                out[f"dset{i}_terms_{k}"] = np.array(digest(v))
            out[f"dset{i}_terms_keys"] = np.array(list(nt.alpha_beta_terms))
            torch.manual_seed(7344)
            out[f"dset{i}_noise"] = np.array(digest(nt.sample_noise(torch.zeros(7, 128, 6))))

    for schedule in ("linear", "cosine"):
        nt = rdatasets.NoisedAnglesDataset(t_host._Inner(), timesteps=50, beta_schedule=schedule)
        for idx, tval in t_host.ITEMS:
            torch.manual_seed(100 + idx)
            item = nt.__getitem__(idx, use_t_val=tval)
            key = f"item_{schedule}_{idx}_{tval}"
            out[key + "_keys"] = np.array(list(item))
            for k, v in item.items():
                out[f"{key}_{k}"] = np.array(digest(torch.as_tensor(v)))

    # sampling.sample: the stock orchestration around the stock loop; the model is the reference-assembled one
    sd, cfg, _, _ = mini_state_dict()
    with tempfile.TemporaryDirectory() as d:
        t_host.write_sample_dir(d)
        r_dset = rdatasets.NoisedAnglesDataset(rdatasets.AnglesEmptyDataset.from_dir(d), timesteps=t_host.SAMPLE_T,
                                               beta_schedule="cosine")
        for i, kw in enumerate(t_host.SAMPLE_KWARGS):
            rec = Recorder(reference_arm.build_model(sd, cfg))
            torch.manual_seed(77)
            got = sampling.sample(rec, r_dset, disable_pbar=True, **kw)
            out[f"sample{i}_n"] = np.array(len(got))
            for j, s in enumerate(got):
                out[f"sample{i}_out_{j}"] = np.array(digest(s))
            out.update(rec.arrays(f"sample{i}"))
        try:
            sampling.sample(rec, r_dset, n=1, sweep_lengths=(30, 30))
            raise AssertionError("the reference accepted an empty length sweep")
        except ValueError:
            pass
    return out


def reference_terms(ref, pred, batch, is_angular, loss="smooth_l1", circle=0.0):
    """The unmodified `_get_loss_terms` with a stand-in `self` whose forward returns `pred`."""
    base = ref.modelling.BertForDiffusionBase
    fns = [base.angular_loss_fn_dict[loss] if a else base.nonangular_loss_fn_dict[loss] for a in is_angular]  # modelling.py:522-527
    me = types.SimpleNamespace(forward=lambda *a, **k: pred, loss_func=fns, circle_lambda=circle, use_pairwise_dist_loss=0.0)
    return ref.modelling.BertForDiffusion._get_loss_terms(me, batch)


def loss(ref):
    out = {}
    for i, (x, y) in enumerate(t_loss.loss_fn_inputs()):
        for b, beta in enumerate(t_loss.BETAS):
            for c, cp in enumerate(t_loss.CIRCLE_PENALTIES):
                out[f"fn{i}_smooth_l1_{b}_{c}"] = ref.losses.radian_smooth_l1_loss(x, y, beta=beta, circle_penalty=cp).numpy()
        out[f"fn{i}_l1"] = ref.losses.radian_l1_loss(x, y).numpy()
    for is_angular in t_loss.TERMS_FEATURES:
        for name in ("smooth_l1", "l1"):
            pred, known, mask = t_loss._batch(seed=len(is_angular), F=len(is_angular))
            batch = {"known_noise": known, "corrupted": known, "t": torch.zeros(known.shape[0], 1, dtype=torch.long),
                     "attn_mask": mask, "position_ids": torch.arange(known.shape[1])[None].expand(known.shape[0], -1)}
            out[f"terms_{t_loss.features_tag(is_angular)}_{name}"] = reference_terms(ref, pred, batch, is_angular, name).numpy()
    for is_angular in t_loss.GRAD_FEATURES:
        pred, known, mask = t_loss._batch(seed=5, F=len(is_angular))
        pred = pred.double().requires_grad_(True)
        batch = {"known_noise": known.double(), "corrupted": known.double(), "t": None, "attn_mask": mask, "position_ids": None}
        torch.mean(reference_terms(ref, pred, batch, is_angular)).backward()
        out[f"grad_{t_loss.features_tag(is_angular)}"] = pred.grad.numpy()
    return out


def loop(ref, oracle):
    import test_oracle_golden as t_golden
    import test_reference_arm as t_arm
    out = {}
    # the stock loop around the oracle forward (test_oracle_golden.py)
    T, lens = t_golden.LIVE_T, t_golden.LIVE_LENGTHS
    betas = ref.beta_schedules.get_variance_schedule("cosine", T)
    noise = t_golden.live_noise()
    rec = Recorder(oracle)
    torch.manual_seed(12)
    out["loop_hist"] = np.array(digest(ref.sampling.p_sample_loop(rec, lens, noise, T, betas, is_angle=[True] * 6, disable_pbar=True)))
    out["loop_betas"] = np.array(digest(betas))
    out["loop_wrap3"] = np.array(digest(ref.utils.modulo_with_wrapped_range(noise * 3)))
    out.update(rec.arrays("loop"))

    # the reference arm of bench.py (test_reference_arm.py)
    sd, cfg, _, _ = mini_state_dict()
    model = reference_arm.build_model(sd, cfg)
    x, t, mask = t_arm.forward_inputs()
    with torch.no_grad():
        out["arm_forward"] = model(x, t, mask).numpy()
    T, lens = t_arm.LOOP_T, t_arm.LOOP_LENGTHS
    betas = ref.beta_schedules.get_variance_schedule("linear", T)
    noise = t_arm.loop_noise()
    torch.manual_seed(5)
    out["arm_loop_hist"] = ref.sampling.p_sample_loop(model, lens, noise.clone(), T, betas, is_angle=[True] * 6,
                                                      disable_pbar=True).numpy()
    out["arm_loop_betas"] = np.array(digest(betas))
    return out


def main():
    torch.set_num_threads(os.cpu_count())
    assert reference_arm.available(), "baseline/_ref is not installed: run __graft_entry__.build() where the reference is"
    sampling, beta_schedules, utils, modelling = reference_arm.load_reference()
    from foldingdiff import datasets, losses  # type: ignore
    ref = types.SimpleNamespace(sampling=sampling, beta_schedules=beta_schedules, utils=utils, modelling=modelling,
                                datasets=datasets, losses=losses)
    sd, cfg, _, _ = mini_state_dict()
    oracle = ofwd.OracleModel(sd, ofwd.OracleConfig(**cfg), [True] * 6).eval()
    save("ref_host.npz", host(ref))
    save("ref_loss.npz", loss(ref))
    save("ref_loop.npz", loop(ref, oracle))


if __name__ == "__main__":
    main()
