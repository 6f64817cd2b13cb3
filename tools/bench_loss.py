#!/usr/bin/env python
"""
Throughput of the loss evaluation (BertForDiffusion._get_loss_terms on the device) at config-2 shape: 512 structures
of lengths 50-127, synthetic production weights, one exhaustive-validation slice of t.  Prints one JSON line:

    python tools/bench_loss.py [--n 512] [--timesteps 1000] [--t-slice 8] [--warmup 2]

Reported: the GPU name and power limit (nvidia-smi in the same run); per noise source ("torch": host draws as in the
reference, "philox": noise drawn on the device) the evaluation rate in chain-timesteps/s over the timed slice and
CUDA-event times of q-sample, forward (valid rows only), loss terms and pairwise term per batch; the same batches
through the all-rows `modelling.forward` for the valid-rows saving; and the full exhaustive pass (N x T forwards)
extrapolated from the slice - flagged as such, not measured.  Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from foldingdiff_b200 import beta_schedules, losses, modelling, synthetic  # noqa: E402
from foldingdiff_b200.datasets import FEATURE_SET_NAMES_TO_FEATURE_NAMES  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def timed(fn, ev):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    ev.append((a, b))
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=512)
    p.add_argument("--timesteps", type=int, default=1000)
    p.add_argument("--t-slice", type=int, default=8, help="timesteps timed (spread over [0, T))")
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--gemm", default="tc3x")
    args = p.parse_args()
    dev = "cuda:0"
    names = FEATURE_SET_NAMES_TO_FEATURE_NAMES["canonical-full-angles"]
    model = modelling.BertForDiffusion(config=modelling.BertConfig(**synthetic.PRODUCTION), ft_is_angular=[True] * 6,
                                       ft_names=names, use_pairwise_dist_loss=[0.1, 1.0, args.timesteps])
    model.load_state_dict(synthetic.synthetic_state_dict(synthetic.PRODUCTION, seed=0))
    model = model.to(dev).set_gemm(args.gemm).eval()
    eng = model.native_engine()
    T, B, N, F = args.timesteps, args.n, 128, 6
    lengths = synthetic.sweep_lengths(B, 50, 127)
    g = torch.Generator().manual_seed(0)
    x0 = torch.zeros(B, N, F)
    mask = torch.zeros(B, N)
    for b, l in enumerate(lengths):
        x0[b, :l] = (torch.rand(l, F, generator=g) * 2 - 1) * torch.pi
        mask[b, :l] = 1.0
    x0, mask_d = x0.to(dev), mask.to(dev)
    tabs = beta_schedules.compute_alphas(beta_schedules.get_variance_schedule("cosine", T))
    sa_tab = tabs["sqrt_alphas_cumprod"].float()
    s1m_tab = tabs["sqrt_one_minus_alphas_cumprod"].float()
    t_list = [int(round(i * (T - 1) / max(1, args.t_slice - 1))) for i in range(args.t_slice)]

    def one(t, noise, ev):
        tt = torch.full((B, 1), t, dtype=torch.long)
        sa, s1m = sa_tab[tt.reshape(-1)].to(dev), s1m_tab[tt.reshape(-1)].to(dev)
        z = torch.randn(B, N, F).to(dev) if noise == "torch" else None  # host draw, as the reference's loader does
        known, corrupted = timed(lambda: losses.q_sample(x0, sa, s1m, [True] * F, [1.0] * F, z=z, seed=1,
                                                         offset=t * B * N * F), ev["q_sample"])
        eng.set_batch(lengths, N, all_rows=False)
        temb = model._time_rows(tt.reshape(-1)).to(dev)
        eps = timed(lambda: eng.forward(corrupted, temb), ev["forward"])
        terms, _ = timed(lambda: losses.loss_terms(eps, known, mask_d, [True] * F), ev["loss"])
        coef = losses.pdist_coefficients(model.use_pairwise_dist_loss, tt.to(dev))
        pd, _ = timed(lambda: losses.pdist_loss(corrupted, eps, x0, sa, s1m, coef, lengths, names), ev["pdist"])
        allrows = timed(lambda: model.forward(corrupted, tt, mask_d), ev["forward_all_rows"])
        return terms, pd, allrows

    result = {"metric": "loss_eval", "gpu_count": 1, "gemm": args.gemm, "n_structures": B, "timesteps": T,
              "lengths": "50-127 (synthetic.sweep_lengths)", "weights": "synthetic production (seed 0)",
              "t_slice": t_list, "warmup_passes": args.warmup}
    name, power = gpu_info()
    result["gpu_name"], result["power_limit"] = name, power
    for noise in ("torch", "philox"):
        for _ in range(args.warmup):
            one(t_list[0], noise, {k: [] for k in ("q_sample", "forward", "loss", "pdist", "forward_all_rows")})
        torch.cuda.synchronize()
        ev = {k: [] for k in ("q_sample", "forward", "loss", "pdist", "forward_all_rows")}
        stop = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        wall0 = torch.cuda.Event(enable_timing=True)
        wall0.record()
        for t in t_list:
            one(t, noise, ev)
        stop.record()
        torch.cuda.synchronize()
        total_ms = wall0.elapsed_time(stop)
        per = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in ev.items()}
        # the loss pass alone (no all-rows comparison forward): q-sample + valid-rows forward + loss + pdist
        loss_ms = per["q_sample"] + per["forward"] + per["loss"] + per["pdist"]
        result[noise] = {
            "ms_per_batch": {k: round(v, 4) for k, v in per.items()},
            "loss_pass_ms_per_batch": round(loss_ms, 4),
            "chain_timesteps_per_s": round(B / (loss_ms / 1e3), 1),
            "wall_ms_for_slice_incl_host": round(total_ms, 2),
            "valid_rows_forward_saving": round(1.0 - per["forward"] / per["forward_all_rows"], 4),
            "exhaustive_pass_s_extrapolated": round(T * loss_ms / 1e3, 2),
        }
    result["note"] = ("exhaustive_pass_s_extrapolated = T x the measured per-batch loss time for one 512-chain batch; "
                      "extrapolated from the timed slice, not measured over all T")
    print(json.dumps(result))


if __name__ == "__main__":
    with torch.no_grad():
        main()
