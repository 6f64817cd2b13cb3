#!/usr/bin/env python
"""
Evaluate a trained foldingdiff model's denoising loss on held-out angle tables, on the GPU.

    python bin/eval_loss.py -m MODEL_DIR --angles DIR [-b 512] [--exhaustive-t | --t T [T ...]]
                            [--noise torch|philox] [--seed S] -o out.json

MODEL_DIR is a training output directory (config.json, training_args.json, models/); DIR holds *.csv.gz angle tables
as bin/sample.py writes them.  The model is built the way the reference's bin/train.py:437-459 builds it (loss,
use_pdist_loss [+ timesteps], circle_reg from training_args.json), the tables are featurised like its validation set
(mean offset, wrap, pad / trim) and noised with its schedule and variance scale.  The output JSON holds val_loss (what
the reference's validation epoch reports), the per-feature terms and, with --exhaustive-t, the loss at every timestep.
--t evaluates every structure at each given timestep instead of a random one.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from foldingdiff_b200 import losses, modelling  # noqa: E402
from foldingdiff_b200.datasets import (FEATURE_SET_NAMES_TO_FEATURE_NAMES, AnglesTableDataset,  # noqa: E402
                                       NoisedAnglesDataset)


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("-m", "--model", required=True, help="model directory (config.json, training_args.json, models/)")
    p.add_argument("--angles", required=True, help="directory of *.csv.gz angle tables")
    p.add_argument("-b", "--batchsize", type=int, default=512, help="structures per batch (default 512)")
    g = p.add_mutually_exclusive_group()
    g.add_argument("--exhaustive-t", action="store_true", help="evaluate every structure at every timestep")
    g.add_argument("--t", type=int, nargs="+", default=None, help="evaluate every structure at these timesteps")
    p.add_argument("--noise", choices=["torch", "philox"], default="torch",
                   help="torch: the reference's draws from torch's generator; philox: drawn on the device")
    p.add_argument("--seed", type=int, default=0, help="torch / Philox seed (default 0)")
    p.add_argument("--gemm", choices=["fp32", "tc3x"], default=None, help="GEMM arithmetic (default: the library's)")
    p.add_argument("--device", default="cuda:0")
    p.add_argument("-o", "--out", required=True, help="output JSON file")
    return p


def build_model(model_dir: str, targs: dict, device: str, gemm=None):
    """bin/train.py:446-459 of the reference: the loss-related kwargs from training_args.json."""
    pdist = targs.get("use_pdist_loss", 0.0)
    pdist = float(pdist) if isinstance(pdist, (int, float)) else [*pdist, targs["timesteps"]]
    model = modelling.BertForDiffusion.from_dir(model_dir, ft_names=FEATURE_SET_NAMES_TO_FEATURE_NAMES[targs["angles_definitions"]],
                                                loss=targs.get("loss", "smooth_l1"),
                                                use_pairwise_dist_loss=pdist, circle_reg=targs.get("circle_reg", 0.0),
                                                l1=targs.get("l1_norm", 0.0), l2=targs.get("l2_norm", 0.0),
                                                lr=targs.get("lr", 5e-5), lr_scheduler=targs.get("lr_scheduler"))
    model = model.to(device).eval()
    return model.set_gemm(gemm) if gemm else model


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    if args.batchsize < 1:
        build_parser().error("--batchsize must be >= 1")
    if not os.path.isfile(os.path.join(args.model, "training_args.json")):
        build_parser().error(f"{args.model} is not a model directory (no training_args.json)")
    if not os.path.isdir(args.angles):
        build_parser().error(f"--angles {args.angles} is not a directory")
    with open(os.path.join(args.model, "training_args.json")) as f:
        targs = json.load(f)
    T = targs["timesteps"]
    if args.t is not None and any(not 0 <= t < T for t in args.t):
        build_parser().error(f"--t values must lie in [0, {T})")
    model = build_model(args.model, targs, args.device, args.gemm)
    tables = AnglesTableDataset.from_model_dir(args.angles, args.model)
    key = "coords" if targs["angles_definitions"] == "cart-coords" else "angles"

    def noised(exhaustive: bool) -> NoisedAnglesDataset:
        return NoisedAnglesDataset(tables, dset_key=key, timesteps=T, exhaustive_t=exhaustive,
                                   beta_schedule=targs["variance_schedule"], nonangular_variance=1.0,
                                   angular_variance=targs["variance_scale"])

    torch.manual_seed(args.seed)
    out = {"model": os.path.abspath(args.model), "n_structures": len(tables), "timesteps": T, "noise": args.noise,
           "seed": args.seed, "batch_size": args.batchsize}
    if args.t is None:
        out.update(losses.validation_loss(model, noised(args.exhaustive_t), args.batchsize, args.noise, args.seed))
    else:
        out["at_t"] = {}
        for t in args.t:
            out["at_t"][str(t)] = losses.validation_loss(model, noised(False), args.batchsize, args.noise, args.seed, t=t)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in out if k in ("val_loss", "n_structures", "terms")}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
