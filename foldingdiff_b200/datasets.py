"""
The dataset-side objects the sampler needs - and only those.

Mirrors the duck-typed contract `sampling.sample` documents at
/root/reference/foldingdiff/sampling.py:150-156:
  * `AnglesEmptyDataset`   (reference datasets.py:569-623): data-free stand-in that carries
    feature names / angularity / pad / training mean offset of a model directory;
  * `NoisedAnglesDataset`  (reference datasets.py:685-886): schedule tables
    (`alpha_beta_terms`), `timesteps`, `sample_noise` (initial wrapped-Gaussian noise,
    :772-799) and the forward-noising `__getitem__` (:801-886) used by the partial-denoise
    path (`get_reconstruction_error`, BASELINE config 5).
The CATH featurisation / caching classes (reference datasets.py:75-566) are training data
plumbing and out of scope.
"""
from __future__ import annotations

import json
import logging
import os
from typing import Dict, Optional

import numpy as np
import torch

from . import beta_schedules, utils

FEATURE_SET_NAMES_TO_ANGULARITY = {
    "canonical": [False, False, False, True, True, True, True, True, True],
    "canonical-full-angles": [True, True, True, True, True, True],
    "canonical-minimal-angles": [True, True, True, True],
    "cart-coords": [False, False, False],
}
FEATURE_SET_NAMES_TO_FEATURE_NAMES = {
    "canonical": ["0C:1N", "N:CA", "CA:C", "phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"],
    "canonical-full-angles": ["phi", "psi", "omega", "tau", "CA:C:1N", "C:1N:1CA"],
    "canonical-minimal-angles": ["phi", "psi", "omega", "tau"],
    "cart-coords": ["x", "y", "z"],
}


class AnglesEmptyDataset:
    """Carries the metadata of a trained model's dataset without any data."""

    def __init__(self, feature_set_key: str, pad: int = 128, mean_offset: Optional[np.ndarray] = None):
        key = "coords" if feature_set_key == "cart-coords" else "angles"
        self.feature_is_angular = {key: FEATURE_SET_NAMES_TO_ANGULARITY[feature_set_key]}
        self.feature_names = {key: FEATURE_SET_NAMES_TO_FEATURE_NAMES[feature_set_key]}
        self.pad = pad
        self._mean_offset = mean_offset
        if mean_offset is not None:
            assert mean_offset.size == len(self.feature_names[key])

    @classmethod
    def from_dir(cls, dirname: str) -> "AnglesEmptyDataset":
        with open(os.path.join(dirname, "training_args.json")) as f:
            targs = json.load(f)
        offset_file = os.path.join(dirname, "training_mean_offset.npy")
        offset = np.load(offset_file) if os.path.isfile(offset_file) else None
        return cls(targs["angles_definitions"], pad=targs["max_seq_len"], mean_offset=offset)

    def get_masked_means(self) -> np.ndarray:
        # The reference raises when the offset file is absent (datasets.py:613-617), which makes
        # sampling.sample() fail on such model dirs; the behaviour is kept.
        if self._mean_offset is None:
            raise NotImplementedError
        return np.copy(self._mean_offset)

    def __len__(self):
        raise NotImplementedError

    def __getitem__(self, index):
        raise NotImplementedError


class NoisedAnglesDataset:
    """Schedule + noise source around a wrapped dataset (which may be an AnglesEmptyDataset)."""

    def __init__(self, dset, dset_key: str = "angles", timesteps: int = 250, exhaustive_t: bool = False,
                 beta_schedule: str = "linear", nonangular_variance: float = 1.0,
                 angular_variance: float = 1.0) -> None:
        assert hasattr(dset, "feature_names") and hasattr(dset, "feature_is_angular")
        assert dset_key in dset.feature_is_angular, f"{dset_key} not in {dset.feature_is_angular}"
        self.dset = dset
        self.dset_key = dset_key
        self.n_features = len(dset.feature_is_angular[dset_key])
        self.nonangular_var_scale = nonangular_variance
        self.angular_var_scale = angular_variance
        self.timesteps = timesteps
        self.schedule = beta_schedule
        self.exhaustive_timesteps = exhaustive_t
        betas = beta_schedules.get_variance_schedule(beta_schedule, timesteps)
        self.alpha_beta_terms = beta_schedules.compute_alphas(betas)

    feature_names = property(lambda self: self.dset.feature_names)
    feature_is_angular = property(lambda self: self.dset.feature_is_angular)
    pad = property(lambda self: self.dset.pad)
    filenames = property(lambda self: self.dset.filenames)

    def sample_length(self, *args, **kwargs):
        return self.dset.sample_length(*args, **kwargs)

    def __len__(self) -> int:
        n = len(self.dset)
        return n * self.timesteps if self.exhaustive_timesteps else n

    def __str__(self) -> str:
        return (f"NoisedAnglesDataset wrapping {self.dset} with {self.schedule}-{self.timesteps}, variance "
                f"scales {self.nonangular_var_scale} / {self.angular_var_scale}")

    def _angular_index(self) -> np.ndarray:
        return np.where(self.dset.feature_is_angular[self.dset_key])[0]

    def sample_noise(self, vals: torch.Tensor) -> torch.Tensor:
        """
        Zero-centred Gaussian noise shaped like `vals` (only its shape/dtype/device are used), each
        feature column scaled by its variance scale, angular columns wrapped into [-pi, pi).
        Draws from torch's global generator for `vals.device`, like the reference.
        """
        noise = torch.randn_like(vals)
        if self.angular_var_scale != 1.0 or self.nonangular_var_scale != 1.0:
            angular = self.dset.feature_is_angular[self.dset_key]
            for j in range(noise.shape[-1]):
                noise[..., j] *= self.angular_var_scale if angular[j] else self.nonangular_var_scale
        idx = self._angular_index()
        noise[..., idx] = utils.modulo_with_wrapped_range(noise[..., idx], -np.pi, np.pi)
        return noise

    def __getitem__(self, index: int, use_t_val: Optional[int] = None,
                    ignore_zero_center: bool = False) -> Dict[str, torch.Tensor]:
        """Forward-noise item `index`: corrupted = sqrt(abar_t) x0 + sqrt(1 - abar_t) noise, wrapped."""
        assert 0 <= index < len(self), f"Index {index} out of bounds for {len(self)}"
        if self.exhaustive_timesteps:
            item_index, time_index = divmod(index, self.timesteps)
            item = self.dset.__getitem__(item_index, ignore_zero_center=ignore_zero_center)
        else:
            item = self.dset.__getitem__(index, ignore_zero_center=ignore_zero_center)
        vals = (item[self.dset_key] if self.dset_key is not None else item).clone()
        assert isinstance(vals, torch.Tensor)

        if use_t_val is not None:
            assert not self.exhaustive_timesteps, "Cannot use specific t in exhaustive mode"
            t = torch.from_numpy(np.clip(np.array([use_t_val]), 0, self.timesteps - 1)).long()
        elif self.exhaustive_timesteps:
            t = torch.tensor([time_index]).long()
        else:
            t = torch.randint(0, self.timesteps, (1,)).long()

        sqrt_abar = self.alpha_beta_terms["sqrt_alphas_cumprod"][t.item()]
        sqrt_1m_abar = self.alpha_beta_terms["sqrt_one_minus_alphas_cumprod"][t.item()]
        noise = self.sample_noise(vals)
        noised = sqrt_abar * vals + sqrt_1m_abar * noise
        idx = self._angular_index()
        noised[:, idx] = utils.modulo_with_wrapped_range(noised[:, idx], -np.pi, np.pi)
        out = {"corrupted": noised, "t": t, "known_noise": noise,
               "sqrt_alphas_cumprod_t": sqrt_abar, "sqrt_one_minus_alphas_cumprod_t": sqrt_1m_abar}
        if isinstance(item, dict):
            assert item.keys().isdisjoint(out.keys())
            item.update(out)
            return item
        return out


class SyntheticAnglesDataset:
    """
    Stand-in for CathCanonicalAnglesOnlyDataset when no PDB files / biotite are available
    (BASELINE config 5 on synthetic inputs): `n` chains of fixed `length`, x0 = wrap(randn * scale),
    left-aligned in a `pad`-long tensor.  Same item keys the reference's datasets return
    ("angles", "attn_mask", "lengths", "position_ids").
    """

    def __init__(self, n: int, length: int, pad: int = 128, feature_set_key: str = "canonical-full-angles",
                 scale: float = 0.5, seed: int = 0, mean_offset: Optional[np.ndarray] = None):
        self.feature_is_angular = {"angles": FEATURE_SET_NAMES_TO_ANGULARITY[feature_set_key]}
        self.feature_names = {"angles": FEATURE_SET_NAMES_TO_FEATURE_NAMES[feature_set_key]}
        self.pad = pad
        self._mean_offset = mean_offset
        g = torch.Generator().manual_seed(seed)
        nf = len(self.feature_names["angles"])
        self._x0 = torch.zeros(n, pad, nf)
        self._x0[:, :length] = utils.modulo_with_wrapped_range(torch.randn(n, length, nf, generator=g) * scale)
        self._length = length
        self.filenames = [f"synthetic_{i}" for i in range(n)]

    def get_masked_means(self):
        return None if self._mean_offset is None else np.copy(self._mean_offset)

    def __len__(self):
        return self._x0.shape[0]

    def __getitem__(self, index, ignore_zero_center: bool = False):
        mask = torch.zeros(self.pad)
        mask[: self._length] = 1.0
        return {"angles": self._x0[index].clone(), "attn_mask": mask,
                "lengths": torch.tensor(self._length, dtype=torch.int64),
                "position_ids": torch.arange(self.pad)}


class AnglesTableDataset:
    """
    Held-out structures given as angle tables, producing the item of the reference's CathCanonicalAnglesOnlyDataset
    (datasets.py:364-460): "angles" (pad, F) fp32, "attn_mask", "position_ids", "lengths".  Wrap it in
    NoisedAnglesDataset to evaluate a model's loss (losses.validation_loss).

    `tables` is a directory of the *.csv.gz angle tables bin/sample.py / writers.py write (read in sorted file-name
    order, pandas index_col=0, feature-name header), or a sequence of (L, F) arrays / DataFrames in the model's feature
    order.  Per item, as the reference does:
      * subtract `mean_offset` (the model dir's training_mean_offset.npy) and wrap the angular columns to [-pi, pi)
      * NaN -> 0
      * pad to `pad`, or trim longer tables by `trim_strategy`: "leftalign" keeps the first `pad` rows, "randomcrop"
        a window drawn from np.random.default_rng(6489), "discard" drops such tables at load (datasets.py:175-183)
    """

    def __init__(self, tables, feature_set_key: str = "canonical-full-angles", pad: int = 128,
                 mean_offset: Optional[np.ndarray] = None, trim_strategy: str = "leftalign"):
        if trim_strategy not in ("leftalign", "randomcrop", "discard"):
            raise ValueError(f"Unknown trim strategy: {trim_strategy}")
        key = "coords" if feature_set_key == "cart-coords" else "angles"
        self.feature_is_angular = {key: FEATURE_SET_NAMES_TO_ANGULARITY[feature_set_key]}
        self.feature_names = {key: FEATURE_SET_NAMES_TO_FEATURE_NAMES[feature_set_key]}
        self._key = key
        self.pad = pad
        self.trim_strategy = trim_strategy
        self.rng = np.random.default_rng(seed=6489)  # datasets.py:111
        self._mean_offset = None if mean_offset is None else np.asarray(mean_offset, dtype=np.float64)
        names = self.feature_names[key]
        if self._mean_offset is not None:
            assert self._mean_offset.size == len(names), f"mean offset has {self._mean_offset.size} entries"
        if isinstance(tables, (str, os.PathLike)):
            import glob
            paths = sorted(glob.glob(os.path.join(os.fspath(tables), "*.csv.gz")))
            if not paths:
                raise FileNotFoundError(f"no *.csv.gz angle tables in {tables}")
            arrays, self.filenames = [], []
            for p in paths:
                arrays.append(self._read_table(p, names))
                self.filenames.append(p)
        else:
            arrays = [self._as_array(t, names) for t in tables]
            self.filenames = [f"table_{i}" for i in range(len(arrays))]
        if trim_strategy == "discard":
            keep = [i for i, a in enumerate(arrays) if a.shape[0] <= pad]
            logging.info(f"Removing structures longer than {pad} keeps {len(keep)}/{len(arrays)}")
            arrays = [arrays[i] for i in keep]
            self.filenames = [self.filenames[i] for i in keep]
        self._tables = arrays

    @staticmethod
    def _read_table(path: str, names) -> np.ndarray:
        import pandas as pd
        df = pd.read_csv(path, index_col=0)
        missing = [n for n in names if n not in df.columns]
        if missing:
            raise ValueError(f"{path}: missing feature columns {missing}")
        return df.loc[:, names].to_numpy(dtype=np.float64)

    @staticmethod
    def _as_array(t, names) -> np.ndarray:
        if hasattr(t, "loc") and hasattr(t, "columns"):
            return t.loc[:, names].to_numpy(dtype=np.float64)
        a = np.asarray(t, dtype=np.float64)
        if a.ndim != 2 or a.shape[1] != len(names):
            raise ValueError(f"expected an (L, {len(names)}) table, got {a.shape}")
        return a

    @classmethod
    def from_model_dir(cls, tables, model_dir: str) -> "AnglesTableDataset":
        """Feature set, pad, trim strategy and mean offset of a training output directory."""
        with open(os.path.join(model_dir, "training_args.json")) as f:
            targs = json.load(f)
        offset_file = os.path.join(model_dir, "training_mean_offset.npy")
        offset = np.load(offset_file) if os.path.isfile(offset_file) else None
        return cls(tables, targs["angles_definitions"], pad=targs["max_seq_len"], mean_offset=offset,
                   trim_strategy=targs.get("trim_strategy", "leftalign"))

    def get_masked_means(self):
        return None if self._mean_offset is None else np.copy(self._mean_offset)

    def __len__(self) -> int:
        return len(self._tables)

    def __getitem__(self, index, ignore_zero_center: bool = False) -> Dict[str, torch.Tensor]:
        if not 0 <= index < len(self):
            raise IndexError("Index out of range")
        angles = self._tables[index].copy()
        if self._mean_offset is not None and not ignore_zero_center:
            angles = angles - self._mean_offset
            idx = np.where(self.feature_is_angular[self._key])[0]
            angles[:, idx] = utils.modulo_with_wrapped_range(angles[:, idx], -np.pi, np.pi)
        np.nan_to_num(angles, copy=False, nan=0)
        l = min(self.pad, angles.shape[0])
        attn_mask = torch.zeros(size=(self.pad,))
        attn_mask[:l] = 1.0
        if angles.shape[0] < self.pad:
            angles = np.pad(angles, ((0, self.pad - angles.shape[0]), (0, 0)), mode="constant", constant_values=0)
        elif angles.shape[0] > self.pad:
            if self.trim_strategy == "randomcrop":
                start = self.rng.integers(0, angles.shape[0] - self.pad)
                angles = angles[start:start + self.pad]
            else:
                angles = angles[: self.pad]
        return {self._key: torch.from_numpy(np.ascontiguousarray(angles)).float(), "attn_mask": attn_mask,
                "position_ids": torch.arange(start=0, end=self.pad, step=1, dtype=torch.long),
                "lengths": torch.tensor(l, dtype=torch.int64)}


logging.getLogger(__name__).addHandler(logging.NullHandler())
